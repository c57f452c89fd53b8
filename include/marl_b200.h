/*
 * libmarl_b200 -- C ABI of the B200-native (sm_100a) value-factorisation learner hot path.
 *
 * The reference (Skylarking/MARL) is pure Python/PyTorch and has no FFI of its own; the
 * entry points below are what a binding for its hot path attaches to.  Each one names the
 * reference code it replaces (paths relative to the reference root).  Conventions:
 *   - every function returns int: 0 = ok, <0 = argument error (MARL_EINVAL), >0 = cudaError_t;
 *   - all data pointers are DEVICE pointers unless the name ends in _host;
 *   - nothing is allocated or freed on behalf of the caller; workspaces are caller-owned;
 *   - `stream` is a cudaStream_t; every call is asynchronous with respect to the host;
 *   - tensors are dense, row-major fp32 in the reference's episode-major layout
 *     (common/replaybuffer.py:19-30), rows of the folded agent batch are (b, n) with n minor
 *     (controller/share_params.py:110); action ids are int64.
 *   - H = rnn_hidden_dim = 64 and E = qmix_hidden_dim = 32 are compile-time constants
 *     (common/arguments.py:88-89); everything else is a run-time size.
 */
#ifndef MARL_B200_H
#define MARL_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MARL_B200_VERSION 100
#define MARL_HIDDEN 64
#define MARL_QMIX_EMBED 32

int marl_version(void);
/* Runtime probe: fills sm count / compute capability of the current device. */
int marl_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* B episodes, L = max_episode_len after truncation (algorithm/q_learner.py:49-66),
 * N agents, A actions, O obs dim, S state dim. */
typedef struct marl_dims { int B, L, N, A, O, S; } marl_dims;

/* One episode batch on the device, fp32, the 11 ReplayBuffer keys (common/replaybuffer.py:19-30):
 * o,o_next [B,L,N,O]  s,s_next [B,L,S]  u [B,L,N] (int64)  r,padded,terminated [B,L]
 * avail_u,avail_u_next,u_onehot [B,L,N,A]. */
typedef struct marl_episode_f32 {
    float* o; float* s; long long* u; float* r; float* o_next; float* s_next;
    float* avail_u; float* avail_u_next; float* u_onehot; float* padded; float* terminated;
} marl_episode_f32;

/* The same 11 keys as the reference hands them to train(): float64, [B, T_src, ...]
 * (u may be float64 or int64: u_is_int64). */
typedef struct marl_episode_f64 {
    const double* o; const void* u; const double* s; const double* r; const double* o_next;
    const double* s_next; const double* avail_u; const double* avail_u_next; const double* u_onehot;
    const double* padded; const double* terminated;
    int u_is_int64;
} marl_episode_f64;

/* ---- environment: env/single_state_matrix_game.py:27-40 (step), :81-120 (episode layout) ----
 * Steps n_envs independent TwoAgentsMatrixGame instances: reward = payoff[a0, a1], terminated = 1,
 * and writes one T=1 episode record per env.  actions: [n_envs, 2] int32 or int64 (action_bytes 4|8).
 * obs_value: 0 reproduces get_obs()/get_state() (what a rollout records), 1 reproduces get_episodes().
 * r64 (nullable): the float64 reward exactly as the reference returns it. */
int marl_matrix_game_step(const double* payoff_host /*[9]*/, const void* actions, int action_bytes,
                          long long n_envs, float obs_value, const marl_episode_f32* out,
                          double* r64, void* stream);
/* Sets *bad_flag_device to 1 if any action is outside {0,1,2} (reference: IndexError). */
int marl_matrix_game_validate_actions(const void* actions, int action_bytes, long long n_envs,
                                      int* bad_flag_device, void* stream);

/* ---- batch ingest: algorithm/q_learner.py:63-78,83 ----
 * float64 [B, T_src, ...] -> fp32 [B, L, ...] (truncation to L and the dtype casts of train(); u is
 * truncated toward zero like th.tensor(..., dtype=th.long)). */
int marl_ingest_f64(const marl_episode_f64* src, int T_src, const marl_dims* d,
                    const marl_episode_f32* dst, void* stream);

/* Device-resident variant: fp32 [B, T_src, ...] (e.g. rows sampled from a device replay buffer) ->
 * the step's working set [B, L, ...]. */
int marl_ingest_f32(const marl_episode_f32* src, int T_src, const marl_dims* d,
                    const marl_episode_f32* dst, void* stream);

/* ---- device replay buffer: common/replaybuffer.py:54-60 (sample) fused with the ingest ----
 * Output episode b of the working set [B, L, ...] is episode episode_idx[b] (device int64, sampled with
 * replacement by the host RNG exactly like the reference) of the ring [size, T_ring, ...], truncated to L. */
int marl_replay_gather_f32(const marl_episode_f32* ring, int T_ring, const long long* episode_idx,
                           const marl_dims* d, const marl_episode_f32* dst, void* stream);

/* ---- agent: network/q_network.py:6-21 unrolled by controller/share_params.py:125-168 ---- */
typedef struct marl_agent_params {
    const float* fc1_w;  /* [H, O+A+N], or as the input blocks select */  const float* fc1_b;  /* [H] */
    const float* w_ih;   /* [3H, H]   */  const float* w_hh;   /* [3H, H] */
    const float* b_ih;   /* [3H]      */  const float* b_hh;   /* [3H] */
    const float* fc2_w;  /* [A, H]    */  const float* fc2_b;  /* [A] */
} marl_agent_params;

typedef struct marl_agent_grads {
    float* fc1_w; float* fc1_b; float* w_ih; float* w_hh; float* b_ih; float* b_hh; float* fc2_w; float* fc2_b;
} marl_agent_grads;

/* One T-step unroll ("stream") of the shared agent over an episode batch.
 * Input row at step t = [obs[b,t,n] | onehot[b,t-shift,n] (zeros when t < shift) | eye(N)[n]]
 * (share_params.py:84-112; shift_onehot=1 is get_current_q_values, 0 is get_next_q_values).
 * Hidden state starts from zeros (init_hidden, :74-76), from h0, or -- h0_from >= 0 -- from the
 * final hidden of an earlier stream of the same call (the carried hidden of q_learner.py:110). */
typedef struct marl_unroll_stream {
    const float* obs;        /* [B,L,N,O] */
    const float* onehot;     /* [B,L,N,A] */
    int shift_onehot;
    int full_input;          /* 1: `obs` already holds the full [O+A+N]-wide input rows (RNNQNet.forward /
                                choose_action, share_params.py:37-61); onehot is ignored */
    int h0_from;             /* -1, or index of an earlier stream in the same call */
    const float* h0;         /* [B*N,H] or NULL */
    marl_agent_params params;
    float* q;                /* out [B,L,N,A], or NULL: skip the fc2 head (a fused mixer evaluates it from `hidden`,
                                see marl_select_fused) */
    float* hidden;           /* out [B,L,N,H], h after each step */
    float* h_last;           /* out [B*N,H] or NULL */
    float* x;                /* workspace/out [B,L,N,H]: relu(fc1) (needed by the backward; the fused input-layer kernel only fills it when `gates` is given) */
    float* gi;               /* workspace [B,L,N,3H] */
    float* gates;            /* out [B,L,N,4H] (r, z, n, W_hn h + b_hn) for the backward, or NULL */
    float* w_ih_t;           /* out [H, 3H] or NULL: params.w_ih transposed (written by the fused input-layer kernel on its way, by one
                                small launch otherwise).  Hand it to marl_unroll_bwd.w_ih_t of the SAME step: the data gradient
                                behind the recurrence then reads both operands along the reduction */
    const int* ep_len;       /* device [B] (marl_episode_lengths) or NULL.  Non-NULL: this stream's recurrence stops each row at
                                its episode's length -- the padded steps behind it (q_learner.py:49-66 keeps them up to the
                                batch maximum) are not computed; `hidden` / `q` keep whatever they held there (finite: the
                                loss masks them) and h_last is the hidden after the last REAL step.  Never set it on a
                                stream another stream continues from (h0_from): the reference carries the hidden state through
                                the padded steps (q_learner.py:96,110), so that one must run to L. */
    const float* padded;     /* [B,L] fp32 or NULL.  Non-NULL (with ep_len): the call computes ep_len from it first -- exactly
                                marl_episode_lengths, launched on a forked lane beside the input layers instead of in front of
                                them -- so ep_len is then an OUTPUT of the call (and of every stream that shares the array) */
    int* row_order;          /* device scratch [B*N] ints or NULL.  When the streams of a chain (a stream and the ones that continue
                                it through h0_from) carry an ep_len and a row_order, the chain's rows (b, n) are dealt to the
                                recurrence CTAs sorted by episode length -- the CTAs that advance the most rows get the shortest
                                ones, rows that advance in lock-step have similar lengths -- instead of in index order.  Results
                                are unchanged (rows are independent); the call fills the array itself.  (Batches of more than 1024
                                episodes keep the index order, here and in the backward.) */
    int* row_order_bwd;      /* out [B*N] ints or NULL (needs an ep_len on some stream of the call): the same deal for the plan
                                of marl_agent_unroll_bwd; hand it to marl_unroll_bwd.row_order of the SAME step */
    int agent_stride;        /* 0: one parameter set shared by all agents (everything above).  Otherwise one network per agent
                                (SeparatedMAC, share_params.py:389-610): `params` points at agent 0's set and agent n+1's set
                                sits agent_stride floats behind agent n's (a multiple of 4).  Every stream of a call carries the
                                same stride.  The input row of (b, t, n) is then
                                [obs | onehot[b,t-shift,n] if last_action | eye(N)[n] if agent_id] (share_params.py:467-506),
                                so fc1_w is [H, O + A*last_action + N*agent_id].  MARL_EINVAL together with full_input, w_ih_t,
                                ep_len, padded, row_order or row_order_bwd */
    int last_action;         /* separated, or shared with input_flags = 1 (ignored otherwise): the input carries the last action */
    int agent_id;            /* separated, or shared with input_flags = 1: the input carries the agent's one-hot id */
    int input_flags;         /* agent_stride == 0 only.  1: last_action / agent_id select the input blocks as for separated
                                networks, [obs | onehot[b,t-shift,n] if last_action | eye(N)[n] if agent_id], so fc1_w is
                                [H, O + A*last_action + N*agent_id] (share_params.py:84-123 with args.last_action /
                                args.reuse_network); onehot may be NULL when last_action is 0.  0: the default
                                [obs | last action | agent id] whatever last_action / agent_id hold.  MARL_EINVAL together
                                with full_input; every stream of a call has the same input width */
} marl_unroll_stream;

/* ep_len[b] = 1 + the last step with padded[b, t] == 0 (at least 1): every step at or beyond it has mask = 0 in the loss
 * (q_learner.py:79,167), i.e. contributes neither to the loss nor to any gradient.  padded [B, L] fp32. */
int marl_episode_lengths(const float* padded, int B, int L, int* ep_len, void* stream);

int marl_agent_unroll_fwd(const marl_dims* d, const marl_unroll_stream* streams, int n_streams, void* stream);

/* BPTT of one unroll (autograd of share_params.py:125-146 as triggered by
 * loss.backward(), q_learner.py:171).  dq [B,L,N,A] and dhidden [B,L,N,H] (either may be NULL) are
 * dL/dq and an external dL/dhidden (QTRAN, qtran_learner.py:119,136).  Gradients are ACCUMULATED
 * into `grads` (caller zeroes).  Workspaces: dhext [B,L,N,H], dgi [B,L,N,3H], dgh [B,L,N,3H],
 * dx [B,L,N,H]. */
typedef struct marl_unroll_bwd {
    const float* obs; const float* onehot; int shift_onehot; int full_input;
    marl_agent_params params;
    const float* hidden; const float* x; const float* gates;
    const float* h0;         /* [B*N,H] initial hidden of the forward, or NULL (zeros) */
    const float* dq; const float* dhidden;
    float* dhext; float* dgi; float* dgh; float* dx;
    float* dh0;              /* out [B*N,H] dL/dh0, or NULL */
    marl_agent_grads grads;
    int dhext_ready;         /* != 0: dhext already holds dq . fc2_w (marl_qmix_td_fwd_bwd wrote it); skip that product */
    const float* w_ih_t;     /* [H, 3H] = params.w_ih transposed as marl_unroll_stream.w_ih_t produced it in this step's forward,
                                or NULL (the data gradient then transposes W_ih while staging it) */
    const int* ep_len;       /* device [B] or NULL.  Non-NULL: the backward chain of a row starts at its episode's last real
                                step; dgi / dgh of the padded steps behind it are written as zeros (what the full chain
                                computes there: every upstream gradient is masked to zero) */
    const int* row_order;    /* [B*N] = marl_unroll_stream.row_order_bwd of this step's forward call, or NULL (index order); only
                                read together with ep_len */
    int agent_stride;        /* as marl_unroll_stream.agent_stride: 0 shared, else one network per agent with `params` and
                                `grads` at agent 0's set and agent n+1's agent_stride floats behind agent n's.  MARL_EINVAL
                                together with full_input, w_ih_t, ep_len or row_order */
    int last_action;         /* as marl_unroll_stream.last_action */
    int agent_id;            /* as marl_unroll_stream.agent_id */
    int input_flags;         /* agent_stride == 0 only: as marl_unroll_stream.input_flags (the forward's value) */
} marl_unroll_bwd;

int marl_agent_unroll_bwd(const marl_dims* d, const marl_unroll_bwd* a, void* stream);

/* ---- action-value selection: algorithm/q_learner.py:100,105,108-117,126-127 ----
 * q_chosen = q_evals.gather(u); q_targets[avail_u_next==0] = -9999999 (IN PLACE, as the reference);
 * double-Q (q_evals_next != NULL): a* = argmax_a of the masked q_evals_next (first max wins),
 * q_targets_chosen = q_targets.gather(a*); else q_targets_chosen = max_a q_targets.
 * Optional (QPLEX): max_q_evals = max_a of q_evals masked by avail_u; q_targets_max = max_a q_targets. */
int marl_q_select(const marl_dims* d, const float* q_evals, const long long* u, const float* q_evals_next,
                  float* q_targets, const float* avail_u_next, const float* avail_u /*nullable*/,
                  float* q_chosen, long long* a_star /*nullable*/, float* q_targets_chosen,
                  float* max_q_evals /*nullable*/, float* q_targets_max /*nullable*/,
                  float* a_star_onehot /*nullable, [B,L,N,A] one-hot of a* (q_learner.py:140-143)*/, void* stream);

/* ---- acting: controller/share_params.py:62-72 for all (env, agent) rows at once ----
 * action[i] = explore[i] ? random_action[i] : argmax_a(q[i, a] masked to -inf where avail[i, a] == 0) (first maximum);
 * avail, explore / random_action and onehot are nullable.  explore / random_action are drawn on the host in the
 * reference's RNG order (one uniform per agent, one choice only when exploring). */
int marl_epsgreedy_select(int rows, int A, const float* q, const float* avail, const unsigned char* explore,
                          const long long* random_action, long long* action, float* onehot, void* stream);

/* One epsilon-greedy step of the shared agent for every row r = e*N + n of n_envs instances, in ONE launch:
 *   in = [obs[r] (O) | last_onehot[r] (A) | eye(N)[n]]  (share_params.py:84-112, never materialised)
 *   x = relu(fc1 in + b1);  h' = GRUCell(x, h_in[r]) (gate order r, z, n);  q = fc2 h' + b2
 *   greedy = first maximum of q masked to -inf where avail[r, a] == 0 (every action masked -> 0).
 * Exploration, at most one form (both given -> MARL_EINVAL):
 *   flag form:    explore[r] (uint8) != 0 takes random_action[r] (int64), drawn on the host in the reference's RNG order;
 *   uniform form: explore_u[r] < eps (float64 compare) takes the min(floor(choice_u[r] * cnt), cnt - 1)-th available
 *                 action (float64), cnt = number of available actions; cnt = 0 gives action 0.
 * obs [rows, O], last_onehot [rows, A], avail [rows, A] (NULL: all available), h_in / h_out [rows, H] (may alias: the
 * hidden state is advanced in place).  Outputs: action [rows] int64; nullable onehot [rows, A] fp32 of the action and
 * q [rows, A], the network's output before the mask.  gate (nullable, device int): when *gate == 0 the launch does
 * nothing (a rollout step after every instance has finished).  All weights are staged on chip: a shape whose
 * fc1 / GRU / fc2 weights do not fit in one block's shared memory returns MARL_EINVAL. */
int marl_agent_act(int n_envs, int N, int A, int O, const marl_agent_params* p, const float* obs,
                   const float* last_onehot, const float* avail, const float* h_in, float* h_out,
                   const unsigned char* explore, const long long* random_action, const double* explore_u,
                   const double* choice_u, double eps, const int* gate, long long* action, float* onehot, float* q,
                   void* stream);

/* marl_agent_act with the input blocks chosen by last_action / agent_id (share_params.py:84-123 with args.last_action /
 * args.reuse_network):
 *   in = [obs[r] (O) | last_onehot[r] (A, only if last_action) | eye(N)[n] (N, only if agent_id)]
 * so p->fc1_w is [64, O + A*last_action + N*agent_id].  Every other argument, the row layout, the exploration forms, gate
 * and the outputs are those of marl_agent_act, which is this call with last_action = agent_id = 1; last_onehot may be NULL
 * when last_action is 0.  MARL_EINVAL when last_action is set and last_onehot is NULL, and in every case marl_agent_act
 * returns it. */
int marl_agent_act_input(int n_envs, int N, int A, int O, int last_action, int agent_id, const marl_agent_params* p,
                         const float* obs, const float* last_onehot, const float* avail, const float* h_in, float* h_out,
                         const unsigned char* explore, const long long* random_action, const double* explore_u,
                         const double* choice_u, double eps, const int* gate, long long* action, float* onehot, float* q,
                         void* stream);

/* marl_agent_act with one network per agent (SeparatedMAC, share_params.py:389-610): row r = e*N + n uses p[n], an
 * array of N parameter sets, and its input is
 *   in = [obs[r] (O) | last_onehot[r] (A, only if last_action) | eye(N)[n] (N, only if agent_id)]  (share_params.py:467-506)
 * so p[n].fc1_w is [64, O + A*last_action + N*agent_id].  Every other argument, the row layout, the exploration forms,
 * gate and the outputs are those of marl_agent_act; last_onehot may be NULL when last_action is 0.  A tile holds up to
 * 32 instances of one agent, so the launch stages each agent's weights in shared memory once per CTA that serves it.
 * MARL_EINVAL when N > 128, when any of the N parameter sets has a NULL pointer, when last_action is set and last_onehot
 * is NULL, or when one agent's weights do not fit in one block's shared memory. */
int marl_agent_act_separated(int n_envs, int N, int A, int O, int last_action, int agent_id, const marl_agent_params* p,
                             const float* obs, const float* last_onehot, const float* avail, const float* h_in,
                             float* h_out, const unsigned char* explore, const long long* random_action,
                             const double* explore_u, const double* choice_u, double eps, const int* gate,
                             long long* action, float* onehot, float* q, void* stream);

/* Philox exploration form: every row draws its own pair from a counter-based generator inside the act launch, so the
 * draws are a pure function of (seed, episode, step, agent) -- the same whichever call or device plays the episode -- and
 * no draw buffer exists.  Philox4x64-10 (Random123's constants and rounds, numpy's np.random.Philox) under key
 * (seed, 0); row r = e*N + n at step `step` uses counter (episode_base + e, step, n, 0) (word 0 wraps modulo 2^64).
 * explore_u = (word0 >> 11) * 2^-53 and choice_u = (word1 >> 11) * 2^-53 (numpy's Generator.random() conversion), then
 * the uniform form's rule: explore iff explore_u < eps (float64), where eps is eps_table[min(e, eps_len - 1)] when
 * eps_table (device float64) is set and the call's eps otherwise. */
typedef struct {
    unsigned long long seed;          /* Philox key word 0 (word 1 = 0) */
    unsigned long long episode_base;  /* counter word 0 of row e*N + n is episode_base + e */
    int step;                         /* counter word 1 (>= 0) */
    const double* eps_table;          /* nullable: instance e explores with eps_table[min(e, eps_len - 1)]; else eps */
    int eps_len;
} marl_act_philox;

/* marl_agent_act_input with the exploration drawn as marl_act_philox describes (no flag or uniform arrays).  MARL_EINVAL
 * when philox is NULL, philox->step < 0, eps_table is set with eps_len < 1, and in every case marl_agent_act_input
 * returns it. */
int marl_agent_act_philox(int n_envs, int N, int A, int O, int last_action, int agent_id, const marl_agent_params* p,
                          const float* obs, const float* last_onehot, const float* avail, const float* h_in, float* h_out,
                          const marl_act_philox* philox, double eps, const int* gate, long long* action, float* onehot,
                          float* q, void* stream);

/* marl_agent_act_separated with the exploration drawn as marl_act_philox describes; MARL_EINVAL as
 * marl_agent_act_philox and marl_agent_act_separated return it. */
int marl_agent_act_separated_philox(int n_envs, int N, int A, int O, int last_action, int agent_id,
                                    const marl_agent_params* p, const float* obs, const float* last_onehot,
                                    const float* avail, const float* h_in, float* h_out, const marl_act_philox* philox,
                                    double eps, const int* gate, long long* action, float* onehot, float* q, void* stream);

/* The pairs marl_agent_act_philox draws, for testing the generator bit for bit: out[r] = (explore_u, choice_u) of row
 * r = e*N + n, [n_envs * N, 2] float64 on the device. */
int marl_philox_uniforms(unsigned long long seed, unsigned long long episode_base, int step, int n_envs, int N,
                         double* out, void* stream);

/* Bookkeeping of the batched multi-step rollout (rollout.py:52-149), one launch per environment step.
 * d: B = n instances, L = T (episode_limit), N, A, O, S; ep: the [n, T, ...] episode buffers (padding pre-filled by the
 * caller: zeros, padded = terminated = 1).  Phase t (1 <= t <= T), for every instance e that was active in step t-1:
 * u, u_onehot, r, terminated, padded = 0 of step t-1 (action / onehot of that step, reward / terminated as env.step
 * returned them), o_next / s_next / avail_u_next of step t-1 = obs / state / avail (the getters read after that step),
 * reward_sum[e] += reward (float64), last[e] = onehot[e], active[e] = !terminated[e].  Then, for t < T, every instance
 * still active gets o / s / avail_u of step t from the same getters, and counters[t] (instances active at the start of
 * step t) and counters[T] (their running sum: the environment steps) grow by the active count.  Phase 0 only opens
 * step 0 (action, onehot, reward, terminated may be NULL).  counters: device int [T + 2], counters[T + 1] is the
 * launch's scratch word (zero between launches).  active_host (nullable): page-locked host int that receives
 * counters[t] once the phase's count is complete, so the host can stop stepping without a synchronisation (the count
 * never increases, so a stale read only costs steps that do nothing).
 * obs [n, N, O], state [n, S], avail [n, N, A] fp32; action [n, N] int64; onehot / last [n, N, A] fp32; reward [n]
 * float64; terminated / active [n] uint8 (0 / 1). */
int marl_rollout_record(const marl_dims* d, int t, const marl_episode_f32* ep, const float* obs, const float* state,
                        const float* avail, const long long* action, const float* onehot, const double* reward,
                        const unsigned char* terminated, unsigned char* active, float* last, double* reward_sum,
                        int* counters, int* active_host, void* stream);

/* ---- TD target + masked MSE: algorithm/q_learner.py:165-168 ----
 * y = r + gamma*q_tot_target*(1-terminated); d = (1-padded)*(y - q_tot);
 * scalars[0] += sum d^2, scalars[1] += sum (1-padded); dq_tot = -2*(1-padded)*d  (UN-normalised:
 * the 1/sum(mask) factor is applied by the optimiser step, after the data-parallel all-reduce). */
int marl_td_loss(int M, const float* q_tot, const float* q_tot_target, const float* r, const float* terminated,
                 const float* padded, float gamma, float* dq_tot, float* scalars, void* stream);

/* ---- VDN: network/mixer.py:15-16 fused with the TD loss and its gradient ----
 * dq [B,L,N,A] receives dL/dq_evals (dense: dq_tot at the chosen action, 0 elsewhere).
 * Learner fusions (all nullable; the same as marl_qmix_td_fwd_bwd's):
 *   fc2_w [A,H] + dhext [B,L,N,H]: also emit dhext = dq . fc2_w (one scaled row of fc2_w per agent, dq has one non-zero
 *     per row); pass it on with marl_unroll_bwd.dhext_ready = 1;
 *   sel: also do marl_q_select's work (q_learner.py:100-117: gather, in-place mask of q_targets, double-Q arg-max);
 *     q_chosen / q_targets_chosen are then OUTPUTS (MARL_EINVAL when 64 N A bytes of staging exceed 160 KB). */
typedef struct marl_select_fused {   /* inputs of marl_q_select, for the fused forms of the mixers below */
    float* q_evals; float* q_evals_next /*nullable: no double-Q*/; float* q_targets; const float* avail_u_next;
    long long* a_star /*nullable out*/;
    /* hidden_evals != NULL: the agents' heads are evaluated here as well (q = fc2_w h + fc2_b, network/q_network.py:21-22):
     * q_evals / q_evals_next / q_targets [B,L,N,A] are then OUTPUTS (q_targets masked as the reference leaves it), computed
     * from the hidden states [B,L,N,H] of the eval net on o, the target net on o_next and (double-Q) the eval net on
     * o_next -- run marl_agent_unroll_fwd with q = NULL.  All seven pointers 16-byte aligned. */
    const float* hidden_evals; const float* hidden_targets; const float* hidden_evals_next;
    const float* fc2_w; const float* fc2_b; const float* fc2_w_target; const float* fc2_b_target;
} marl_select_fused;
int marl_vdn_td_fwd_bwd(const marl_dims* d, float* q_chosen, float* q_targets_chosen,
                        const long long* u, const float* r, const float* terminated, const float* padded,
                        float gamma, float* q_tot, float* q_tot_target, float* dq, float* scalars,
                        const float* fc2_w, float* dhext, const marl_select_fused* sel, void* stream);

/* ---- QMIX: network/mixer.py:57-80 ----
 * Hyper-network weights are passed concatenated (the host lays the parameters out that way):
 *   wcat [C, S], bcat [C] with C = N*E + 3E rows in the order
 *   hyper_w1 (N*E) | hyper_b1 (E) | hyper_w2 (E) | hyper_b2.0 (E);  wb2 [E], bb2 [1] = hyper_b2.2. */
typedef struct marl_qmix_params { const float* wcat; const float* bcat; const float* wb2; const float* bb2; } marl_qmix_params;
typedef struct marl_qmix_grads { float* wcat; float* bcat; float* wb2; float* bb2; } marl_qmix_grads;

/* q_tot[M] = QMixMixer(q[M,N], s[M,S]);  hy [M,C] workspace keeps the hyper-network outputs for the backward. */
int marl_qmix_fwd(int M, int N, int S, const marl_qmix_params* p, const float* q, const float* s,
                  float* hy, float* q_tot, void* stream);
/* Given dq_tot[M]: dq[M,N] and accumulated parameter gradients. dhy [M,C] workspace. */
int marl_qmix_bwd(int M, int N, int S, const marl_qmix_params* p, const float* q, const float* s,
                  const float* hy, const float* dq_tot, float* dhy, float* dq, const marl_qmix_grads* g, void* stream);
/* Learner fusion (q_learner.py:161-168 + backward): eval mixer on (q_chosen, s), target mixer on
 * (q_targets_chosen, s_next), TD loss, gradient to the eval mixer parameters and dense dq [B,L,N,A].
 * With fc2_w / dhext the kernel also emits dhext = dq . fc2_w (dq has one non-zero per row, so this is one scaled row
 * of fc2_w per agent): pass it on with marl_unroll_bwd.dhext_ready = 1.
 * With sel the kernel also does marl_q_select's work (q_learner.py:100-117: gather, in-place mask of q_targets, double-Q
 * arg-max) for its own sample: q_chosen / q_targets_chosen are then OUTPUTS and no marl_q_select call is needed
 * (MARL_EINVAL when 64 N A bytes of staging exceed 160 KB: call marl_q_select yourself then). */
int marl_qmix_td_fwd_bwd(const marl_dims* d, const marl_qmix_params* p, const marl_qmix_params* p_target,
                         const float* s, const float* s_next, float* q_chosen, float* q_targets_chosen,
                         const long long* u, const float* r, const float* terminated, const float* padded, float gamma,
                         float* hy, float* hy_target, float* dhy, float* q_tot, float* q_tot_target,
                         float* dq, const marl_qmix_grads* g, float* scalars, int flags,
                         const float* fc2_w /*nullable, [A,H]*/, float* dhext /*nullable, [B,L,N,H]*/,
                         const marl_select_fused* sel /*nullable*/, void* stream);
/* The state-only halves of the QMIX step, so that a caller can overlap them with the agent unrolls:
 * flags bit 0 of marl_qmix_td_fwd_bwd = hy / hy_target were already filled by marl_qmix_hyper_fwd,
 * bit 1 = leave dwcat/dbcat to a later marl_qmix_hyper_wgrad(dhy). */
int marl_qmix_hyper_fwd(int M, int N, int S, const marl_qmix_params* p, const float* s, float* hy, void* stream);
int marl_qmix_hyper_wgrad(int M, int N, int S, const float* s, const float* dhy, const marl_qmix_grads* g, void* stream);

/* two_hyper_layers = True (network/mixer.py:36-43): hyper_w1 / hyper_w2 are Linear(S, hh) - ReLU - Linear(hh, .).
 *   w_in [2 hh, S] = hyper_w1.0 | hyper_w2.0 (b_in likewise), w1_out [N*E, hh] = hyper_w1.2, w2_out [E, hh] = hyper_w2.2,
 *   w_b1 [E, S] = hyper_b1, w_b20 [E, S] = hyper_b2.0.
 * marl_qmix_hyper2_fwd fills the hy layout the mixing kernel reads ([w1 | b1 | w2 | b2.0], h [M, 2 hh] keeps the hidden
 * layers); run marl_qmix_td_fwd_bwd / marl_qmix_fwd|bwd kernels with flags = 3 on that hy (their wcat / bcat are then
 * unused) and finish with marl_qmix_hyper2_bwd(dhy) (dh [M, 2 hh] workspace; gradients are accumulated). */
typedef struct marl_qmix_hyper2 {
    const float* w_in; const float* b_in; const float* w1_out; const float* b1_out; const float* w2_out; const float* b2_out;
    const float* w_b1; const float* b_b1; const float* w_b20; const float* b_b20; int hh;
} marl_qmix_hyper2;
typedef struct marl_qmix_hyper2_grads {
    float* w_in; float* b_in; float* w1_out; float* b1_out; float* w2_out; float* b2_out;
    float* w_b1; float* b_b1; float* w_b20; float* b_b20;
} marl_qmix_hyper2_grads;
int marl_qmix_hyper2_fwd(int M, int N, int S, const marl_qmix_hyper2* p, const float* s, float* h, float* hy, void* stream);
int marl_qmix_hyper2_bwd(int M, int N, int S, const marl_qmix_hyper2* p, const float* s, const float* h, const float* dhy,
                         float* dh, const marl_qmix_hyper2_grads* g, void* stream);
/* Mixing only (q_tot from a filled hy; backward to dhy / dq / hyper_b2.2): the kernels behind marl_qmix_fwd / _bwd
 * without their hyper-network GEMMs. */
int marl_qmix_mix_fwd(int M, int N, const marl_qmix_params* p, const float* q, const float* hy, float* q_tot, void* stream);
int marl_qmix_mix_bwd(int M, int N, const marl_qmix_params* p, const float* q, const float* hy, const float* dq_tot,
                      float* dhy, float* dq, const marl_qmix_grads* g, void* stream);

/* ---- QPLEX: DMAQer + DMAQ_SI_Weight, network/mixer.py:85-288 (adv_hypernet_layers = 3) ----
 * Parameters are passed layer-concatenated (the host lays them out that way), K = num_kernel,
 * he = hypernet_embed, ae = adv_hypernet_embed:
 *   w1s [2he + 2K*ae, S]  rows: hyper_w_final.0 | V.0 | key_extractors.k.0 (k=0..K-1) | agents_extractors.k.0
 *   w1a [K*ae, S + N*A]   action_extractors.k.0        (input = [states | actions], never materialised)
 *   w2  [3K, ae, ae]      key.k.2 | agents.k.2 | action.k.2
 *   w3k [K, ae]           key.k.4          w3n [2K, N, ae]  agents.k.4 | action.k.4
 *   wfv [2, N, he]        hyper_w_final.2 | V.2            (biases b* in the same order)
 * Workspaces (kept for the backward): h1 [M, 2he + 3K*ae], h2 [M, 3K*ae], o3 [M, K + 2K*N], wv [M, 2N]. */
/* layers = adv_hypernet_layers (network/mixer.py:115-145; 0 means 3).  2: no w2 / b2, the output layers (w3k / w3n) read the
 * extractor block of h1; 1: single-Linear extractors, w3k = [K key rows | K*N agents rows] x S, w3n = [K*N, S + N*A], no w1a /
 * b1a / w2 / b2 and w1s / b1s hold only hyper_w_final.0 | V.0 (h1 [M, 2he]). */
typedef struct marl_qplex_dims { int N, A, S, he, ae, K, weighted_head, is_minus_one, layers; } marl_qplex_dims;
typedef struct marl_qplex_params {
    const float *w1s, *b1s, *w1a, *b1a, *w2, *b2, *w3k, *b3k, *w3n, *b3n, *wfv, *bfv;
} marl_qplex_params;
typedef struct marl_qplex_grads { float *w1s, *b1s, *w1a, *b1a, *w2, *b2, *w3k, *b3k, *w3n, *b3n, *wfv, *bfv; } marl_qplex_grads;
typedef struct marl_qplex_ws { float *h1, *h2, *o3, *wv; } marl_qplex_ws;

/* DMAQer.forward for M samples: v_tot = sum_n (w q + v)  (is_v=True, mixer.py:211-220) and, when `actions`
 * [M, N*A] and max_q [M,N] are given, a_tot = sum_n adv (lambda - 1) with adv = (w q + v) - (w max_q + v)
 * detached (calc_adv, mixer.py:222-247).  q_tot = v_tot + a_tot.  Any of the three outputs may be NULL. */
int marl_qplex_fwd(int M, const marl_qplex_dims* d, const marl_qplex_params* p, const float* q, const float* s,
                   const float* actions, const float* max_q, const marl_qplex_ws* ws,
                   float* v_tot, float* a_tot, float* q_tot, void* stream);
/* Backward for dL/dv_tot and dL/da_tot (either may be NULL; the learner passes dL/dq_tot for both):
 * dq [M,N] and accumulated parameter gradients.  a_tot trains only the lambda heads (adv is detached).
 * dws: workspaces for d(h1), d(h2), d(o3), d(wv), same shapes as ws. */
int marl_qplex_bwd(int M, const marl_qplex_dims* d, const marl_qplex_params* p, const float* q, const float* s,
                   const float* actions, const float* max_q, const marl_qplex_ws* ws, const float* dv_tot,
                   const float* da_tot, const marl_qplex_ws* dws, float* dq, const marl_qplex_grads* g, void* stream);
/* dq_dense [B,L,N,A] = dq_small [B,L,N] scattered to the chosen action u (autograd of gather, q_learner.py:100). */
int marl_scatter_dq(const marl_dims* d, const float* dq_small, const long long* u, float* dq_dense, void* stream);

/* ---- QTRAN-base: QtranQBase / QtranV (network/mixer.py:355-418) ----
 * One "joint net" shape serves both: per-agent encoder Linear(D,D)-ReLU-Linear(D,D) on rows
 * [hidden | action one-hot] (D = H + A_enc; A_enc = 0 for QtranV), sum over agents, head
 * Linear(S+D,qh)-ReLU-Linear(qh,qh)-ReLU-Linear(qh,1) on [state | encoding].
 *   QtranQBase: we1/we2 = hidden_action_encoding.{0,2}, w0/w2/w4 = q.{0,2,4}
 *   QtranV    : we1/we2 = hidden_encoding.{0,2},        w0/w2/w4 = v.{0,2,4}
 * Workspaces (kept for the backward): e1 [M*N, D], es [M, D], enc [M, D], a1 [M, qh], a2 [M, qh]. */
typedef struct marl_qtran_net_params { const float *we1, *be1, *we2, *be2, *w0, *b0, *w2, *b2, *w4, *b4; } marl_qtran_net_params;
typedef struct marl_qtran_net_grads { float *we1, *be1, *we2, *be2, *w0, *b0, *w2, *b2, *w4, *b4; } marl_qtran_net_grads;
typedef struct marl_qtran_net_ws { float *e1, *es, *enc, *a1, *a2; } marl_qtran_net_ws;

/* out[M] = net(s [M,S], hidden [M*N,H], actions [M*N,A_enc] or NULL). */
int marl_qtran_net_fwd(int M, int N, int S, int A_enc, int qh, const marl_qtran_net_params* p, const float* s,
                       const float* hidden, const float* actions, const marl_qtran_net_ws* ws, float* out, void* stream);
/* Given dout[M]: accumulated parameter gradients and dL/dhidden [M*N,H] (written, or added when
 * accumulate_dhidden != 0; NULL to skip).  dws: same shapes as ws. */
int marl_qtran_net_bwd(int M, int N, int S, int A_enc, int qh, const marl_qtran_net_params* p, const float* s,
                       const float* hidden, const float* actions, const marl_qtran_net_ws* ws, const float* dout,
                       const marl_qtran_net_ws* dws, float* dhidden, int accumulate_dhidden,
                       const marl_qtran_net_grads* g, void* stream);
/* Greedy actions (algorithm/qtran_learner.py:103-114,129,143): eval side masked with -999999 by avail_u,
 * target side masked IN PLACE with -9999999 by avail_u_next; one-hots of both argmaxes, the eval argmax,
 * max_a of the masked eval Q and the Q of the taken action. */
int marl_qtran_select(const marl_dims* d, const float* q_evals, float* q_targets, const float* avail_u,
                      const float* avail_u_next, const long long* u, float* opt_onehot_eval, float* opt_onehot_target,
                      long long* opt_action_eval, float* q_max_eval, float* q_taken, void* stream);
/* L_td + lambda_opt L_opt + lambda_nopt L_nopt (qtran_learner.py:116-152) and its gradients w.r.t.
 * joint_q (d_joint_q [M]), v (d_v [M]) and the individual Q-values (dq [B,L,N,A]); UN-normalised like
 * marl_td_loss: scalars += {loss_sum, mask_sum}; loss_parts += {sum l_td, sum l_opt, sum l_nopt}. */
int marl_qtran_losses_fwd_bwd(const marl_dims* d, const float* joint_q, const float* joint_q_target,
                              const float* joint_q_hat, const float* v, const float* q_max_eval, const float* q_taken,
                              const long long* opt_action_eval, const long long* u, const float* avail_u, const float* r,
                              const float* terminated, const float* padded, float gamma, float lambda_opt,
                              float lambda_nopt, float* d_joint_q, float* d_v, float* dq, float* scalars,
                              float* loss_parts, void* stream);

/* ---- clip_grad_norm_ + optimiser: algorithm/q_learner.py:172-173 ----
 * grads holds d/dtheta of the UN-normalised loss sum; scalars = {loss_sum, mask_sum} (after the
 * all-reduce in data-parallel runs).  g = grads/mask_sum; total_norm = ||g||_2;
 * g *= min(1, max_norm/(total_norm+1e-6)) (torch/nn/utils/clip_grad.py); grads is overwritten with the
 * clipped g (what p.grad holds after the reference's train()); loss_out[0] = loss_sum/mask_sum,
 * loss_out[1] = total_norm.  partials: workspace of marl_optim_partials() floats.
 * Launches: n <= 4096: one CTA; n <= 2^18: one thread-block cluster of 8 CTAs exchanging the partial sums of
 * squares through distributed shared memory; larger: a reduction launch + an update launch.  All deterministic.
 * Adam: the step count is `step` (>= 1), or -- when step_counter is non-NULL -- a device int32 that the
 * call itself pre-increments (so a captured CUDA graph can be replayed). */
int marl_optim_partials(void);
int marl_clip_rmsprop_step(float* params, float* grads, float* square_avg, long long n, const float* scalars,
                           float max_norm, float lr, float alpha, float eps, float* partials, float* loss_out,
                           void* stream);
int marl_clip_adam_step(float* params, float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                        const float* scalars, float max_norm, float lr, float beta1, float beta2, float eps,
                        int step, int* step_counter /*nullable, device*/, float* partials, float* loss_out,
                        void* stream);

/* ---- data parallel without a library collective: SURVEY.md section 8(e) ----
 * The one exchange of the data-parallel step -- sum of the flat [grad | loss_sum | mask_sum] buffer over the ranks -- done
 * INSIDE the clip + optimiser launch over NVLink peer memory (one GPU per process, one node):
 *   marl_peer_alloc:  cudaMalloc'd, zeroed, cudaIpc-exportable memory; every rank puts its gradient buffer
 *                     (n + 2 floats) and a flag array (2 * MARL_PEER_MAX_WORLD uint32) there;
 *   marl_peer_export / _open / _close: the 64-byte cudaIpc handle of an allocation / map a peer's allocation;
 *   marl_clip_step_peer: what marl_clip_rmsprop_step / marl_clip_adam_step do AFTER an all-reduce, but reading the
 *     W gradient buffers directly (summed in rank order on every rank: replicas stay bit-identical), between two
 *     flag barriers ("gradients complete" / "done reading").  n <= 2^18, n % 4 == 0, 16-byte aligned buffers,
 *     grads == pg->grads[pg->rank].  epoch / error: device words of the caller (zero-initialised); *error becomes 1
 *     when a peer does not arrive within ~30 s (the step's results are then invalid).  Graph-capturable. */
#define MARL_PEER_MAX_WORLD 8
#define MARL_PEER_HANDLE_BYTES 64
typedef struct marl_peer_group {
    int world, rank;
    const float* grads[MARL_PEER_MAX_WORLD];
    unsigned* flags[MARL_PEER_MAX_WORLD];
    unsigned* epoch; int* error;
} marl_peer_group;
int marl_peer_alloc(size_t bytes, void** ptr);
int marl_peer_free(void* ptr);
int marl_peer_export(const void* ptr, unsigned char* handle /* MARL_PEER_HANDLE_BYTES */);
int marl_peer_open(const unsigned char* handle, void** ptr);
int marl_peer_close(void* ptr);
int marl_clip_step_peer(int adam, float* params, float* grads, float* m1, float* m2 /*Adam only*/, long long n,
                        float max_norm, float lr, float c1 /*alpha | beta1*/, float c2 /*beta2*/, float eps,
                        int* step_counter /*Adam only, device*/, float* loss_out, const marl_peer_group* pg, void* stream);

/* 1 when the fused VDN (qmix = 0) / QMIX (qmix = 1) mixing kernel can stage the action selection (heads = 0) or the
 * selection plus the agents' fc2 heads (heads = 1) of an [N, A] problem in shared memory. */
int marl_select_fits(int qmix, int N, int A, int heads);

/* ---- dense-layer primitives (nn.Linear and its autograd duals) ----
 * The operators above call these internally; they are exported for the parity tests and tools/gemm_bench.py.
 * Row-major fp32 operands with explicit pitches (in floats), 3xTF32 on the tensor cores (csrc/tgemm.cu when the
 * operands are TMA-addressable, csrc/linear.cu otherwise).  Replace torch.nn.functional.linear and its backward
 * (network/q_network.py:17,20; network/mixer.py:45-55):
 *   marl_linear_fwd  : y[M,N]   = act(x[M,K] . w[N,K]^T + bias[N])        (bias nullable, relu 0/1)
 *   marl_linear_dgrad: dx[M,K]  = (dy[M,N] . w[N,K]) * (relu_src[M,K] > 0) (relu_src nullable)
 *   marl_linear_wgrad: dw[N,K] += dy[M,N]^T . x[M,K] ; db[N] += column sums of dy (db nullable)
 * marl_set_scratch registers a caller-owned device arena (>= 64 MB recommended) for the split weight-gradient
 * partials; without it the weight gradients fall back to the atomic kernels of csrc/linear.cu. */
int marl_set_scratch(void* device_ptr, size_t bytes);
/* 1: the row splits of every weight gradient are written to the scratch arena and added in a fixed order by a second launch
 * (bitwise reproducible gradients; measured +13 us per weight gradient at the 2s3z sizes); 0 (default; env
 * MARL_B200_DETERMINISTIC=1 flips it): they meet in fp32 atomics (run-to-run differences of 1 ulp).  Returns the previous setting. */
int marl_set_deterministic(int on);
/* routes the TMA-addressable dense layers through csrc/tgemm.cu (1) or csrc/linear.cu (0, default; env MARL_B200_TGEMM);
 * returns the previous setting.  Captured CUDA graphs keep the path they were captured with. */
int marl_tgemm_enable(int on);
/* debug: (tag, clock64) phase trace of CTA 0 of the following tgemm launches; see tools/gemm_trace.py */
int marl_tgemm_trace(int on, long long* host_out /* 2048 words or NULL */);
int marl_linear_fwd(const float* x, int ldx, const float* w, int ldw, const float* bias, float* y, int ldy,
                    int M, int N, int K, int relu, void* stream);
int marl_linear_dgrad(const float* dy, int lddy, const float* w, int ldw, const float* relu_src, int ldrs, float* dx,
                      int lddx, int M, int N, int K, void* stream);
int marl_linear_wgrad(const float* dy, int lddy, const float* x, int ldx, float* dw, int ldw, float* db, int M, int N,
                      int K, void* stream);

/* ---- built-in launch profiler (bench.py roofline leg) ----
 * When enabled, every kernel launch of the library is bracketed by CUDA events on its stream.
 * marl_profile_collect synchronises the device and writes "kernel,count,total_ms\n" lines. */
/* FP32 FMA throughput probe (the compute-roofline denominator bench.py reports against):
 * launches `blocks` x 256 threads x 8 independent FMA chains x `iters`; *flops_out = FLOPs issued. */
int marl_fma_probe(float* scratch_device, int iters, int blocks, double* flops_out_host, void* stream);
/* Fused input layers of the agent unroll (csrc/front.cu: fc1 -> ReLU -> W_ih of every stream of marl_agent_unroll_fwd in one
 * persistent launch; default on, MARL_B200_FRONT=0 turns it off).  Returns the previous setting.  No reference counterpart. */
int marl_front_enable(int on);
/* 1 when [p, p + bytes) is page-locked host memory the current device can read in place (the host pointer is the device
 * pointer), else 0.  No reference counterpart: lets ReplayBuffer.store_episode (common/replaybuffer.py:30-61) hand pinned
 * episode arrays to marl_ingest_f64 without a staging copy. */
int marl_host_registered(const void* p, size_t bytes);
/* The same for n ranges in one call: 1 when all of them qualify. */
int marl_host_registered_all(const void* const* p, const size_t* bytes, int n);
/* Occupies the stream for ~us microseconds (<= 100000) so that later launches queue up behind it. */
int marl_spin_us(int us, void* stream);
int marl_profile_enable(int on);
int marl_profile_collect(char* buf_host, int buflen);
/* "kernel,start_us,end_us\n" per recorded launch, relative to the first one; records are kept. */
int marl_profile_timeline(char* buf_host, int buflen);

#ifdef __cplusplus
}
#endif
#endif /* MARL_B200_H */
