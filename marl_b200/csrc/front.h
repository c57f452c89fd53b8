// Internal (non-ABI): fused input layers of the recurrent agent (csrc/front.cu).
#pragma once
#include "linear.h"

namespace marl {

constexpr int kFrontMaxStreams = 4;

struct FrontStream {
    LinOperand in;          // [rows, I] agent input (composite [obs | last action | agent id] or plain)
    float* x;               // [rows, 64]  relu(fc1(in))
    float* gi;              // [rows, 192] W_ih x + b_ih
    int vec_in;             // 128-bit loads legal on the first source
    int store_x;            // x is only needed by the backward pass: streams that record no gates skip its 256 B per row
};

// streams that share one parameter set (eval on o and on o_next; target on o_next) are served by the same CTAs
struct FrontSet {
    const float* w1; const float* b1; const float* w_ih; const float* b_ih;
    int vec_w1;
    int n_streams; int stream[kFrontMaxStreams];
    int cta0, n_ctas;       // CTAs [cta0, cta0 + n_ctas) of the grid work on this set
    float* w_ih_t;          // [64, 192] or null: W_ih transposed for the backward's data gradient, written by this set's CTAs
};

struct FrontArgs {
    FrontStream s[kFrontMaxStreams];
    FrontSet set[kFrontMaxStreams];
    int n_sets;
    int rows;               // rows per stream
    int I;                  // input width (<= 256)
    int hidden;             // rnn_hidden_dim: the kernel is built for 64 and declines any other width
    int tiles_per_stream;
    long long* trace;       // debug phase trace of CTA 0 (marl_tgemm_trace), else null
};

bool front_enabled();
// false: the shapes do not qualify (I > 256, hidden != 64, misaligned outputs) -- the caller runs the layers one by one.
// budget: 0 = up to one CTA per SM; > 0 = at most that many CTAs, trimmed to the fewest that keep the tiles per CTA
bool front_plan(FrontArgs& a, int n_streams, int budget = 0);
int front_launch(const FrontArgs& a, int n_streams, int prio, cudaStream_t st);

}  // namespace marl
