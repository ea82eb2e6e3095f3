// Internal launch-function declarations shared between translation units.
#pragma once
#include <cuda_bf16.h>
#include "las_common.cuh"

namespace las {

// ---- fp32 (LAS_MODE_FP32) kernels: kernels_f32.cu ------------------------------------------------------

// C[M,N] = act(A[M,K] . W[N,K]^T + bias[N]);  A row stride lda, W row stride ldw, C row stride ldc.
int launch_sgemm_nt_bias(const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                         int M, int N, int K, bool relu, cudaStream_t st);

// One recurrent cell update for a batch.  x part: [x . W_ih^T] + [pre_add] + [b_ih]; h part: [h_prev . W_hh^T] + [b_hh].
// LSTM (4 gates i,f,g,o) and RNN (1 gate, tanh) use x part + h part; GRU (r,z,n) keeps them apart for the n gate:
// n = tanh(x_n + r * h_n), h' = (1 - z) * n + z * h_prev (torch nn.GRU).
struct CellArgs {
  const float* x;       // nullable, [B, Kx] row stride x_ld
  int x_ld, Kx;
  const float* w_ih;    // [4H, Kx]
  const float* h_prev;  // nullable (== zeros), [B, H] row stride h_ld
  long long h_ld;
  const float* w_hh;    // [4H, H]
  const float* pre_add; // nullable, [B, 4H] row stride pre_ld (already contains the biases)
  long long pre_ld;
  const float* b_ih;    // nullable
  const float* b_hh;    // nullable
  float* c;             // [B, H] in/out, dense
  float* h_out;         // [B, H] row stride hout_ld
  long long hout_ld;
  const int32_t* lengths;  // nullable [B]: rows with t >= lengths[b] keep c and write h = 0 (length-mask extension)
  int t;
};
int launch_lstm_cell_f32(const CellArgs* args, int ndir, int B, int H, cudaStream_t st, int cell = 0);

struct AttendArgs {
  const float* state;   // [B, Hs] row stride state_ld : top-layer decoder state
  int state_ld;
  const float* enc;     // [B, U, E]
  const float* psi;     // [B, U, D]
  const float* w_phi;   // [D, Hs]
  const float* b_phi;
  const float* w_cd;    // [V, Hs+E]   (nullable => attention only)
  const float* b_cd;
  const int32_t* enc_lengths;  // nullable
  int B, U, E, Hs, V, D;
  int rows_per_utt;     // 0 or 1: one decoder row per utterance; R > 1: rows b*R .. b*R+R-1 share enc / psi / enc_lengths of utterance b
  int relu;
  int heads;            // >= 1; phi has D*heads outputs, each head attends over the same psi
  const float* w_dr;    // [E, E*heads] (heads > 1)
  const float* b_dr;    // [E]
  // outputs
  float* score_out;     // nullable, [heads, B, U]
  float* ctx_out;       // [B, E] row stride ctx_ld
  int ctx_ld;
  float* logp_out;      // [B, V]     (when w_cd)
  int32_t* token_out;   // nullable [B]
  // next-step input word (when w_cd): one of gt_dense row / gt_index / greedy / raw
  float* word_out;      // nullable [B, V] row stride word_ld
  int word_ld;
  const float* gt_dense_step;   // nullable [B, V] row stride gt_ld (already offset to this step)
  long long gt_ld;
  const int32_t* gt_index_step; // nullable [B] stride gt_index_ld
  int gt_index_ld;
  int decode_mode;
  unsigned long long sample_seed;  // LAS_DECODE_SAMPLE
  int step;
  const int32_t* nll_label_step;  // nullable [B] stride nll_label_ld: label of this step for the fused NLL term
  int nll_label_ld;
  float* nll_term_out;            // nullable [B]
  // generic tensor-core path: the next step's layer-0 GEMM operand row [word V | context E] in the 16-bit operand format
  __nv_bfloat16* op_out;          // nullable [B, >= V+E] row stride op_ld
  long long op_ld;
  int op_f16;
  long long* trace;               // nullable test hook (attend_cluster_kernel): clock64 stamps of CTA 0
};
int launch_attend_f32(const AttendArgs& a, cudaStream_t st);
// same step, heads == 1: a cluster of C = 1 / 2 / 4 / 8 CTAs per utterance (gen_step.cu); pdl = programmatic dependent launch
constexpr int AC_THREADS = 512;  // its threads read 16-byte aligned encoder rows four features each: E <= 4 * AC_THREADS
int launch_attend_cluster(const AttendArgs& a, int C, bool pdl, cudaStream_t st);

// xin[b, 0:V] = onehot(0), xin[b, V:V+E] = enc[b, 0, :]   (model/las_model.py:193-198)
int launch_speller_init(float* xin, int xin_ld, const float* enc, int B, int U, int E, int V, cudaStream_t st);
// strided 2-D copy of fp32 rows
int launch_copy2d(float* dst, long long dst_ld, const float* src, long long src_ld, int rows, int cols, cudaStream_t st);

// out[b] = (in[b] + 1) / 2, clamped to [0, cap]: valid steps of the next pyramid layer
int launch_pyramid_lengths(const int32_t* in, int32_t* out, int B, int cap, cudaStream_t st);

int launch_nll_sums(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len,
                    float* out2, cudaStream_t st);

// generic tensor-core decoder step (LAS_MODE_BF16 beyond the persistent decoder's shapes; kernels_f32.cu)
int launch_gen_pack_w(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, __nv_bfloat16* dst, float* bias, int cell,
                      int H, int Kx, int Kxp, int Kp, bool f16, cudaStream_t st);
int launch_gen_build_a(const float* x, long long x_ld, const float* h, long long h_ld, __nv_bfloat16* A, int B, int H, int Kx, int Kxp, int Kp,
                       bool f16, cudaStream_t st);
int launch_gen_cell(const float* pre, long long ldb, long long ldr, const float* bias, const float* h_prev, long long h_ld, float* c, float* h_out,
                    long long hout_ld, int B, int H, int cell, cudaStream_t st);

// beam search (beam_search.cu): B utterances of K rows each
// xin[r, 0:V] = onehot(0), xin[r, V:V+E] = enc[r / K, 0, :]; score[r] = 0 for r % K == 0, else -inf; fin[r] = 0
int launch_beam_init(float* xin, int xin_ld, const float* enc, float* score, int32_t* fin, int B, int K, int U, int E, int V, cudaStream_t st);
struct BeamStepArgs {
  const float* logp;       // [B*K, V] this step's log-probabilities
  float* score;            // [B*K] in/out
  int32_t* fin;            // [B*K] in/out: the row has emitted eos
  int32_t* parent;         // [B, K] this step's back-pointers (slice of [S, B, K])
  int32_t* token;          // [B, K]
  float* token_logp;       // [B, K]
  float* h;                // [sl, B*K, Hs] the state the next step reads; permuted in place
  float* c;                // nullable [sl, B*K, Hs]
  float* xin;              // [B*K, xld]: word [V] | context [E]; word written, context permuted
  int xld;
  int B, K, V, E, Hs, sl, eos;
};
int launch_beam_step(const BeamStepArgs& a, cudaStream_t st);
struct BeamFinalArgs {
  const float* score;      // [B*K]
  const int32_t* parent;   // [S, B, K]
  const int32_t* token;
  const float* token_logp;
  int32_t* tokens_out;     // [B, N, S]
  float* token_logp_out;   // nullable [B, N, S]
  int32_t* lengths_out;    // [B, N]
  float* scores_out;       // [B, N]
  int32_t* src_rows;       // nullable [B, N, S_out]: decoder row (b*K + parent) of each token's step, -1 from the length on
  int B, K, N, eos;
  int S_run;               // steps run: the back-pointers hold S_run steps (every row has ended if S_run < S_out)
  int S_out;               // steps of the outputs; [S_run, S_out) is padded with eos / 0
  float alpha;
};
int launch_beam_finalize(const BeamFinalArgs& a, cudaStream_t st);
// attn [B, N, S, heads, U] from the per-step attention of every decoder row, work [S, heads, B*K, U], along src_rows [B, N, S]
int launch_beam_attention_trace(const float* work, const int32_t* src_rows, float* attn, int B, int K, int N, int S, int heads, int U,
                                cudaStream_t st);
// *steps_done = step if every fin[0 .. n) is set; otherwise *steps_done is left unchanged
int launch_beam_all_ended(const int32_t* fin, int n, int step, int32_t* steps_done, cudaStream_t st);

// <eos> early exit bookkeeping (las_decode_io.early_exit): `state` = 66 int32 {stop, steps decoded, done[64]} per launch group
int launch_eos_check(const int32_t* tokens, int Bfull, int b0, int Bc, int s_begin, int s_end, int eos, int32_t* state, cudaStream_t st);
int launch_eos_fill(const int32_t* state, int S, int Bfull, int b0, int Bc, int V, int U, int heads, int eos, float* logp, float* attn, int32_t* tokens,
                    float* nll_terms, int32_t* steps_done, cudaStream_t st);
int launch_label_smoothing(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len, float ls,
                           float* per_utt, cudaStream_t st);

}  // namespace las
