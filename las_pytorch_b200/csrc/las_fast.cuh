// LAS_MODE_BF16 path: tcgen05 / cluster / persistent kernels (fast_*.cu).  Internal interface used by las_api.cu.
#pragma once
#include <cuda.h>

#include "las_common.cuh"

namespace las {

bool fast_listener_fits(const las_listener_dims* d);
size_t fast_listener_packed_bytes(const las_listener_dims* d);
int fast_listener_pack(const las_lstm_weights* w_host, const las_listener_dims* d, void* packed, bool f16, cudaStream_t st);
size_t fast_listener_workspace_bytes(const las_listener_dims* d);
int fast_listener_forward(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d, float* enc,
                          int32_t* enc_lengths, void* ws, bool f16, cudaStream_t st);

bool fast_speller_fits(const las_speller_dims* d);
size_t fast_speller_packed_bytes(const las_speller_dims* d);
int fast_speller_pack(const las_speller_weights* w, const las_speller_dims* d, void* packed_fast, bool f16, cudaStream_t st);
size_t fast_speller_workspace_bytes(const las_speller_dims* d);
// What the persistent decoder reads from the fp32 block of the speller's pack and workspace (layout: las_api.cu speller_layout)
struct SpellerF32Inputs {
  const float *b_phi, *b_psi, *b_cd;
  float* psi;  // [B, U, D] psi(enc), computed here when the caller passes no io->psi
};
int fast_speller_decode(const las_decode_io* io, const SpellerF32Inputs& f32, const void* packed_fast, const las_speller_dims* d, int steps,
                        int decode_mode, int relu, void* ws_fast, bool f16, cudaStream_t st);

// segments / launch groups of the persistent decoder (fast_speller.cu), stages of the listener (fast_listener.cu), and the
// serving pipeline that interleaves them (fast_pipeline.cu)
int fast_speller_decode_segment(const las_decode_io* io, const SpellerF32Inputs& f32, const void* packed_fast, const las_speller_dims* d,
                                int b0, int Bc, int s_begin, int s_count, bool first_seg, bool last_seg, int decode_mode, int relu,
                                void* ws_fast, bool f16, bool beside, cudaStream_t st);  // beside: shares the chip with the listener
int fast_speller_max_group(const las_speller_dims* d);
int fast_speller_ctas(const las_speller_dims* d, bool beside);  // CTAs of one persistent launch covering d->B utterances
int fast_listener_stage(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d, float* enc,
                        int32_t* enc_lengths, void* ws, int stage, int bc, int* resident, int max_ctas, bool f16, cudaStream_t st);
int fast_listener_rec_ctas(const las_listener_dims* d, int bc);
int fast_side_stream(cudaStream_t* s);
struct PipePlan {
  int bc;       // the recurrence's batch chunk (16 / 32 / 64); 0: the listener does not fit next to the decoder
  bool beside;  // the listener's stages run beside ONE decoder launch; otherwise the decoder is cut into segments around the GEMMs
};
PipePlan fast_pipeline_plan(const las_listener_dims* ld, const las_speller_dims* sd, int steps);
int fast_pipeline_step(const las_decode_io* io, const SpellerF32Inputs& spl_f32, const void* spl_packed_fast, const las_speller_dims* sd,
                       int steps, int decode_mode, int relu, void* spl_ws_fast, const float* x, const int32_t* x_lengths, const void* lis_packed,
                       const las_listener_dims* ld, float* enc, int32_t* enc_lengths, void* lis_ws, bool f16, cudaStream_t st);

// fast_gemm.cu
int launch_gemm_bf16_tc(const __nv_bfloat16* A, long long lda, const __nv_bfloat16* W, long long ldw, const float* bias, float* C,
                        long long ldc, int M, int N, int K, bool f16, cudaStream_t st, bool relu = false);
// Listener input projection with a time-major output: A is the layer input [B, Tl, K] (bf16, row pitch K, utterance pitch
// Tl*K) read through a 3-D tensor map, row r = t*Bp + b of C [Tl*Bp, N] (Bp = listener_padded_batch(B)).  Tiles are
// issued in the order the recurrence consumes them (front time steps with the forward direction's columns, back time steps
// with the backward direction's); `flags` (nullable, [m_tiles*n_tiles] zeroed counters) get +1 per finished epilogue warp
// (4 per tile).  max_ctas > 0 limits the persistent grid (the recurrence runs concurrently on the other SMs).
int listener_padded_batch(int B);
int launch_gemm_listener(const __nv_bfloat16* A, int B, int Tl, int K, const __nv_bfloat16* W, const float* bias, float* C, int N,
                         uint32_t* flags, int max_ctas, bool f16, cudaStream_t st);
int launch_umma_probe(const void* A, const void* B, float* D, int N, int K, int a_sw128, int b_sw128, int variant, cudaStream_t st);
int launch_f32_to_bf16(const float* src, __nv_bfloat16* dst, size_t n, bool f16, cudaStream_t st);
int make_tmap_bf16_box(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows);
int make_tmap_bf16_nd(CUtensorMap* tm, const void* base, int rank, const unsigned long long* dims, const unsigned long long* strides,
                      const unsigned* box);

// gen_step.cu: fused generic decoder step (stacked-cell layer = one launch; see the file header)
struct GenStepMaps {
  CUtensorMap w, a[2];  // packed weights [R, Kp]; the layer's operand rows [B, Kp] of even / odd steps (per-stage box)
  CUtensorMap a_ind[2], a_dep[2];  // the same rows, one box for all independent / all dependent K blocks
};
int gen_step_make_maps(GenStepMaps* m, const __nv_bfloat16* w, const __nv_bfloat16* act0, const __nv_bfloat16* act1, int H, int G, int B, int Kxp,
                       int Kp);
int launch_gen_cell_step(const GenStepMaps& m, int parity, const float* bias, float* c, const float* h_prev, long long h_ld, float* h_out,
                         long long hout_ld, __nv_bfloat16* o1, long long o1_ld, __nv_bfloat16* o2, long long o2_ld, int B, int H, int cell,
                         int Kxp, int Kp, bool pdl, bool f16, cudaStream_t st, int trace_slot = 0);

}  // namespace las
