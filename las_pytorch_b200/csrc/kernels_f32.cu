// LAS_MODE_FP32 kernels: fp32 operands, fp32 FMA accumulation, precise expf/tanhf.
// This is the correctness mode (north_star: log-probs within 1e-4 of the reference); it is also the first CUDA
// path every faster kernel is validated against.  Kernels here are straightforward CUDA-core code.
#include <cuda_bf16.h>

#include "las_kernels.cuh"
#include "attend_tail.cuh"

namespace las {

// =========================================================================================================
// SGEMM  C = act(A . W^T + bias)     (reference: the x.W_ih^T half of nn.LSTM, model/las_model.py:90, and
//                                     TimeDistributed(psi), model/las_model.py:279)
// 128x128x16 tile, 256 threads, 8x8 register micro-tile (split 4+4 so smem reads are float4 and conflict-free).
// =========================================================================================================
constexpr int GM = 128, GN = 128, GK = 16;

__global__ void __launch_bounds__(256)
sgemm_nt_bias_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W, int ldw,
                     const float* __restrict__ bias, float* __restrict__ C, int ldc, int M, int N, int K, int relu,
                     int vec_ok) {
  __shared__ __align__(16) float As[GK][GM + 4];
  __shared__ __align__(16) float Ws[GK][GN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += GK) {
    // stage A and W tiles (transposed into [k][row])
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = tid + i * 256;
      const int row = idx >> 2, kq = (idx & 3) * 4;
      float va[4] = {0.f, 0.f, 0.f, 0.f}, vw[4] = {0.f, 0.f, 0.f, 0.f};
      const int gm = m0 + row, gn = n0 + row, gk = k0 + kq;
      if (gm < M) {
        const float* p = A + (size_t)gm * lda + gk;
        if (vec_ok && gk + 3 < K) {
          const float4 t = *reinterpret_cast<const float4*>(p);
          va[0] = t.x; va[1] = t.y; va[2] = t.z; va[3] = t.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) if (gk + j < K) va[j] = p[j];
        }
      }
      if (gn < N) {
        const float* p = W + (size_t)gn * ldw + gk;
        if (vec_ok && gk + 3 < K) {
          const float4 t = *reinterpret_cast<const float4*>(p);
          vw[0] = t.x; vw[1] = t.y; vw[2] = t.z; vw[3] = t.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) if (gk + j < K) vw[j] = p[j];
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        As[kq + j][row] = va[j];
        Ws[kq + j][row] = vw[j];
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Ws[kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Ws[kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (gn >= N) continue;
      float v = acc[i][j] + (bias ? bias[gn] : 0.f);
      if (relu) v = fmaxf(v, 0.f);
      C[(size_t)gm * ldc + gn] = v;
    }
  }
}

int launch_sgemm_nt_bias(const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                         int M, int N, int K, bool relu, cudaStream_t st) {
  if (M <= 0 || N <= 0) return LAS_OK;
  const int vec_ok = (lda % 4 == 0) && (ldw % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
  dim3 grid((N + GN - 1) / GN, (M + GM - 1) / GM);
  sgemm_nt_bias_kernel<<<grid, 256, 0, st>>>(A, lda, W, ldw, bias, C, ldc, M, N, K, relu ? 1 : 0, vec_ok);
  LAS_LAUNCH_OK("sgemm_nt_bias_kernel");
  return LAS_OK;
}

// =========================================================================================================
// LSTM cell step (torch nn.LSTM equations, gate order i,f,g,o).  Used for the listener recurrence
// (model/las_model.py:90; pre_add = the precomputed input projection, one launch per time step covering both
// directions) and for the speller's stacked cells (model/las_model.py:179).
// Tile: 32 batch rows x 8 hidden units (x4 gates), K streamed in chunks of 32 through smem.
// =========================================================================================================
constexpr int CB = 32, CJ = 8, CK = 32;

struct CellArgs2 {
  CellArgs d[2];
};

__device__ __forceinline__ void cell_accumulate(const float* __restrict__ src, long long src_ld, int K,
                                                const float* __restrict__ w, int H, int b0, int j0, int B, int G,
                                                float (&As)[CB][CK + 1], float (&Ws)[4 * CJ][CK + 1], float (&acc)[4]) {
  const int tid = threadIdx.x;
  const int tb = tid / CJ, tj = tid % CJ;
  for (int k0 = 0; k0 < K; k0 += CK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      const int r = idx / CK, cc = idx % CK;
      const int gk = k0 + cc;
      const int gb = b0 + r;
      As[r][cc] = (gb < B && gk < K) ? src[(long long)gb * src_ld + gk] : 0.f;
      const int g = r / CJ, jj = r % CJ;
      const int gj = j0 + jj;
      Ws[r][cc] = (g < G && gj < H && gk < K) ? w[(size_t)(g * H + gj) * K + gk] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < CK; ++kk) {
      const float av = As[tb][kk];
#pragma unroll
      for (int g = 0; g < 4; ++g) acc[g] = fmaf(av, Ws[g * CJ + tj][kk], acc[g]);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) lstm_cell_f32_kernel(CellArgs2 args, int B, int H, int cell) {
  const CellArgs& a = args.d[blockIdx.z];
  __shared__ float As[CB][CK + 1];
  __shared__ float Ws[4 * CJ][CK + 1];
  const int j0 = blockIdx.x * CJ, b0 = blockIdx.y * CB;
  const int G = cell == LAS_CELL_LSTM ? 4 : (cell == LAS_CELL_GRU ? 3 : 1);
  float ax[4] = {0.f, 0.f, 0.f, 0.f}, ah[4] = {0.f, 0.f, 0.f, 0.f};  // x part / h part of the gate pre-activations
  if (a.x) cell_accumulate(a.x, a.x_ld, a.Kx, a.w_ih, H, b0, j0, B, G, As, Ws, ax);
  if (a.h_prev) cell_accumulate(a.h_prev, a.h_ld, H, a.w_hh, H, b0, j0, B, G, As, Ws, ah);

  const int tb = threadIdx.x / CJ, tj = threadIdx.x % CJ;
  const int b = b0 + tb, j = j0 + tj;
  if (b >= B || j >= H) return;
  if (a.lengths && a.t >= a.lengths[b]) {  // padded step: state untouched, output zero
    a.h_out[(long long)b * a.hout_ld + j] = 0.f;
    return;
  }
  const int GH = G * H;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (g < G) {
      if (a.pre_add) ax[g] += a.pre_add[(long long)b * a.pre_ld + g * H + j];
      if (a.b_ih) ax[g] += a.b_ih[g * H + j];
      if (a.b_hh) ah[g] += a.b_hh[g * H + j];
    }
  }
  (void)GH;
  if (cell == LAS_CELL_LSTM) {
    const float ig = sigmoid_precise(ax[0] + ah[0]);
    const float fg = sigmoid_precise(ax[1] + ah[1]);
    const float gg = tanhf(ax[2] + ah[2]);
    const float og = sigmoid_precise(ax[3] + ah[3]);
    const float c_new = fg * a.c[(size_t)b * H + j] + ig * gg;
    a.c[(size_t)b * H + j] = c_new;
    a.h_out[(long long)b * a.hout_ld + j] = og * tanhf(c_new);
  } else if (cell == LAS_CELL_GRU) {
    const float hp = a.h_prev ? a.h_prev[(long long)b * a.h_ld + j] : 0.f;
    const float rg = sigmoid_precise(ax[0] + ah[0]);
    const float zg = sigmoid_precise(ax[1] + ah[1]);
    const float ng = tanhf(ax[2] + rg * ah[2]);
    a.h_out[(long long)b * a.hout_ld + j] = (1.0f - zg) * ng + zg * hp;
  } else {
    a.h_out[(long long)b * a.hout_ld + j] = tanhf(ax[0] + ah[0]);
  }
}

__global__ void pyramid_lengths_kernel(const int32_t* in, int32_t* out, int B, int cap) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) out[b] = min(max((in[b] + 1) / 2, 0), cap);
}
int launch_pyramid_lengths(const int32_t* in, int32_t* out, int B, int cap, cudaStream_t st) {
  pyramid_lengths_kernel<<<(B + 127) / 128, 128, 0, st>>>(in, out, B, cap);
  LAS_LAUNCH_OK("pyramid_lengths_kernel");
  return LAS_OK;
}

int launch_lstm_cell_f32(const CellArgs* args, int ndir, int B, int H, cudaStream_t st, int cell) {
  CellArgs2 a2;
  a2.d[0] = args[0];
  a2.d[1] = args[ndir > 1 ? 1 : 0];
  dim3 grid((H + CJ - 1) / CJ, (B + CB - 1) / CB, ndir);
  lstm_cell_f32_kernel<<<grid, 256, 0, st>>>(a2, B, H, cell);
  LAS_LAUNCH_OK("lstm_cell_f32_kernel");
  return LAS_OK;
}

// =========================================================================================================
// Attention + character distribution + feedback for one decoder step; one CTA per utterance.
// model/las_model.py:276-297 (phi, energy, softmax, context), :181-182 (cat, Linear, LogSoftmax),
// :216-227 (teacher forcing / raw / greedy feedback), :236 (next input = [word || context]).
// smem: state[Hs] q[D] score[U] vec[Hs+E] logits[V] red[32]
// =========================================================================================================
__global__ void __launch_bounds__(1024) attend_f32_kernel(AttendArgs a) {
  extern __shared__ float sm[];
  const int NH = a.heads;
  float* s_state = sm;                 // Hs
  float* s_q = s_state + a.Hs;         // D * heads
  float* s_score = s_q + a.D * NH;     // U
  float* s_ctx = s_score + a.U;        // E
  float* s_logit = s_ctx + a.E;        // V
  float* s_red = s_logit + a.V;        // 32
  float* s_ctxh = s_red + 32;          // E * heads (heads > 1 only)
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;

  for (int k = tid; k < a.Hs; k += blockDim.x) s_state[k] = a.state[(size_t)b * a.state_ld + k];
  __syncthreads();

  // q = act(W_phi . state + b_phi)   (:278); D*heads outputs, split per head below (:303-305)
  if (!a.w_phi) {  // use_mlp_in_attention=False (:283-285): query is the raw decoder state
    for (int d = tid; d < a.D; d += blockDim.x) s_q[d] = s_state[d];
  }
  for (int d = wid; a.w_phi && d < a.D * NH; d += nw) {
    const float* wr = a.w_phi + (size_t)d * a.Hs;
    float p = 0.f;
    for (int k = lane; k < a.Hs; k += 32) p = fmaf(wr[k], s_state[k], p);
    p = warp_sum(p);
    if (lane == 0) {
      p += a.b_phi[d];
      s_q[d] = a.relu ? fmaxf(p, 0.f) : p;
    }
  }
  __syncthreads();

  const int bu = a.rows_per_utt > 1 ? b / a.rows_per_utt : b;  // the utterance whose encoder features row b attends over
  const int ulen = a.enc_lengths ? min(max(a.enc_lengths[bu], 1), a.U) : a.U;
  const float* psib = a.psi + (size_t)bu * a.U * a.D;
  const float* encb = a.enc + (size_t)bu * a.U * a.E;
  for (int hd = 0; hd < NH; ++hd) {
    // energy[u] = <q_head, psi[b,u,:]>   (:289-291 / :299-305)
    const float* qh = s_q + hd * a.D;
    for (int u = wid; u < a.U; u += nw) {
      const float* pr = psib + (size_t)u * a.D;
      float p = 0.f;
      for (int d = lane; d < a.D; d += 32) p = fmaf(qh[d], pr[d], p);
      p = warp_sum(p);
      if (lane == 0) s_score[u] = (u < ulen) ? p : -INFINITY;
    }
    __syncthreads();

    // softmax over U   (:292)
    float m = -INFINITY;
    for (int u = tid; u < a.U; u += blockDim.x) m = fmaxf(m, s_score[u]);
    m = block_reduce_max(m, s_red);
    float ssum = 0.f;
    for (int u = tid; u < a.U; u += blockDim.x) {
      const float e = expf(s_score[u] - m);
      s_score[u] = e;
      ssum += e;
    }
    ssum = block_reduce_sum(ssum, s_red);
    const float inv = 1.0f / ssum;
    for (int u = tid; u < a.U; u += blockDim.x) {
      const float p = s_score[u] * inv;
      s_score[u] = p;
      if (a.score_out) a.score_out[((size_t)hd * a.B + b) * a.U + u] = p;
    }
    __syncthreads();

    // context[e] = sum_u score[u] * enc[b,u,e]   (:293-297 / :306-312)
    for (int e = tid; e < a.E; e += blockDim.x) {
      float acc = 0.f;
      int u = 0;
      for (; u + 8 <= a.U; u += 8) {  // eight rows in flight; the sum keeps its u-ascending order
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = encb[(size_t)(u + j) * a.E + e];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc = fmaf(s_score[u + j], x[j], acc);
      }
      for (; u < a.U; ++u) acc = fmaf(s_score[u], encb[(size_t)u * a.E + e], acc);
      if (NH == 1) {
        s_ctx[e] = acc;
        a.ctx_out[(size_t)b * a.ctx_ld + e] = acc;
        if (a.op_out) a.op_out[(size_t)b * a.op_ld + a.V + e] = op_from_f32(acc, a.op_f16);
      } else {
        s_ctxh[hd * a.E + e] = acc;
      }
    }
    __syncthreads();
  }
  if (NH > 1) {  // context = dim_reduce(cat(per-head contexts))   (:313)
    const int KR = a.E * NH;
    for (int e = wid; e < a.E; e += nw) {
      const float* wr = a.w_dr + (size_t)e * KR;
      float p = 0.f;
      for (int k = lane; k < KR; k += 32) p = fmaf(wr[k], s_ctxh[k], p);
      p = warp_sum(p);
      if (lane == 0) {
        p += a.b_dr[e];
        s_ctx[e] = p;
        a.ctx_out[(size_t)b * a.ctx_ld + e] = p;
        if (a.op_out) a.op_out[(size_t)b * a.op_ld + a.V + e] = op_from_f32(p, a.op_f16);
      }
    }
  }
  if (!a.w_cd) return;
  __syncthreads();

  // logits = W_cd . [state || context] + b_cd ; log_softmax   (:181-182)
  const int KC = a.Hs + a.E;
  for (int v = wid; v < a.V; v += nw) {
    const float* wr = a.w_cd + (size_t)v * KC;
    float p = 0.f;
    for (int k = lane; k < a.Hs; k += 32) p = fmaf(wr[k], s_state[k], p);
    for (int k = lane; k < a.E; k += 32) p = fmaf(wr[a.Hs + k], s_ctx[k], p);
    p = warp_sum(p);
    if (lane == 0) s_logit[v] = p + a.b_cd[v];
  }
  __syncthreads();
  attend_tail(a, b, s_logit, s_red);
}

int launch_attend_f32(const AttendArgs& a, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((size_t)a.Hs + (size_t)a.D * a.heads + a.U + a.E + a.V + 32 + (a.heads > 1 ? (size_t)a.E * a.heads : 0));
  if (smem > 200 * 1024) return fail(LAS_EINVAL, "attention step needs %zu bytes of shared memory (U=%d too long)", smem, a.U);
  if (smem > 48 * 1024) {
    LAS_CUDA_OK(cudaFuncSetAttribute(attend_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  // one CTA per utterance; wide models get more warps (one context feature per thread, more rows of W_phi / W_cd / psi in flight)
  const int threads = (a.E >= 1024 || a.Hs >= 1024) ? 1024 : (a.E >= 512 ? 512 : 256);
  attend_f32_kernel<<<a.B, threads, smem, st>>>(a);
  LAS_LAUNCH_OK("attend_f32_kernel");
  return LAS_OK;
}

// =========================================================================================================
__global__ void speller_init_kernel(float* xin, int xin_ld, const float* enc, int B, int U, int E, int V) {
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < V + E; i += blockDim.x) {
    float v;
    if (i < V) v = (i == 0) ? 1.f : 0.f;              // <sos> one-hot, utils/functions.py:54-63
    else v = enc[(size_t)b * U * E + (i - V)];         // listener_feature[:, 0, :], model/las_model.py:198
    xin[(size_t)b * xin_ld + i] = v;
  }
}
int launch_speller_init(float* xin, int xin_ld, const float* enc, int B, int U, int E, int V, cudaStream_t st) {
  speller_init_kernel<<<B, 128, 0, st>>>(xin, xin_ld, enc, B, U, E, V);
  LAS_LAUNCH_OK("speller_init_kernel");
  return LAS_OK;
}

__global__ void copy2d_kernel(float* dst, long long dst_ld, const float* src, long long src_ld, int rows, int cols) {
  const long long n = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols, c = i % cols;
    dst[r * dst_ld + c] = src[r * src_ld + c];
  }
}
int launch_copy2d(float* dst, long long dst_ld, const float* src, long long src_ld, int rows, int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return LAS_OK;
  const long long n = (long long)rows * cols;
  const int blocks = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
  copy2d_kernel<<<blocks, 256, 0, st>>>(dst, dst_ld, src, src_ld, rows, cols);
  LAS_LAUNCH_OK("copy2d_kernel");
  return LAS_OK;
}

// solver/solver.py:62,70-77: NLLLoss(ignore_index=0) numerator / denominator, deterministic single-CTA reduce.
__global__ void nll_sums_kernel(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int L,
                                float* out2) {
  __shared__ float red[32];
  float num = 0.f, den = 0.f;
  for (int i = threadIdx.x; i < B * L; i += blockDim.x) {
    const int b = i / L, s = i % L;
    const int lab = labels[(size_t)b * S_lab + s];
    if (lab != 0 && lab < V) {
      num -= logp[((size_t)s * B + b) * V + lab];
      den += 1.f;
    }
  }
  num = block_reduce_sum(num, red);
  den = block_reduce_sum(den, red);
  if (threadIdx.x == 0) { out2[0] = num; out2[1] = den; }
}
int launch_nll_sums(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len,
                    float* out2, cudaStream_t st) {
  int L = max_label_len < S ? max_label_len : S;
  if (S_lab < L) L = S_lab;
  nll_sums_kernel<<<1, 1024, 0, st>>>(logp, labels, S, S_lab, B, V, L, out2);
  LAS_LAUNCH_OK("nll_sums_kernel");
  return LAS_OK;
}

// solver/solver.py:33-45 label_smoothing_loss, per utterance: sum_s [ (1-ls) logp[s,b,lab] + (ls/V) sum_v logp[s,b,v] ] / #labelled steps.
// labels < 0 mark the all-zero rows of the reference's one-hot target (no contribution); the caller takes -mean over b.
__global__ void __launch_bounds__(256) label_smoothing_kernel(const float* logp, const int32_t* labels, int S_lab, int B, int V, int L, float ls,
                                                              float* per_utt) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  float acc = 0.f, cnt = 0.f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int s = warp; s < L; s += nwarp) {  // one warp per step: coalesced read of the V log-probs
    const int lab = labels[(size_t)b * S_lab + s];
    if (lab < 0 || lab >= V) continue;
    const float* row = logp + ((size_t)s * B + b) * V;
    float sum = 0.f;
    for (int v = lane; v < V; v += 32) sum += row[v];
    sum = warp_sum(sum);
    if (lane == 0) {
      acc += (1.0f - ls) * row[lab] + (ls / (float)V) * sum;
      cnt += 1.f;
    }
  }
  acc = block_reduce_sum(acc, red);
  cnt = block_reduce_sum(cnt, red);
  if (threadIdx.x == 0) per_utt[b] = acc / cnt;  // cnt == 0 -> nan, as the reference's division by seq_len == 0
}
int launch_label_smoothing(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len, float ls,
                           float* per_utt, cudaStream_t st) {
  int L = max_label_len < S ? max_label_len : S;
  if (S_lab < L) L = S_lab;
  label_smoothing_kernel<<<B, 256, 0, st>>>(logp, labels, S_lab, B, V, L, ls, per_utt);
  LAS_LAUNCH_OK("label_smoothing_kernel");
  return LAS_OK;
}

// ---- <eos> early exit (SURVEY.md section 8 row f4; extension: the reference always runs max_label_len steps, model/las_model.py:205-209)
// After each segment: has every utterance of this launch group emitted <eos> by now?  If so, raise `stop` (the following segment
// launches return at once) and record where the group stopped.
// state [66] int32: [0] stop flag, [1] steps the group decoded, [2..66) per-utterance done flags (zeroed at the start of a group)
__global__ void eos_check_kernel(const int32_t* tokens, int Bfull, int b0, int Bc, int s_begin, int s_end, int eos, int32_t* state) {
  int32_t *stop = state, *group_steps = state + 1, *done = state + 2;
  const int b = threadIdx.x;
  int d = 1;
  if (b < Bc) {
    d = done[b];
    for (int s = s_begin; s < s_end && !d; ++s) d = tokens[(size_t)s * Bfull + b0 + b] == eos;
    done[b] = d;
  }
  const int all = __syncthreads_and(d);
  if (threadIdx.x == 0 && *stop == 0) {
    *group_steps = s_end;
    if (all) *stop = 1;
  }
}
// steps this group did not decode: tokens = <eos>, log-probs / attention = 0; steps_done (nullable) = max over the groups
__global__ void eos_fill_kernel(const int32_t* state, int S, int Bfull, int b0, int Bc, int V, int U, int heads, int eos, float* logp, float* attn,
                                int32_t* tokens, float* nll_terms, int32_t* steps_done) {
  const int s0 = state[1];
  if (blockIdx.x == 0 && threadIdx.x == 0 && steps_done) atomicMax(steps_done, s0);
  const size_t n = (size_t)(S - s0) * Bc;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int s = s0 + (int)(i / Bc), b = b0 + (int)(i % Bc);
    const size_t row = (size_t)s * Bfull + b;
    if (tokens) tokens[row] = eos;
    if (nll_terms) nll_terms[row] = 0.f;
    for (int v = 0; v < V; ++v) logp[row * V + v] = 0.f;
    if (attn)  // [S, heads, B, U]
      for (int h = 0; h < heads; ++h)
        for (int u = 0; u < U; ++u) attn[(((size_t)s * heads + h) * Bfull + b) * U + u] = 0.f;
  }
}

int launch_eos_check(const int32_t* tokens, int Bfull, int b0, int Bc, int s_begin, int s_end, int eos, int32_t* state, cudaStream_t st) {
  eos_check_kernel<<<1, 64, 0, st>>>(tokens, Bfull, b0, Bc, s_begin, s_end, eos, state);
  LAS_LAUNCH_OK("eos_check_kernel");
  return LAS_OK;
}
int launch_eos_fill(const int32_t* state, int S, int Bfull, int b0, int Bc, int V, int U, int heads, int eos, float* logp, float* attn, int32_t* tokens,
                    float* nll_terms, int32_t* steps_done, cudaStream_t st) {
  eos_fill_kernel<<<64, 256, 0, st>>>(state, S, Bfull, b0, Bc, V, U, heads, eos, logp, attn, tokens, nll_terms, steps_done);
  LAS_LAUNCH_OK("eos_fill_kernel");
  return LAS_OK;
}

// =========================================================================================================
// Generic tensor-core decoder step (LAS_MODE_BF16 for the shapes / variants the persistent decoder does not hold on chip:
// 1024-wide cells, GRU / RNN cells; las_api.cu speller_step): per layer and step
//     A = bf16([x | h_prev])  ->  tcgen05 GEMM with the packed [R, Kp] bf16 weights (+ bias)  ->  fp32 cell update.
// Packed rows R: LSTM 4H (i,f,g,o), RNN H, GRU 4H = (r, z, n_x, n_h) -- the n gate's input and hidden parts are kept apart
// (torch: n = tanh(W_in x + b_in + r * (W_hn h + b_hn))) by giving them separate rows with a zero block each.
// K columns: x part in [0, Kx), zero padding up to Kxp, h part in [Kxp, Kxp + H), zero padding up to Kp.
// =========================================================================================================
__global__ void gen_pack_w_kernel(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, __nv_bfloat16* dst, float* bias,
                                  int cell, int H, int Kx, int Kxp, int Kp, int f16) {
  const int R = (cell == LAS_CELL_RNN) ? H : 4 * H;
  const size_t n = (size_t)R * Kp;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % Kp), row = (int)(i / Kp);
    const int blk = row / H, j = row % H;
    float v = 0.f;
    // source gate block of this packed row, and which parts (x / h) it carries
    int src = blk;
    bool use_x = true, use_h = true;
    if (cell == LAS_CELL_GRU) {
      if (blk == 2) use_h = false;                // n_x
      if (blk == 3) { src = 2; use_x = false; }   // n_h
    }
    if (k < Kx) { if (use_x) v = w_ih[((size_t)src * H + j) * Kx + k]; }
    else if (k >= Kxp && k < Kxp + H) { if (use_h) v = w_hh[((size_t)src * H + j) * H + (k - Kxp)]; }
    dst[i] = op_from_f32(v, f16);
    if (k == 0) bias[row] = (use_x ? b_ih[src * H + j] : 0.f) + (use_h ? b_hh[src * H + j] : 0.f);
  }
}
int launch_gen_pack_w(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, __nv_bfloat16* dst, float* bias, int cell,
                      int H, int Kx, int Kxp, int Kp, bool f16, cudaStream_t st) {
  gen_pack_w_kernel<<<592, 256, 0, st>>>(w_ih, w_hh, b_ih, b_hh, dst, bias, cell, H, Kx, Kxp, Kp, f16);
  LAS_LAUNCH_OK("gen_pack_w_kernel");
  return LAS_OK;
}
// A[b, :] = bf16([x[b, 0:Kx] | 0 | h[b, 0:H] | 0]); h == nullptr reads as zeros
__global__ void gen_build_a_kernel(const float* x, long long x_ld, const float* h, long long h_ld, __nv_bfloat16* A, int B, int H, int Kx, int Kxp,
                                   int Kp, int f16) {
  const size_t n = (size_t)B * Kp;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % Kp), b = (int)(i / Kp);
    float v = 0.f;
    if (k < Kx) v = x[(long long)b * x_ld + k];
    else if (h && k >= Kxp && k < Kxp + H) v = h[(long long)b * h_ld + (k - Kxp)];
    A[i] = op_from_f32(v, f16);
  }
}
int launch_gen_build_a(const float* x, long long x_ld, const float* h, long long h_ld, __nv_bfloat16* A, int B, int H, int Kx, int Kxp, int Kp,
                       bool f16, cudaStream_t st) {
  const size_t n = (size_t)B * Kp;
  gen_build_a_kernel<<<(unsigned)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592), 256, 0, st>>>(x, x_ld, h, h_ld, A, B, H, Kx, Kxp, Kp, f16);
  LAS_LAUNCH_OK("gen_build_a_kernel");
  return LAS_OK;
}
// Gate pre-activations -> cell update in fp32.  pre(b, r) = pre[b * ldb + r * ldr] (+ bias[r] when given): either [B, R] with the
// biases already added by the GEMM's epilogue (ldb = R, ldr = 1) or the transposed [R, B] a small-batch GEMM writes (ldb = 1, ldr = B).
// h_prev nullable (zeros); c is not touched for GRU / RNN.
__global__ void gen_cell_kernel(const float* pre, long long ldb, long long ldr, const float* bias, const float* h_prev, long long h_ld, float* c,
                                float* h_out, long long hout_ld, int B, int H, int cell) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i % H;
  auto P = [&](int r) { return pre[(long long)b * ldb + (long long)r * ldr] + (bias ? bias[r] : 0.f); };
  float h;
  if (cell == LAS_CELL_LSTM) {
    const float ig = sigmoid_precise(P(j)), fg = sigmoid_precise(P(H + j)), gg = tanhf(P(2 * H + j)), og = sigmoid_precise(P(3 * H + j));
    const float cn = fg * c[(size_t)b * H + j] + ig * gg;
    c[(size_t)b * H + j] = cn;
    h = og * tanhf(cn);
  } else if (cell == LAS_CELL_GRU) {
    const float hp = h_prev ? h_prev[(long long)b * h_ld + j] : 0.f;
    const float rg = sigmoid_precise(P(j)), zg = sigmoid_precise(P(H + j));
    const float ng = tanhf(P(2 * H + j) + rg * P(3 * H + j));
    h = (1.0f - zg) * ng + zg * hp;
  } else {
    h = tanhf(P(j));
  }
  h_out[(long long)b * hout_ld + j] = h;
}
int launch_gen_cell(const float* pre, long long ldb, long long ldr, const float* bias, const float* h_prev, long long h_ld, float* c, float* h_out,
                    long long hout_ld, int B, int H, int cell, cudaStream_t st) {
  gen_cell_kernel<<<(B * H + 255) / 256, 256, 0, st>>>(pre, ldb, ldr, bias, h_prev, h_ld, c, h_out, hout_ld, B, H, cell);
  LAS_LAUNCH_OK("gen_cell_kernel");
  return LAS_OK;
}

}  // namespace las
