// Beam search on the step-per-launch decoder (include/las_b200.h las_speller_beam_search): the initial rows, the per-step selection
// and state reorder, and the final ranking and back-trace.  Each utterance owns K consecutive decoder rows; one CTA per utterance
// touches them, so the reorder needs no second launch and no scratch copy.
#include "las_kernels.cuh"

namespace las {

namespace {

constexpr int BS_MAX_K = 32;
constexpr int BS_CHUNK = 128;  // columns per pass of the in-place row permutation

// candidate order: higher score first, then lower parent, then lower token (total, so the selection is deterministic)
__device__ __forceinline__ bool beats(float va, int pa, int ta, float vb, int pb, int tb) {
  return va > vb || (va == vb && (pa < pb || (pa == pb && ta < tb)));
}

__global__ void beam_init_kernel(float* xin, int xin_ld, const float* enc, float* score, int32_t* fin, int K, int U, int E, int V) {
  const int r = blockIdx.x, b = r / K;
  for (int i = threadIdx.x; i < V + E; i += blockDim.x)
    xin[(size_t)r * xin_ld + i] = (i < V) ? (i == 0 ? 1.f : 0.f) : enc[(size_t)b * U * E + (i - V)];  // <sos> one-hot | enc[b, 0]
  if (threadIdx.x == 0) {
    score[r] = (r % K == 0) ? 0.f : -INFINITY;  // one live row: step 0 yields no duplicates
    fin[r] = 0;
  }
}

// One CTA per utterance, one warp per row for the per-row top K, then a rank-based merge of the K*K survivors.
__global__ void __launch_bounds__(1024) beam_step_kernel(const BeamStepArgs a) {
  __shared__ float c_val[BS_MAX_K * BS_MAX_K];
  __shared__ float c_lp[BS_MAX_K * BS_MAX_K];
  __shared__ int c_tok[BS_MAX_K * BS_MAX_K];
  __shared__ int s_slot[BS_MAX_K], s_par[BS_MAX_K], s_tok[BS_MAX_K];
  __shared__ int s_moved;
  __shared__ float s_tile[BS_MAX_K * BS_CHUNK];
  const int b = blockIdx.x, K = a.K, r0 = b * K;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;

  // ---- per-row top K: repeated warp arg-max over the candidates ranked below the previous pick
  for (int k = wid; k < K; k += nw) {
    const float sk = a.score[r0 + k];
    const bool finished = a.fin[r0 + k] != 0;
    const float* lp = a.logp + (size_t)(r0 + k) * a.V;
    int j = 0;
    if (sk != -INFINITY && finished) {  // a finished hypothesis only continues as itself, with <eos> at log-prob 0
      if (lane == 0) {
        c_val[k * K] = sk;
        c_tok[k * K] = a.eos;
        c_lp[k * K] = 0.f;
      }
      j = 1;
    } else if (sk != -INFINITY) {
      float last_v = INFINITY;
      int last_t = -1;
      for (; j < K; ++j) {
        float bv = -INFINITY;
        int bt = 0x7fffffff;
        for (int v = lane; v < a.V; v += 32) {
          const float x = sk + lp[v];
          const bool below = x < last_v || (x == last_v && v > last_t);
          if (below && x != -INFINITY && (x > bv || (x == bv && v < bt))) { bv = x; bt = v; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
          if (ov > bv || (ov == bv && ot < bt)) { bv = ov; bt = ot; }
        }
        if (bv == -INFINITY) break;  // fewer than K finite candidates in this row
        if (lane == 0) {
          c_val[k * K + j] = bv;
          c_tok[k * K + j] = bt;
          c_lp[k * K + j] = lp[bt];
        }
        last_v = bv;
        last_t = bt;
      }
    }
    for (int i = j + lane; i < K; i += 32) c_val[k * K + i] = -INFINITY;  // empty places
  }
  if (tid < K) s_slot[tid] = -1;
  __syncthreads();

  // ---- merge: a candidate's rank is the number of candidates that beat it; the K best fill slots 0..K-1
  for (int i = tid; i < K * K; i += blockDim.x) {
    const float vi = c_val[i];
    if (vi == -INFINITY) continue;
    const int pi = i / K, ti = c_tok[i];
    int rank = 0;
    for (int q = 0; q < K * K && rank < K; ++q) {
      const float vq = c_val[q];
      if (vq != -INFINITY && beats(vq, q / K, c_tok[q], vi, pi, ti)) ++rank;
    }
    if (rank < K) s_slot[rank] = i;
  }
  if (tid == 0) s_moved = 0;
  __syncthreads();

  if (tid < K) {
    const int i = s_slot[tid];
    // a slot without a finite candidate keeps its own (unused) state and scores -inf
    const int p = i >= 0 ? i / K : tid;
    const int t = i >= 0 ? c_tok[i] : a.eos;
    a.parent[r0 + tid] = p;
    a.token[r0 + tid] = t;
    a.token_logp[r0 + tid] = i >= 0 ? c_lp[i] : 0.f;
    a.score[r0 + tid] = i >= 0 ? c_val[i] : -INFINITY;
    a.fin[r0 + tid] = (t == a.eos) ? 1 : 0;
    s_par[tid] = p;
    s_tok[tid] = t;
    if (p != tid) atomicOr(&s_moved, 1);
  }
  __syncthreads();

  // ---- fed-back word of every new row
  for (int i = tid; i < K * a.V; i += blockDim.x) {
    const int k = i / a.V, v = i % a.V;
    a.xin[(size_t)(r0 + k) * a.xld + v] = (v == s_tok[k]) ? 1.f : 0.f;
  }
  if (!s_moved) return;

  // ---- rows take their parent's state: h and c of every layer, and the context; column chunk by column chunk through shared memory
  const int nbuf = 2 * a.sl + 1;
  for (int q = 0; q < nbuf; ++q) {
    float* base;
    long long ld;
    int width;
    if (q < a.sl) {
      base = a.h + ((size_t)q * a.B * K + r0) * a.Hs; ld = a.Hs; width = a.Hs;
    } else if (q < 2 * a.sl) {
      if (!a.c) continue;
      base = a.c + ((size_t)(q - a.sl) * a.B * K + r0) * a.Hs; ld = a.Hs; width = a.Hs;
    } else {
      base = a.xin + (size_t)r0 * a.xld + a.V; ld = a.xld; width = a.E;
    }
    for (int c0 = 0; c0 < width; c0 += BS_CHUNK) {
      const int cw = min(BS_CHUNK, width - c0);
      for (int i = tid; i < K * cw; i += blockDim.x) {
        const int k = i / cw, col = i % cw;
        s_tile[k * BS_CHUNK + col] = base[k * ld + c0 + col];
      }
      __syncthreads();
      for (int i = tid; i < K * cw; i += blockDim.x) {
        const int k = i / cw, col = i % cw;
        base[k * ld + c0 + col] = s_tile[s_par[k] * BS_CHUNK + col];
      }
      __syncthreads();
    }
  }
}

// One warp per utterance: lane k traces slot k back through the back-pointers of the S_run steps that were run; outputs have S_out
// steps, the tail padded as a full run would have left it (every row had ended, so eos at log-prob 0).  src_rows records, along the
// same path, the decoder row (b*K + parent) whose attention produced each token, -1 from the length on.
__global__ void __launch_bounds__(32) beam_finalize_kernel(const BeamFinalArgs a) {
  const int b = blockIdx.x, k = threadIdx.x, K = a.K, S = a.S_run;
  const size_t bk = (size_t)a.B * K;
  float sc = -INFINITY, key = -INFINITY;
  int len = 0;
  if (k < K) {
    sc = a.score[(size_t)b * K + k];
    if (sc != -INFINITY) {
      len = S;
      int j = k;
      for (int t = S - 1; t >= 0; --t) {
        const size_t o = t * bk + (size_t)b * K + j;
        if (a.token[o] == a.eos) len = t + 1;
        j = a.parent[o];
      }
      key = sc / powf((float)len, a.alpha);
    }
  }
  // rank by (key desc, slot asc)
  int rank = 0;
  for (int q = 0; q < K; ++q) {
    const float kq = __shfl_sync(0xffffffffu, key, q);
    if (kq > key || (kq == key && q < k)) ++rank;
  }
  if (k >= K || rank >= a.N) return;
  const size_t out = ((size_t)b * a.N + rank) * a.S_out;
  a.lengths_out[(size_t)b * a.N + rank] = len;
  a.scores_out[(size_t)b * a.N + rank] = sc;
  for (int t = S; t < a.S_out; ++t) {
    a.tokens_out[out + t] = a.eos;
    if (a.token_logp_out) a.token_logp_out[out + t] = 0.f;
    if (a.src_rows) a.src_rows[out + t] = -1;
  }
  int j = k;
  for (int t = S - 1; t >= 0; --t) {
    const size_t o = t * bk + (size_t)b * K + j;
    const bool live = t < len;  // a -inf slot has length 0: all <eos>
    a.tokens_out[out + t] = live ? a.token[o] : a.eos;
    if (a.token_logp_out) a.token_logp_out[out + t] = live ? a.token_logp[o] : 0.f;
    j = a.parent[o];
    if (a.src_rows) a.src_rows[out + t] = live ? b * K + j : -1;
  }
}

// attn[b, n, t, h, :] = work[t, h, src_rows[b, n, t], :], zeros where src_rows is -1 (t >= length).  Block (b*N + n, chunk of t).
constexpr int BT_STEPS = 8;  // steps per CTA
__global__ void __launch_bounds__(256) beam_attention_trace_kernel(const float* work, const int32_t* src_rows, float* attn, int BK, int S,
                                                                   int heads, int U) {
  const int bn = blockIdx.x, t0 = blockIdx.y * BT_STEPS, hu = heads * U;
  for (int t = t0; t < min(S, t0 + BT_STEPS); ++t) {
    const int row = src_rows[(size_t)bn * S + t];
    float* dst = attn + ((size_t)bn * S + t) * hu;
    for (int i = threadIdx.x; i < hu; i += blockDim.x) {
      const int h = i / U, u = i - h * U;
      dst[i] = row >= 0 ? work[(((size_t)t * heads + h) * BK + row) * U + u] : 0.f;
    }
  }
}

// *steps_done = step when every one of the n rows has ended (fin != 0; a -inf slot counts as ended), else left as it is.
__global__ void __launch_bounds__(256) beam_all_ended_kernel(const int32_t* fin, int n, int step, int32_t* steps_done) {
  int all = 1;
  for (int i = threadIdx.x; i < n; i += blockDim.x) all &= fin[i] != 0;
  if (__syncthreads_and(all) && threadIdx.x == 0) *steps_done = step;
}

}  // namespace

int launch_beam_init(float* xin, int xin_ld, const float* enc, float* score, int32_t* fin, int B, int K, int U, int E, int V, cudaStream_t st) {
  beam_init_kernel<<<B * K, 128, 0, st>>>(xin, xin_ld, enc, score, fin, K, U, E, V);
  LAS_LAUNCH_OK("beam_init_kernel");
  return LAS_OK;
}

int launch_beam_step(const BeamStepArgs& a, cudaStream_t st) {
  LAS_REQUIRE(a.K >= 1 && a.K <= BS_MAX_K, "beam width %d is not in [1, %d]", a.K, BS_MAX_K);
  const int threads = a.K * 32 < 128 ? 128 : a.K * 32;
  beam_step_kernel<<<a.B, threads, 0, st>>>(a);
  LAS_LAUNCH_OK("beam_step_kernel");
  return LAS_OK;
}

int launch_beam_finalize(const BeamFinalArgs& a, cudaStream_t st) {
  LAS_REQUIRE(a.K >= 1 && a.K <= BS_MAX_K && a.N >= 1 && a.N <= a.K, "beam width %d / n-best %d out of range", a.K, a.N);
  LAS_REQUIRE(a.S_run >= 1 && a.S_run <= a.S_out, "steps run %d is not in [1, %d]", a.S_run, a.S_out);
  beam_finalize_kernel<<<a.B, 32, 0, st>>>(a);
  LAS_LAUNCH_OK("beam_finalize_kernel");
  return LAS_OK;
}

int launch_beam_attention_trace(const float* work, const int32_t* src_rows, float* attn, int B, int K, int N, int S, int heads, int U,
                                cudaStream_t st) {
  beam_attention_trace_kernel<<<dim3(B * N, (S + BT_STEPS - 1) / BT_STEPS), 256, 0, st>>>(work, src_rows, attn, B * K, S, heads, U);
  LAS_LAUNCH_OK("beam_attention_trace_kernel");
  return LAS_OK;
}

int launch_beam_all_ended(const int32_t* fin, int n, int step, int32_t* steps_done, cudaStream_t st) {
  beam_all_ended_kernel<<<1, 256, 0, st>>>(fin, n, step, steps_done);
  LAS_LAUNCH_OK("beam_all_ended_kernel");
  return LAS_OK;
}

}  // namespace las
