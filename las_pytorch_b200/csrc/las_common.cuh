// Shared host/device helpers for the LAS B200 library (internal; the public surface is include/las_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "las_b200.h"

namespace las {

// ---- error plumbing: thread-local message, integer status (never abort) -------------------------------
char* err_buf();
int fail(int code, const char* fmt, ...);
void count_launch(int n = 1);

#define LAS_CUDA_OK(expr)                                                                       \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return ::las::fail(LAS_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define LAS_LAUNCH_OK(name)                                                                     \
  do {                                                                                          \
    cudaError_t _e = cudaGetLastError();                                                        \
    if (_e != cudaSuccess)                                                                      \
      return ::las::fail(LAS_ECUDA, "launch of %s failed: %s (%s:%d)", name, cudaGetErrorString(_e), __FILE__, __LINE__); \
    ::las::count_launch();                                                                      \
  } while (0)

#define LAS_REQUIRE(cond, ...)                                 \
  do {                                                         \
    if (!(cond)) return ::las::fail(LAS_EINVAL, __VA_ARGS__);  \
  } while (0)

#define LAS_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != LAS_OK) return _s; \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Carves sub-buffers out of one caller-provided allocation (256-byte aligned pieces).
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
  size_t total() const { return align_up(off, 256); }
};

int sm_count();  // cached per device

// ---- las_debug_set_option switches and the las_debug_set_trace buffer -----------------------------------
// Process-wide, written only by those two entry points (las_api.cu: its table maps each key of include/las_b200.h to a field
// here and to the values it takes), read by the launchers at their decision points through debug_options().  Defaults are the
// paths every call takes unless a test or a measurement asks for another.
struct DebugOptions {
  int ctx_tmem = 1;           // persistent decoder: context through tensor memory (0: CUDA cores only)
  int rec_overlap = 1;        // listener: input-projection GEMM concurrent with the recurrence (0: in front of it)
  int gemm_direct_store = 0;  // tcgen05 GEMM: row-per-thread global stores instead of the TMA-store epilogue
  int rec_force_bc = 0;       // listener: batch chunk per recurrence cluster (0: pick_bc)
  int att_split = 1;          // persistent decoder: long encoders split over a 2-CTA cluster (0: never)
  int gen_fused = 1;          // fused generic decoder step and the cluster attention kernel (0: unfused step, one-CTA attention)
  int gen_cluster = 0;        // CTAs per utterance of that attention cluster (0: by batch)
  int dec_groups = 1;         // persistent decoder: two utterance groups through the LSTM CTAs (0: lockstep)
  int dec_units = 0;          // persistent decoder: hidden units per LSTM CTA (16 / 32; 0: lstm_plan)
  int pipe_beside = 1;        // serving pipeline: the beside schedule where the chip has room for it (0: always segmented)
  int pipe_split[8] = {};     // serving pipeline: decoder steps of segment l (0: proportional to the layer's time steps)
  long long* trace = nullptr;  // device buffer of clock64 / globaltimer stamps, laid out as below (nullable)
  long long* trace_at(int offset) const { return trace ? trace + offset : nullptr; }
};
const DebugOptions& debug_options();

// Layout of the trace buffer, in int64 elements.  A caller provides TRACE_DEC_CTA + 8 * sm_count() of them wherever a persistent
// decoder can run (include/las_b200.h).
constexpr int TRACE_REC = 0;        // [64 steps][8]: the layer-0 recurrence, CTA 0 (fast_listener.cu)
constexpr int TRACE_GEN = 0;        // generic decoder step, CTA 0 of each kernel (gen_step.cu): the attention at TRACE_GEN, layer l's
constexpr int TRACE_GEN_SLOT = 16;  // cell step at TRACE_GEN + TRACE_GEN_SLOT * (1 + l); shares the front with the recurrence's block
constexpr int TRACE_DEC = 512;      // [5 roles][32 steps][8]: the persistent decoder's role CTAs (fast_speller.cu)
constexpr int TRACE_DEC_CTA = TRACE_DEC + 5 * 32 * 8;  // [CTA][8]: every CTA of the persistent decoder at step 8

// 16-bit GEMM operand format of the tensor-core modes: bf16 (LAS_MODE_BF16) or IEEE fp16 (LAS_MODE_F16: same kernels, same speed, 10
// mantissa bits instead of 7; the model's operands -- weights, activations in [-1,1], filterbank features -- sit far inside fp16's
// range).  las_api.cu's layout resolvers set `f16` from the mode of the call, and every launcher of 16-bit operands takes it as an
// argument.  Operand buffers are typed __nv_bfloat16 throughout (16-bit containers); `f16` says how the bits are produced / read.
#ifdef __CUDACC__
__device__ __forceinline__ __nv_bfloat16 op_from_f32(float x, int f16) {
  if (f16) {
    const __half h = __float2half_rn(x);
    return *reinterpret_cast<const __nv_bfloat16*>(&h);
  }
  return __float2bfloat16_rn(x);
}
__device__ __forceinline__ __nv_bfloat162 op2_from_f32(float a, float b, int f16) {
  if (f16) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const __nv_bfloat162*>(&h);
  }
  return __floats2bfloat162_rn(a, b);
}
__device__ __forceinline__ float op_to_f32(__nv_bfloat16 v, int f16) {
  if (f16) return __half2float(*reinterpret_cast<const __half*>(&v));
  return __bfloat162float(v);
}
__device__ __forceinline__ float2 op2_to_f32(__nv_bfloat162 v, int f16) {
  if (f16) return __half22float2(*reinterpret_cast<const __half2*>(&v));
  return __bfloat1622float2(v);
}
#endif

// ---- optional per-phase device timing (bench.py roofline): cudaEvent pairs around named launch groups ----
// Disabled by default (zero overhead beyond one thread-local load).  las_prof_enable(1) turns it on for the
// calling thread; las_prof_report() synchronises the recorded events and formats "name ms launches" lines.
struct ProfScope {
  int slot = -1;
  cudaStream_t st;
  ProfScope(const char* name, cudaStream_t stream);
  ~ProfScope();
};

// ---- counter-based uniform generator for LAS_DECODE_SAMPLE: splitmix64 of (seed, step, utterance) -> [0, 1) ----------
__host__ __device__ __forceinline__ float las_uniform(uint64_t seed, uint32_t step, uint32_t b) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * ((uint64_t)step + 1) + 0xD1B54A32D192ED03ull * ((uint64_t)b + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}
// index drawn from p_i = lp_i / sum_j lp_j (what Categorical(probs=log-probs) samples from), inverse-CDF over V entries
__host__ __device__ __forceinline__ int las_sample_logp_as_probs(const float* lp, int V, float u) {
  float tot = 0.f;
  for (int v = 0; v < V; ++v) tot += lp[v];
  const float target = u * tot;  // tot < 0: the cumulative sum decreases towards tot
  float acc = 0.f;
  for (int v = 0; v < V; ++v) {
    acc += lp[v];
    if (acc <= target) return v;
  }
  return V - 1;
}

// ---- device math ---------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoid_precise(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace las
