// Cross-batch serving pipeline (LAS_MODE_BF16): batch i+1's Listener runs UNDER batch i's decoder.
//
// At batch 64 the decoder (128 CTAs, ~3.8 ms) and the listener's recurrence (~1.7 ms) are both latency-bound and leave the chip
// mostly idle, but they cannot simply share it: the decoder is a cooperative kernel that owns 128 of the 148 SMs, and the
// input-projection GEMMs want all of them.  The pipeline therefore cuts the decoder's step loop into L segments (state carried
// on the device, bit-identical to one launch; fast_speller.cu) and interleaves the listener's stages of the NEXT batch:
//
//   caller's stream S:  cast, GEMM_0 | seg_0 ........... | GEMM_1 | seg_1 ..... | GEMM_2 | seg_2 .. |
//   side stream     R:               | recurrence_0 .... |        | rec_1 ..... |        | rec_2 .. |
//
// The GEMMs run alone on the whole chip between two segments; each recurrence runs on the <= 20 SMs the decoder leaves free (one
// 64-utterance chunk per direction: 2 clusters of 8 CTAs at H = 256).  Segment lengths are proportional to the layers' time steps
// (800 / 400 / 200 at T = 1600).  A recurrence's clusters must be placed before the decoder segment takes its 128 SMs (a cluster
// needs 8 free SMs inside one GPC): the recurrence kernel reports residency through a counter that a one-thread kernel on S waits
// for before the segment is launched.
#include "las_fast.cuh"
#include "las_kernels.cuh"

namespace las {

namespace {

// Residency is a placement matter only (nothing read here is produced by the kernel waited for), so the wait is bounded: after
// 1 ms the decoder segment is launched regardless and the recurrence simply runs when SMs free up.
__global__ void wait_resident_kernel(const int* flag, int target) {
  long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v >= target) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t - t0 > 1000000LL) break;
    __nanosleep(100);
  }
}

struct PipeEvents {
  int dev = -1;
  cudaEvent_t gemm_done[8] = {}, rec_done[8] = {};
  int* resident = nullptr;  // [8] device counters
};
thread_local PipeEvents g_pe;
int pipe_events(PipeEvents** out) {
  int dev = -1;
  LAS_CUDA_OK(cudaGetDevice(&dev));
  if (g_pe.dev != dev) {
    if (g_pe.dev >= 0) {
      for (int i = 0; i < 8; ++i) { cudaEventDestroy(g_pe.gemm_done[i]); cudaEventDestroy(g_pe.rec_done[i]); }
      cudaFree(g_pe.resident);
      g_pe = PipeEvents();
    }
    for (int i = 0; i < 8; ++i) {
      LAS_CUDA_OK(cudaEventCreateWithFlags(&g_pe.gemm_done[i], cudaEventDisableTiming));
      LAS_CUDA_OK(cudaEventCreateWithFlags(&g_pe.rec_done[i], cudaEventDisableTiming));
    }
    LAS_CUDA_OK(cudaMalloc(&g_pe.resident, sizeof(int) * 8));
    g_pe.dev = dev;
  }
  *out = &g_pe;
  return LAS_OK;
}

}  // namespace

// Can the listener of `ld` run next to the decoder of `sd`?  Returns the recurrence's batch chunk (16 / 32 / 64) or 0.
int fast_pipeline_bc(const las_listener_dims* ld, const las_speller_dims* sd, int steps) {
  if (ld->L > 8 || steps < 4 * ld->L) return 0;
  if (sd->B > fast_speller_max_group(sd)) return 0;  // the decoder itself runs in several launch groups: no room for a pipeline
  const int dec_ctas = fast_speller_ctas(sd);
  const int free_sms = sm_count() - dec_ctas;
  for (int bc = 16; bc <= 64; bc *= 2)
    if (fast_listener_rec_ctas(ld, bc) <= free_sms) return bc;
  return 0;
}

int fast_pipeline_step(const las_decode_io* io, const SpellerF32Inputs& spl_f32, const void* spl_packed_fast, const las_speller_dims* sd,
                       int steps, int decode_mode, int relu, void* spl_ws_fast, const float* x, const int32_t* x_lengths, const void* lis_packed,
                       const las_listener_dims* ld, float* enc, int32_t* enc_lengths, void* lis_ws, bool f16, cudaStream_t st) {
  const int bc = fast_pipeline_bc(ld, sd, steps);
  if (bc == 0 || io->early_exit) {
    // no room next to the decoder (or a decoder that may stop early): one after the other
    LAS_TRY(fast_speller_decode(io, spl_f32, spl_packed_fast, sd, steps, decode_mode, relu, spl_ws_fast, f16, st));
    return fast_listener_forward(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, f16, st);
  }
  PipeEvents* pe = nullptr;
  LAS_TRY(pipe_events(&pe));
  cudaStream_t side = nullptr;
  LAS_TRY(fast_side_stream(&side));
  const int L = ld->L;
  // decoder segment lengths: proportional to the layers' recurrence times -- their time steps (T/2, T/4, ...), layer 0 a little cheaper
  // per step (fused input projection: 2.25 vs 2.55 us in the 64-utterance form) --, even, the remainder in the last one
  int seg[8], used = 0;
  {
    auto weight = [&](int l) { return (double)(ld->T >> (l + 1)) * (l == 0 ? 0.88 : 1.0); };
    const int* split = debug_options().pipe_split;
    double tot = 0;
    for (int l = 0; l < L; ++l) tot += weight(l);
    for (int l = 0; l < L; ++l) {
      int n = split[l] > 0 ? split[l] : (int)(steps * weight(l) / tot);
      n &= ~1;
      if (n < 2) n = 2;
      if (l == L - 1 || used + n > steps - 2 * (L - 1 - l)) n = (l == L - 1) ? steps - used : ((steps - used - 2 * (L - 1 - l)) & ~1);
      seg[l] = n;
      used += n;
    }
  }
  const int rec_ctas = fast_listener_rec_ctas(ld, bc);
  const int Bc = sd->B;
  LAS_CUDA_OK(cudaMemsetAsync(pe->resident, 0, sizeof(int) * 8, st));
  LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 0, bc, nullptr, f16, st));
  LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 1, bc, nullptr, f16, st));
  LAS_CUDA_OK(cudaEventRecord(pe->gemm_done[0], st));
  int sb = 0;
  for (int l = 0; l < L; ++l) {
    // recurrence of layer l on the side stream, placed first ...
    LAS_CUDA_OK(cudaStreamWaitEvent(side, pe->gemm_done[l], 0));
    LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 2 + 2 * l, bc, pe->resident + l, f16, side));
    LAS_CUDA_OK(cudaEventRecord(pe->rec_done[l], side));
    // ... then the decoder's segment on the SMs it leaves free
    wait_resident_kernel<<<1, 1, 0, st>>>(pe->resident + l, rec_ctas);
    LAS_LAUNCH_OK("wait_resident_kernel");
    LAS_TRY(fast_speller_decode_segment(io, spl_f32, spl_packed_fast, sd, 0, Bc, sb, seg[l], sb == 0, l == L - 1, decode_mode, relu, spl_ws_fast,
                                        f16, st));
    sb += seg[l];
    LAS_CUDA_OK(cudaStreamWaitEvent(st, pe->rec_done[l], 0));
    if (l + 1 < L) {
      LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 3 + 2 * l, bc, nullptr, f16, st));
      LAS_CUDA_OK(cudaEventRecord(pe->gemm_done[l + 1], st));
    }
  }
  return LAS_OK;
}

}  // namespace las
