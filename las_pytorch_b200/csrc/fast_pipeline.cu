// Cross-batch serving pipeline (LAS_MODE_BF16): batch i+1's Listener runs UNDER batch i's decoder.
//
// At batch 64 the decoder (~3.3 ms) and the listener's recurrences are both latency-bound and leave the chip mostly idle, but the
// decoder is a cooperative kernel that holds its SMs for the whole decode: 96 of the 148 at c3 in its beside form (2 x 16 LSTM CTAs of
// 32 hidden units + 64 attention CTAs), 128 in its standalone form (16-unit LSTM CTAs).  Two schedules (fast_pipeline_plan):
//
// beside -- where the decoder leaves room for the recurrence clusters and >= 32 SMs for the GEMMs (c3: 52 free SMs, 32-utterance
// recurrence chunks = 4 clusters of 8):
//   caller's stream S:  cast, GEMM_0 | decoder, all steps, one launch ....................................... | wait R |
//   side stream     R:               | recurrence_0 ........ | GEMM_1 | rec_1 ...... | GEMM_2 | rec_2 .. |
// The GEMMs are capped to the SMs the decoder leaves; the later recurrences land in the SMs the first one leaves.  Nothing forces
// that placement: a later recurrence that finds no GPC with 8 free SMs waits for the decoder to end -- a longer step, same results.
//
// segmented -- otherwise: the decoder's step loop is cut into L segments (state carried on the device, bit-identical to one launch;
// fast_speller.cu) and the GEMMs run alone on the whole chip between two of them:
//   caller's stream S:  cast, GEMM_0 | seg_0 ........... | GEMM_1 | seg_1 ..... | GEMM_2 | seg_2 .. |
//   side stream     R:               | recurrence_0 .... |        | rec_1 ..... |        | rec_2 .. |
// Segment lengths are proportional to the layers' time steps (800 / 400 / 200 at T = 1600).
//
// In both, a recurrence's clusters must be placed before a decoder launch takes its SMs (a cluster needs 8 free SMs inside one GPC):
// the recurrence kernel reports residency through a counter that a one-thread kernel on S waits for before the launch.
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

// Can the listener of `ld` run next to the decoder of `sd`, and how?  Beside, where the decoder in its beside form (32-unit LSTM CTAs,
// fast_speller.cu lstm_plan) leaves room for the recurrence clusters and >= 32 SMs for the GEMMs; segmented otherwise, next to the
// decoder's standalone form.  The recurrence takes the smallest chunk whose clusters fit the free SMs (the fastest per serial step).
// The one reader of debug key 31.
PipePlan fast_pipeline_plan(const las_listener_dims* ld, const las_speller_dims* sd, int steps) {
  PipePlan pp{0, false};
  if (ld->L > 8 || steps < 4 * ld->L) return pp;
  if (sd->B > fast_speller_max_group(sd)) return pp;  // the decoder itself runs in several launch groups: no room for a pipeline
  auto chunk = [&](int free_sms) {
    for (int bc = 16; bc <= 64; bc *= 2)
      if (fast_listener_rec_ctas(ld, bc) <= free_sms) return bc;
    return 0;
  };
  const int free_beside = sm_count() - fast_speller_ctas(sd, true);
  if (debug_options().pipe_beside != 0 && free_beside >= 32 && chunk(free_beside) > 0) return {chunk(free_beside), true};
  pp.bc = chunk(sm_count() - fast_speller_ctas(sd, false));
  return pp;
}

int fast_pipeline_step(const las_decode_io* io, const SpellerF32Inputs& spl_f32, const void* spl_packed_fast, const las_speller_dims* sd,
                       int steps, int decode_mode, int relu, void* spl_ws_fast, const float* x, const int32_t* x_lengths, const void* lis_packed,
                       const las_listener_dims* ld, float* enc, int32_t* enc_lengths, void* lis_ws, bool f16, cudaStream_t st) {
  const PipePlan pp = fast_pipeline_plan(ld, sd, steps);
  const int bc = pp.bc;
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
  const int rec_ctas = fast_listener_rec_ctas(ld, bc);
  const int Bc = sd->B;
  LAS_CUDA_OK(cudaMemsetAsync(pe->resident, 0, sizeof(int) * 8, st));
  LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 0, bc, nullptr, 0, f16, st));
  LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 1, bc, nullptr, 0, f16, st));
  LAS_CUDA_OK(cudaEventRecord(pe->gemm_done[0], st));
  if (pp.beside) {
    // layer 0's recurrence placed first, then the whole decode as one launch on the SMs it leaves; the later layers' GEMMs (on the
    // SMs the decoder leaves) and recurrences (on the SMs the first one leaves) follow on the side stream while the decoder runs
    const int gemm_ctas = sm_count() - fast_speller_ctas(sd, true);
    LAS_CUDA_OK(cudaStreamWaitEvent(side, pe->gemm_done[0], 0));
    LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 2, bc, pe->resident, 0, f16, side));
    wait_resident_kernel<<<1, 1, 0, st>>>(pe->resident, rec_ctas);
    LAS_LAUNCH_OK("wait_resident_kernel");
    LAS_TRY(fast_speller_decode_segment(io, spl_f32, spl_packed_fast, sd, 0, Bc, 0, steps, true, true, decode_mode, relu, spl_ws_fast, f16, true, st));
    for (int l = 1; l < L; ++l) {
      LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 1 + 2 * l, bc, nullptr, gemm_ctas, f16, side));
      LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 2 + 2 * l, bc, nullptr, 0, f16, side));
    }
    LAS_CUDA_OK(cudaEventRecord(pe->rec_done[L - 1], side));
    LAS_CUDA_OK(cudaStreamWaitEvent(st, pe->rec_done[L - 1], 0));
    return LAS_OK;
  }
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
  int sb = 0;
  for (int l = 0; l < L; ++l) {
    // recurrence of layer l on the side stream, placed first ...
    LAS_CUDA_OK(cudaStreamWaitEvent(side, pe->gemm_done[l], 0));
    LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 2 + 2 * l, bc, pe->resident + l, 0, f16, side));
    LAS_CUDA_OK(cudaEventRecord(pe->rec_done[l], side));
    // ... then the decoder's segment on the SMs it leaves free
    wait_resident_kernel<<<1, 1, 0, st>>>(pe->resident + l, rec_ctas);
    LAS_LAUNCH_OK("wait_resident_kernel");
    LAS_TRY(fast_speller_decode_segment(io, spl_f32, spl_packed_fast, sd, 0, Bc, sb, seg[l], sb == 0, l == L - 1, decode_mode, relu, spl_ws_fast,
                                        f16, false, st));
    sb += seg[l];
    LAS_CUDA_OK(cudaStreamWaitEvent(st, pe->rec_done[l], 0));
    if (l + 1 < L) {
      LAS_TRY(fast_listener_stage(x, x_lengths, lis_packed, ld, enc, enc_lengths, lis_ws, 3 + 2 * l, bc, nullptr, 0, f16, st));
      LAS_CUDA_OK(cudaEventRecord(pe->gemm_done[l + 1], st));
    }
  }
  return LAS_OK;
}

}  // namespace las
