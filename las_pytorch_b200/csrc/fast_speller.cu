// LAS_MODE_BF16 speller: the whole attention-decoder step loop (model/las_model.py:209-236) as ONE persistent
// cooperative kernel.  No launch, host sync or PCIe traffic between decode steps.
//
// CTA roles (one CTA per SM, all co-resident; cudaLaunchAttributeCooperative guarantees it):
//   * LSTM CTAs: layer l, block nb owns 16 hidden units (64 gate columns, unit-major / gate-minor).  Its slice of
//     [W_hh | W_word | W_in] (bf16, 128-byte-swizzled K-major atoms) stays on chip for all S steps as the A operand
//     (the critical input's part in tensor memory, the rest in shared memory); the B operand is the activation matrix
//     [batch (N), K] streamed per step by TMA:
//       part 0   the layer's own h_{s-1}            (ready long before it is needed; accumulator 0)
//       part 1a  the critical input: the context of step s-1 (layer 0) / the lower layer's fresh h (accumulator 1)
//       part 1b  layer 0 only, and only when the fed-back word is a dense vector (decode_mode 0, dense teacher
//                forcing, the first step): the word atom.  For greedy decoding / index teacher forcing the word is
//                an index, and the epilogue adds the matching column of W_word straight from the resident atom.
//     tcgen05.mma accumulates in TMEM; the epilogue thread of a gate row holds the cell state c of four (unit, batch)
//     cells in registers (fp32) and writes h (bf16 operand copy for the TMA consumers; fp32 flag-in-data copy for the
//     attention CTAs).
//   * attention CTAs: one per utterance.  W_phi, W_cd (bf16) and psi(enc)[b] (fp32) are resident in shared memory,
//     enc[b]^T in tensor memory; per step: q = relu(W_phi h + b), energies, length-masked softmax, context (UMMA with
//     the scores as the B operand), publish the context, then character distribution, log-softmax, argmax / teacher
//     forcing, publish the word.  The context is published BEFORE the character distribution is evaluated, so layer 0's
//     context GEMM of the next step overlaps the logits of this one.
// Hand-offs (measured in tools/microbench.cu: a release/acquire counter hop costs ~1.0 us + ~0.8 us of TMA, a
// self-validating store ~0.5 us):
//   * matrix hand-offs consumed by TMA (h -> LSTM CTAs, context / dense word -> layer 0): global buffers double-buffered
//     by step parity + monotonically increasing release/acquire counters; fence.proxy.async orders the TMA reads;
//   * top-layer h -> attention CTA and greedy token -> layer 0: 8-byte {value, step tag} slots written with one store
//     and polled by the consumer itself (no fence, no counter): the data is its own flag.
#include <cuda.h>
#include <string.h>

#include "las_fast.cuh"
#include "las_kernels.cuh"
#include "umma.cuh"

namespace las {

int make_tmap_bf16_box(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows);  // fast_gemm.cu
int make_tmap_bf16_atoms(CUtensorMap* tm, const void* base, long long rows, int atoms, long long ld, int box_rows, int box_atoms);

namespace {

constexpr int DEC_NW = 64;        // gate columns per block of the packed image (16 hidden units x 4 gates)
constexpr int DEC_UNITS = DEC_NW / 4;
constexpr int DEC_MAX_STAGES = 16;
constexpr int DEC_THREADS = 512;
constexpr int DEC_VP = 64;        // one-hot / word columns padded to one 64-wide K atom
constexpr int WATOM_BYTES = DEC_NW * 128;  // B atom: 64 gate columns x 64 bf16
constexpr int MAX_SL = 4;
constexpr int CTR_CTX = MAX_SL, CTR_WORD = MAX_SL + 1, N_CTR = MAX_SL + 2;
constexpr int ATT_MAXP = 3;       // encoder steps per attention CTA <= ATT_MAXP * 256
typedef unsigned long long u64;

struct DecParams {
  CUtensorMap tm_h[MAX_SL][2];  // hbuf[l][parity]  bf16 [B, Hs]   one 64-column atom per copy (set where Hs % 64 != 0)
  CUtensorMap tm_x[2];          // xbuf[parity]     bf16 [B, E]   the context fed to layer 0 (same pitch as an h buffer)
  CUtensorMap tm_w[2];          // wbuf[parity]     bf16 [B, VP]  the dense word fed to layer 0 (one atom)
  CUtensorMap tm_h3[MAX_SL][2]; // the same buffers as {64 k, B, atoms}: one copy brings a whole activation part (set where Hs % 64 == 0)
  CUtensorMap tm_x3[2];
  const uint8_t* w_img[MAX_SL]; // [Hs/16][atoms_l] swizzled 64x64 bf16 atoms: h part, (layer 0: word atom), input part
  const float* bias[MAX_SL];    // [4*Hs] b_ih + b_hh in unit-major / gate-minor order
  __nv_bfloat16* hbuf[MAX_SL][2];
  __nv_bfloat16* xbuf[2];
  __nv_bfloat16* wbuf[2];
  u64* h_ll;                    // [B, Hs] {fp32 h of the top layer, step tag}
  u64* tok_ll;                  // [ncl, B] {token fed back, step tag}: one private copy per layer-0 CTA (no polling hot spot)
  const float* c_init;          // nullable [sl, c_init_rows, Hs], row of utterance b: c_init_b0 + b
  float* h_out;                 // nullable [sl, Bfull, Hs]
  float* c_out;                 // nullable [sl, c_out_rows, Hs], row c_out_b0 + b
  int c_init_rows, c_init_b0, c_out_rows, c_out_b0;  // the caller's [sl,Bfull,Hs] tensors or the workspace's per-launch carry buffer
  // Segmented decode (cross-batch pipeline, <eos> early exit): this launch covers the global steps [s0, s0 + steps).  Counters, tags
  // and buffer parities are launch-local (s0 is even, so parities line up); outputs, labels and the sampling counter use s0 + s.
  int s0;
  const int32_t* tok_init;      // nullable [B]: the token fed back by global step s0 - 1 (index-word modes, s0 > 0)
  int32_t* tok_carry;           // nullable [B]: receives the token fed back by this launch's last step
  const int32_t* stop;          // nullable: *stop != 0 -> every CTA returns at once (all utterances have emitted <eos>)
  const __nv_bfloat16* enc;     // [B, U, E] bf16
  const float* psi;             // [B, U, D] fp32
  const __nv_bfloat16* w_phi;   // [D, Hs] bf16
  const float* b_phi;
  const __nv_bfloat16* w_cd;    // [V, Hs + E] bf16
  const float* b_cd;
  const float* gt_dense;        // nullable [B, gt_steps, V]
  const int32_t* gt_index;      // nullable [B, gt_steps]
  const int32_t* enc_lengths;   // nullable [B]
  float* logp;                  // [S, B, V]
  float* attn;                  // nullable [S, B, U]
  int32_t* tokens;              // nullable [S, B]
  const int32_t* nll_labels;    // nullable [B, nll_steps]
  float* nll_terms;             // nullable [S, B]
  int nll_steps;
  float* word_out;              // nullable [B, V]
  float* ctx_out;               // nullable [B, E]
  uint32_t* sync;               // counters, 32 uint32 apart: [l] = h_ready[l], [CTR_CTX], [CTR_WORD]
  int B;      // utterances handled by this launch (one attention CTA each)
  int Bfull;  // batch pitch of the caller's tensors; this launch covers utterances [b0, b0 + B)
  int b0;
  int U, E, Hs, sl, V, D, steps, decode_mode, relu, gt_steps, ncl, k_in_smem;
  int wreg;  // 1: every attention thread keeps its chunks of W_phi in registers (D <= 64, Hs <= 512); no shared-memory copy
  unsigned long long sample_seed;  // LAS_DECODE_SAMPLE
  int word_gather;  // 1: the fed-back word is an index (greedy argmax / gt_index); 0: a dense vector (part 1b)
  int f16;          // GEMM operand format: 0 = bf16 (LAS_MODE_BF16), 1 = IEEE fp16 (LAS_MODE_F16)
  int att_split;    // 2: every utterance is attended by a CLUSTER of two CTAs, each holding half of the encoder steps (long encoders:
                    // all of enc[b]^T stays in tensor memory; partial softmax / context combined through DSMEM); 1: one CTA
  int ctx_tmem;     // > 0: enc[b]^T is resident in the attention CTA's tensor memory and the context is a UMMA
  int ctx_ntm;      // 128-feature tiles of enc[b]^T held in tensor memory: E/128 = all of them; fewer (long encoders, e.g. U = 375:
                    // 2 of 4) = hybrid, the remaining features are reduced on the CUDA cores from the L2-resident bf16 copy
  int groups, gsz;  // utterance groups pipelined through the LSTM CTAs (1, or 2 groups of gsz = 32 rows) -- see lstm_role_ts
  int units;        // hidden units per LSTM CTA (16 or 32; lstm_plan); ncl = ceil(Hs / units)
  int nstages, stage_bytes;  // activation slots: [64 batch rows x 64 bf16], 128-byte swizzled; last slot = word atom
  long long* trace;  // nullable test hook (TRACE_DEC): [5 roles][32 steps][8] globaltimer stamps (layer-0 CTA 0, top-layer CTA 0, attention CTA 0, ...)
};

__device__ __forceinline__ long long gtimer() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// per-CTA stamps of step 8 (spread across CTAs): behind the role trace, [gridDim][8] (las_common.cuh TRACE_DEC_CTA)
#define DEC_TRACE_ALL(slot) do { if (p.trace && s == 8) p.trace[TRACE_DEC_CTA - TRACE_DEC + blockIdx.x * 8 + (slot)] = gtimer(); } while (0)
#define DEC_TRACE(role, slot) do { if (p.trace && s < 32) p.trace[((role) * 32 + s) * 8 + (slot)] = gtimer(); } while (0)

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(tanh_fast(0.5f * x), 0.5f, 0.5f); }

__device__ __forceinline__ uint32_t ld_acquire(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// spin with relaxed loads, then one acquire load to synchronise (tools/microbench.cu: the cheapest correct pairing
// with red.release on this part)
__device__ __forceinline__ void wait_counter(const uint32_t* ctr, uint32_t target) {
  ptx::SpinGuard g;
  while (ld_relaxed(ctr) < target) g.tick();
  (void)ld_acquire(ctr);
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ uint32_t* counter(const DecParams& p, int idx, int grp = 0) { return p.sync + (grp * N_CTR + idx) * 32; }

// flag-in-data slots: one aligned 8-byte store carries the value and the step tag, so the consumer needs no fence
__device__ __forceinline__ u64 ll_pack(uint32_t value, uint32_t tag) { return ((u64)tag << 32) | value; }
__device__ __forceinline__ u64 ll_load(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void ll_store(u64* p, u64 v) { asm volatile("st.relaxed.gpu.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ uint32_t ll_wait(const u64* p, uint32_t tag) {
#if LAS_GUARD_LL
  ptx::SpinGuard g;
#endif
  u64 v = ll_load(p);
  while ((uint32_t)(v >> 32) != tag) {
#if LAS_GUARD_LL
    g.tick();
#endif
    v = ll_load(p);
  }
  return (uint32_t)v;
}

// Activation vectors read by the GEMV phases (h, context) are stored permuted: the 8 floats that go with the 16-byte
// weight chunk cc sit as two float4 at float4 index (cc / 8) * 16 + (cc % 8) and 8 float4 further on, so that the lanes
// of a quarter warp (consecutive chunks) read consecutive float4 -- one conflict-free wavefront per load.
__device__ __forceinline__ int xpos(int k) {
  const int cc = k >> 3, w = k & 7;
  return ((((cc >> 3) << 4) + ((w >> 2) << 3) + (cc & 7)) << 2) + (w & 3);
}
__device__ __forceinline__ const float4* xchunk(const float* xb, int cc) { return reinterpret_cast<const float4*>(xb) + ((cc >> 3) << 4) + (cc & 7); }
__device__ __forceinline__ uint4 lds128(const void* ptr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(ptx::smem_u32(ptr)));
  return v;
}
// dot product of 8 bf16 weights (one 16-byte chunk) with 8 fp32 activations
__device__ __forceinline__ float dot8(const uint4& w, const float4& x0, const float4& x1, float acc, int f16) {
  const __nv_bfloat162* w2 = reinterpret_cast<const __nv_bfloat162*>(&w);
  const float2 a = op2_to_f32(w2[0], f16), b = op2_to_f32(w2[1], f16), c = op2_to_f32(w2[2], f16), d = op2_to_f32(w2[3], f16);
  acc = fmaf(a.x, x0.x, acc); acc = fmaf(a.y, x0.y, acc); acc = fmaf(b.x, x0.z, acc); acc = fmaf(b.y, x0.w, acc);
  acc = fmaf(c.x, x1.x, acc); acc = fmaf(c.y, x1.y, acc); acc = fmaf(d.x, x1.z, acc); acc = fmaf(d.y, x1.w, acc);
  return acc;
}

// ------------------------------------------------------------------------------------------------------------
// LSTM role, weights-stationary operand roles ("TS form")
// ------------------------------------------------------------------------------------------------------------
// The weights are the A operand and the activations (one part at a time, see the file header) the B operand:
//     D[gate row (64 of the 128 TMEM lanes), batch (N = 64)] = W_slice[64(128), K] . act[batch, K]^T
// so that the layer's critical input weights (context / lower-layer h part, K = 512 -> 256 tensor-memory columns) are the A operand
// IN TENSOR MEMORY: a tcgen05.mma with A in TMEM issues at its ~32-cycle math floor (N = 64), against ~57 cycles when both
// operands come from shared memory (tools/microbench.cu: the shared-memory A read is exposed).  The part's 32 instructions take
// ~0.55 us of each layer's critical path instead of ~1.05 us.  The own-h part (ready long before it is needed) takes both operands
// from shared memory, in the same roles, so both parts land in accumulators of the same orientation.
// M = 128 always.  A CTA owns 16 units (64 gate rows; lanes 64..127 hold zeros, the instruction costs the same for M = 64 and 128)
// or 32 units (128 gate rows, every lane used: half as many CTAs for the same MMAs per step).  A 32-unit CTA n is built from the
// 16-unit packed image: rows 0..63 of each [128 rows x 64 k] atom are that atom of image block 2n, rows 64..127 that of block 2n+1
// (zeros past Hs) -- in the 128-byte-swizzled layout simply the two 8 KB halves of a 16 KB atom.
// Epilogue: thread = gate row (lane; unit-major / gate-minor, so the four gates of a unit sit in four adjacent lanes), 16 batch
// columns per warp; a 4x4 transpose inside each 4-lane group (two shuffle stages, as in the listener's recurrence) leaves every
// lane with (i, f, g, o) of one (unit, batch) cell -- 4 cells per thread and iteration, cell state in registers.  Eight epilogue
// warps cover the TMEM lane quadrants the CTA's rows occupy (2 or 4) x the 16-column slices (4 or 2).
template <int F16>
__device__ void lstm_role_ts(const DecParams& p, uint8_t* smem, int l, int nb) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool first = (l == 0), top = (l == p.sl - 1);
  const int nh = (p.Hs + 63) / 64;
  const int nc = first ? (p.E + 63) / 64 : (p.Hs + 63) / 64;
  const int nwd = first ? 1 : 0;
  const int natoms = nh + nwd + nc;                      // atoms of one image block
  const int UNITS = p.units, ROWS = 4 * UNITS, HALVES = UNITS / DEC_UNITS, nblk = p.Hs / DEC_UNITS;
  const int ST_PITCH = UNITS + 4;                        // staging row pitch (floats): 16-byte aligned, conflict-free reads
  const int NBUF = p.nstages, STAGE_BYTES = p.stage_bytes;
  const int wslot = NBUF - 1;
  // shared-memory weight atom: [ROWS gate rows x 64 k], SW128.  The M = 128 MMAs of a 16-unit CTA read 128 rows: lanes 64..127 take
  // the 8 KB behind each atom (the next atom, or a zero pad behind the last one) and are never read back.
  const int SATOM = ROWS * 128, WPAD = HALVES == 1 ? WATOM_BYTES : 0;
  uint8_t* abuf = smem;                                  // NBUF x STAGE_BYTES activation slots ([gsz batch rows x 64 k], SW128)
  uint8_t* wsm = abuf + (size_t)NBUF * STAGE_BYTES;      // (nh + nwd) weight atoms: own-h part, (layer 0) word atom; + WPAD
  float* bias_s = reinterpret_cast<float*>(wsm + (size_t)(nh + nwd) * SATOM + WPAD);
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + ROWS);
  uint64_t* full = bars;
  uint64_t* part_empty = bars + DEC_MAX_STAGES;
  uint64_t* tmem_full = part_empty + 1;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  float* s_st = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 2) + 15) & ~uintptr_t(15));  // [64 batch rows][ST_PITCH]
  constexpr int EPI_WARPS = 8, EPI_THREADS = EPI_WARPS * 32, PROD_WARP = 2, MMA_WARP = 3;
  // tensor-memory map: critical weights [0, nc*32), accumulator of the own-h part, accumulator of the critical part (64 columns each)
  const uint32_t a_cols = (uint32_t)nc * 32u, acc0 = a_cols, acc1 = a_cols + 64u;
  // image block of the CTA's row half hf (rows [64 hf, 64 hf + 64)), or -1: no such half / past Hs (zeros)
  auto src_block = [&](int hf) { const int b = nb * HALVES + hf; return (hf < HALVES && b < nblk) ? b : -1; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < NBUF; ++i) ptx::mbar_init(&full[i], 1);
    ptx::mbar_init(part_empty, 1);
    ptx::mbar_init(tmem_full, 1);
    ptx::mbar_init(tmem_empty, EPI_THREADS);
    ptx::fence_mbar_init();
  }
  if (warp == MMA_WARP) ptx::tmem_alloc(tmem_slot, 512);
  {  // own-h (+ word) atoms + bias -> shared memory, each atom from HALVES 8 KB image atoms (a 32-unit CTA: two), then the pad
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (int i = threadIdx.x; i < ((nh + nwd) * SATOM + WPAD) / 16; i += DEC_THREADS) {
      const int a = i / (SATOM / 16), hf = (i / (WATOM_BYTES / 16)) % HALVES, o = i % (WATOM_BYTES / 16);
      const int b = a < nh + nwd ? src_block(hf) : -1;
      reinterpret_cast<uint4*>(wsm)[i] = b >= 0 ? reinterpret_cast<const uint4*>(p.w_img[l] + ((size_t)b * natoms + a) * WATOM_BYTES)[o] : z;
    }
    if (threadIdx.x < ROWS) bias_s[threadIdx.x] = nb * ROWS + threadIdx.x < 4 * p.Hs ? p.bias[l][nb * ROWS + threadIdx.x] : 0.f;
  }
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (warp < 4) {
    // critical-part weights: global image atoms (128-byte swizzle undone) -> registers -> tensor memory, lane = gate row, two bf16 per
    // column.  Not staged in shared memory: a 32-unit CTA's 8 atoms of 16 KB would not fit next to the own-h part.
    const int row = warp * 32 + lane, r64 = row & 63, b = src_block(row >> 6);
    for (int i = 0; i < nc; ++i) {
      const uint8_t* rb = p.w_img[l] + ((size_t)(b < 0 ? 0 : b) * natoms + nh + nwd + i) * WATOM_BYTES + (r64 >> 3) * 1024 + (r64 & 7) * 128;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0;
        if (b >= 0) {
          q0 = *reinterpret_cast<const uint4*>(rb + (((2 * kk) ^ (row & 7)) << 4));
          q1 = *reinterpret_cast<const uint4*>(rb + (((2 * kk + 1) ^ (row & 7)) << 4));
        }
        const uint32_t v[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        ptx::tmem_st_32x32b_x8(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)i * 32u + (uint32_t)kk * 8u, v);
      }
    }
    ptx::tmem_st_wait();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const int S = p.steps;
  // Utterance groups (p.groups = 2 x p.gsz = 32 rows at batch 64): the decoder step is a ring of three stages (layer 0 -> layer 1 ->
  // attention -> layer 0) and with the whole batch in lockstep every stage idles two thirds of the time.  The LSTM CTAs therefore serve
  // the groups alternately -- iteration it = s * groups + grp -- with per-group counters, 32-row activation boxes and N = 32 MMAs, while
  // the attention CTAs (one per utterance anyway) simply follow their group's counters.  Every buffer is indexed by utterance row, a
  // cell's state stays with one thread, and an output column's sum does not depend on N: bit-identical to groups = 1.
  const int G = p.groups, GSZ = p.gsz;
  const int trole = (nb == 0 && l == 0) ? 0 : ((nb == 0 && top) ? 1 : -1);

  if (warp == PROD_WARP) {
    // ============================ TMA producer ============================
    // A part lands as consecutive [GSZ batch rows x 64 k] atoms in slots 0, 1, ... and completes on full[0].  Where Hs (= E) is a
    // multiple of 64 it is ONE 3-D copy over the {64 k, batch, atoms} view of the hand-off buffer: issuing eight 2-D copies took
    // ~0.55 us (~68 ns each), all of it on the critical path.  That view cannot describe a row of any other length; there every
    // atom is a 2-D copy, and TMA fills the columns past Hs with zeros (the weights' columns there are zeros too).
    const bool whole_atoms = p.Hs % 64 == 0;
    auto load_part = [&](const CUtensorMap* tm3, const CUtensorMap* tm2, int na, int row0) {
      if (whole_atoms) ptx::tma_load_3d(abuf, tm3, &full[0], 0, row0, 0);
      else
        for (int i = 0; i < na; ++i) ptx::tma_load_2d(abuf + (size_t)i * STAGE_BYTES, tm2, &full[0], i * 64, row0);
    };
    int n = 0;
    for (int it = 0; it < S * G; ++it) {
      const int s = it / G, grp = it - s * G, row0 = grp * GSZ;
      const int Bg = min(p.B - row0, GSZ);  // utterances of this group
      const uint32_t* own_ctr = counter(p, l, grp);
      const uint32_t* in_ctr = first ? counter(p, CTR_CTX, grp) : counter(p, l - 1, grp);
      const uint32_t* word_ctr = counter(p, CTR_WORD, grp);
      const int par = s & 1;
      if (n > 0) ptx::mbar_wait(part_empty, (uint32_t)((n - 1) & 1));
      ++n;
      if (lane == 0) wait_counter(own_ctr, (uint32_t)s * p.ncl);
      __syncwarp();
      fence_proxy_async_global();
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(&full[0], nh * STAGE_BYTES);
        load_part(&p.tm_h3[l][par], &p.tm_h[l][par], nh, row0);
      }
      __syncwarp();
      ptx::mbar_wait(part_empty, (uint32_t)((n - 1) & 1));
      ++n;
      if (ptx::elect_one()) ptx::mbar_arrive_expect_tx(&full[0], nc * STAGE_BYTES);
      __syncwarp();
      if (lane == 0) {
        wait_counter(in_ctr, first ? (uint32_t)s * Bg : (uint32_t)(s + 1) * p.ncl);
        if (trole >= 0 && grp == 0) DEC_TRACE(trole, 0);
        if (grp == 0) DEC_TRACE_ALL(0);
      }
      __syncwarp();
      fence_proxy_async_global();
      if (lane == 0 && trole >= 0 && grp == 0) DEC_TRACE(4, 6 + trole);
      {
        const CUtensorMap* tm3 = first ? &p.tm_x3[par] : &p.tm_h3[l - 1][par ^ 1];
        const CUtensorMap* tm2 = first ? &p.tm_x[par] : &p.tm_h[l - 1][par ^ 1];
        if (ptx::elect_one()) {
          if (trole == 0 && grp == 0) DEC_TRACE(4, 0);
          load_part(tm3, tm2, nc, row0);
          if (trole == 0 && grp == 0) DEC_TRACE(4, 2);
        }
        __syncwarp();
      }
      if (lane == 0 && trole >= 0 && grp == 0) DEC_TRACE(trole, 1);
      if (first && (p.s0 + s == 0 || !p.word_gather)) {
        if (lane == 0) wait_counter(word_ctr, (uint32_t)s * Bg);
        __syncwarp();
        fence_proxy_async_global();
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&full[wslot], STAGE_BYTES);
          ptx::tma_load_2d(abuf + (size_t)wslot * STAGE_BYTES, &p.tm_w[par], &full[wslot], 0, row0);
        }
        __syncwarp();
      }
    }
  } else if (warp == MMA_WARP) {
    // ============================ MMA issuer ============================
    const UmmaLayout lact{1, 0, 1024, (uint32_t)STAGE_BYTES}, lw{1, 0, 1024, (uint32_t)SATOM};
    const uint32_t idesc = umma_idesc_bf16(128, (uint32_t)GSZ, F16);  // M = 128 gate-row lanes (ROWS used), N = the group's batch columns
    const uint32_t a0 = ptx::smem_u32(abuf), w_addr = ptx::smem_u32(wsm);
    uint32_t phase0 = 0, phasew = 0;
    for (int it = 0; it < S * G; ++it) {
      const int s = it / G, grp = it - s * G;
      const bool wd = first && (p.s0 + s == 0 || !p.word_gather);
      ptx::mbar_wait(tmem_empty, (uint32_t)((it & 1) ^ 1));
      ptx::tc_fence_after();
      // ---- part 0: own h_{s-1}; both operands from shared memory (weights = A, activations = B)
      ptx::mbar_wait(&full[0], phase0);
      phase0 ^= 1u;
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        for (int i = 0; i < nh; ++i) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::umma_bf16(tmem + acc0, umma_smem_desc(lw, w_addr + i * SATOM, k * 16), umma_smem_desc(lact, a0 + i * STAGE_BYTES, k * 16),
                           idesc, !(i == 0 && k == 0));
        }
        ptx::umma_commit(part_empty);
      }
      __syncwarp();
      if (lane == 0 && trole >= 0 && grp == 0) DEC_TRACE(trole, 6);
      // ---- part 1: the critical input; weights from tensor memory, activations from shared memory.  Lean loop: the A operand
      // advances 8 columns per instruction, the B descriptor 32 bytes inside an atom and one slot between atoms.
      ptx::mbar_wait(&full[0], phase0);
      phase0 ^= 1u;
      ptx::tc_fence_after();
      if (lane == 0 && trole >= 0 && grp == 0) DEC_TRACE(4, 3 + 2 * trole);
      if (ptx::elect_one()) {
        uint32_t a = tmem;
        uint64_t bd_atom = umma_smem_desc(lact, a0, 0);
        const uint64_t atom_step = (uint64_t)(STAGE_BYTES >> 4);
        for (int i = 0; i < nc; ++i) {
          uint64_t bd = bd_atom;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            ptx::umma_bf16_ts(tmem + acc1, a, bd, idesc, !(i == 0 && k == 0));
            a += 8;
            bd += 2;
          }
          bd_atom += atom_step;
        }
        if (!wd) {
          ptx::umma_commit(part_empty);
          ptx::umma_commit(tmem_full);
        }
      }
      __syncwarp();
      if (wd) {  // dense word vector (first step, decode_mode 0, dense teacher forcing): its atom, shared-memory form
        ptx::mbar_wait(&full[wslot], phasew);
        phasew ^= 1u;
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::umma_bf16(tmem + acc1, umma_smem_desc(lw, w_addr + nh * SATOM, k * 16), umma_smem_desc(lact, a0 + wslot * STAGE_BYTES, k * 16),
                           idesc, 1u);
          ptx::umma_commit(part_empty);
          ptx::umma_commit(tmem_full);
        }
        __syncwarp();
      }
      if (lane == 0 && trole >= 0 && grp == 0) DEC_TRACE(trole, 2);
    }
  } else if (UNITS == DEC_UNITS ? (warp & 3) < 2 : (warp >= 4 && warp < 4 + EPI_WARPS)) {
    // ============================ epilogue: gates, cell state, h ============================
    // 16 units: warps with quadrant 0 / 1 (rows 0..63) x 4 slices = 64 columns (the whole batch, or both groups side by side);
    // 32 units: warps 4..11, two per quadrant (the producer and MMA warps sit in quadrants 2 and 3) x 2 slices = the 32 columns of
    // the group being served, so every thread keeps the cells of both groups
    const int NQ = ROWS / 32, NS = EPI_WARPS / NQ;  // TMEM lane quadrants, 16-column slices
    const int q = warp & 3, cs = UNITS == DEC_UNITS ? warp >> 2 : (warp >> 2) - 1;  // gate rows 32q..32q+31, slice cs
    const int row = q * 32 + lane;                 // gate row of this CTA = 4 * unit + gate
    const int jj = row >> 2, g = row & 3;
    const bool bit0 = (g & 1) != 0, bit1 = (g & 2) != 0;
    const int u = nb * UNITS + jj;                 // hidden unit
    const bool unit_ok = u < p.Hs;                 // (the upper half of the last 32-unit CTA where Hs % 32 == 16)
    const bool lead = (warp == (UNITS == DEC_UNITS ? 0 : 4) && lane == 0);
    const int spg = GSZ / 16, per = NS / spg;      // slices per group; groups the slices serve side by side (1 or 2)
    const int sg = cs / spg, cw = cs % spg;        // the slice serves groups grp with grp % per == sg, columns [16cw, 16cw+16) of them
    const uint32_t acc_col = (uint32_t)(cw * 16);
    const int CPR = UNITS / 8, RPW = 16 / CPR;     // hand-off: 16-byte chunks per row, rows per warp
    float c[2][4];                                 // cell state, slot k = grp / per
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int grp = k * per + sg;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int b = grp * GSZ + cw * 16 + 4 * m + g;
        c[k][m] = (grp < G && b < p.B && unit_ok && p.c_init) ? p.c_init[((size_t)l * p.c_init_rows + p.c_init_b0 + b) * p.Hs + u] : 0.f;
      }
    }
    const float4 bias4 = *reinterpret_cast<const float4*>(bias_s + 4 * jj);
    const uint8_t* watom = wsm + (size_t)nh * SATOM;  // layer 0: word atom [ROWS gate rows x 64 vocabulary entries]
    for (int it = 0; it < S * G; ++it) {
      const int s = it / G, grp = it - s * G, k = grp / per;
      const int bw = grp * GSZ + cw * 16;          // first batch row of this warp's slice
      const bool warp_live = grp % per == sg && bw < p.B;
      int bm[4];
#pragma unroll
      for (int m = 0; m < 4; ++m) bm[m] = bw + 4 * m + g;  // this thread's cell m: (unit u, batch bm[m])
      uint32_t* my_ready = counter(p, l, grp);
      // bias + (index word) the token's column of W_word for this unit's four gate rows, per cell -- before the accumulators are ready.
      // The warp's 16 batches are polled by 16 lanes (ONE L2 round trip; four dependent polls per thread cost ~2.4 us and made the
      // token the critical path) and handed to the cells' owners by shuffles.
      float4 pb[4];
      int tokl = -1;
      const bool gather = first && p.s0 + s > 0 && p.word_gather && warp_live;
      if (gather) {
        const int bb = bw + (lane & 15);
        if (bb < p.B)
          tokl = p.gt_index ? p.gt_index[(size_t)(p.b0 + bb) * p.gt_steps + (p.s0 + s - 1)]
                            : (s > 0 ? (int)ll_wait(p.tok_ll + (size_t)nb * p.B + bb, (uint32_t)s) : p.tok_init[bb]);
      }
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        pb[m] = bias4;
        const int tok = __shfl_sync(0xffffffffu, tokl, 4 * m + g);
        if (gather && tok >= 0 && tok < p.V) {
          const uint32_t tok_off = (uint32_t)(tok & 7) * 2u, tok_chunk = (uint32_t)(tok >> 3);
          float wv[4];
#pragma unroll
          for (int gg = 0; gg < 4; ++gg) {
            const uint32_t rr = (uint32_t)(4 * jj + gg);
            const uint32_t off = (rr >> 3) * 1024u + (rr & 7u) * 128u + (((tok_chunk ^ (rr & 7u)) & 7u) << 4) + tok_off;
            wv[gg] = op_to_f32(*reinterpret_cast<const __nv_bfloat16*>(watom + off), F16);
          }
          pb[m].x += wv[0]; pb[m].y += wv[1]; pb[m].z += wv[2]; pb[m].w += wv[3];
        }
      }
      if (lead && trole == 0 && grp == 0) DEC_TRACE(4, 1);
      ptx::mbar_wait(tmem_full, (uint32_t)(it & 1));
      if (lead && trole >= 0 && grp == 0) DEC_TRACE(trole, 3);
      if (lead && grp == 0) DEC_TRACE_ALL(1);
      ptx::tc_fence_after();
      float h[4] = {0.f, 0.f, 0.f, 0.f}, cc[4];
      if (warp_live) {
        uint32_t x0[16], x1[16];
        ptx::tmem_ld_32x32b_x16(tmem + ((uint32_t)(q * 32) << 16) + acc0 + acc_col, x0);
        ptx::tmem_ld_32x32b_x16(tmem + ((uint32_t)(q * 32) << 16) + acc1 + acc_col, x1);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          // lane g holds its gate's pre-activations for batches 4m..4m+3 of the slice; after the 4x4 transpose inside the 4-lane
          // group it holds all four gates (i,f,g,o) of batch 4m+g
          float v0 = __uint_as_float(x0[4 * m]) + __uint_as_float(x1[4 * m]), v1 = __uint_as_float(x0[4 * m + 1]) + __uint_as_float(x1[4 * m + 1]),
                v2 = __uint_as_float(x0[4 * m + 2]) + __uint_as_float(x1[4 * m + 2]), v3 = __uint_as_float(x0[4 * m + 3]) + __uint_as_float(x1[4 * m + 3]);
          {
            const float s01 = bit0 ? v0 : v1, s23 = bit0 ? v2 : v3;
            const float r01 = __shfl_xor_sync(0xffffffffu, s01, 1), r23 = __shfl_xor_sync(0xffffffffu, s23, 1);
            v0 = bit0 ? r01 : v0; v1 = bit0 ? v1 : r01;
            v2 = bit0 ? r23 : v2; v3 = bit0 ? v3 : r23;
          }
          {
            const float s02 = bit1 ? v0 : v2, s13 = bit1 ? v1 : v3;
            const float r02 = __shfl_xor_sync(0xffffffffu, s02, 2), r13 = __shfl_xor_sync(0xffffffffu, s13, 2);
            v0 = bit1 ? r02 : v0; v2 = bit1 ? v2 : r02;
            v1 = bit1 ? r13 : v1; v3 = bit1 ? v3 : r13;
          }
          const float pi = v0 + pb[m].x, pf = v1 + pb[m].y, pg = v2 + pb[m].z, po = v3 + pb[m].w;
          const float cn = sigmoid_fast(pf) * (k ? c[1][m] : c[0][m]) + sigmoid_fast(pi) * tanh_fast(pg);
          if (k) c[1][m] = cn;
          else c[0][m] = cn;
          cc[m] = cn;
          h[m] = sigmoid_fast(po) * tanh_fast(cn);
        }
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(tmem_empty);
      const int np = (s + 1) & 1;
      // hand-off: the block through shared memory ([batch row][UNITS + 4 floats], conflict-free 16-byte reads), then every warp
      // writes RPW whole rows of the bf16 operand copy (full 32-byte sectors instead of one partial sector per batch row)
      // top layer: the {h, tag} slots the attention CTAs poll leave straight from the registers, before the staging barrier
      // (0.11 us/step faster than staged whole-row stores)
      if (top && warp_live && unit_ok) {
        const uint32_t tag = (uint32_t)(s + 1);
#pragma unroll
        for (int m = 0; m < 4; ++m)
          if (bm[m] < p.B) ll_store(p.h_ll + (size_t)bm[m] * p.Hs + u, ll_pack(__float_as_uint(h[m]), tag));
      }
      if (warp_live) {
#pragma unroll
        for (int m = 0; m < 4; ++m) s_st[bm[m] * ST_PITCH + jj] = h[m];
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const int r0 = grp * GSZ + (cw * NQ + q) * RPW;  // this warp's rows
      if (lane < 16 && warp_live) {
        const int rw = r0 + lane / CPR, ch = lane % CPR, u0 = nb * UNITS + ch * 8;
        if (rw < p.B && u0 < p.Hs) {
          const float* y = s_st + rw * ST_PITCH + ch * 8;
          const float4 y0 = *reinterpret_cast<const float4*>(y), y1 = *reinterpret_cast<const float4*>(y + 4);
          const __nv_bfloat162 t0 = op2_from_f32(y0.x, y0.y, F16), t1 = op2_from_f32(y0.z, y0.w, F16);
          const __nv_bfloat162 t2 = op2_from_f32(y1.x, y1.y, F16), t3 = op2_from_f32(y1.z, y1.w, F16);
          *reinterpret_cast<uint4*>(p.hbuf[l][np] + (size_t)rw * p.Hs + u0) =
              make_uint4(*reinterpret_cast<const uint32_t*>(&t0), *reinterpret_cast<const uint32_t*>(&t1),
                         *reinterpret_cast<const uint32_t*>(&t2), *reinterpret_cast<const uint32_t*>(&t3));
        }
      }
      if (s == S - 1 && warp_live && unit_ok) {
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          if (bm[m] < p.B) {
            if (p.h_out) p.h_out[((size_t)l * p.Bfull + p.b0 + bm[m]) * p.Hs + u] = h[m];
            if (p.c_out) p.c_out[((size_t)l * p.c_out_rows + p.c_out_b0 + bm[m]) * p.Hs + u] = cc[m];
          }
        }
      }
      if (lead && trole >= 0 && grp == 0) DEC_TRACE(trole, 4);
      if (lead && grp == 0) DEC_TRACE_ALL(2);
      asm volatile("bar.sync 1, 256;" ::: "memory");  // all rows stored; the release below is cumulative over the barrier
      if (lead) {
        red_release_add(my_ready, 1u);
        if (trole >= 0 && grp == 0) DEC_TRACE(trole, 5);
        if (grp == 0) DEC_TRACE_ALL(3);
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) ptx::tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------------------
// attention role (one utterance)
// ------------------------------------------------------------------------------------------------------------
// padded psi row (floats): KS % 32 == 8, so that the 8 lanes of a quarter warp (4 encoder steps x 2 halves, 16-byte
// chunks interleaved between the halves) hit 8 different 16-byte bank groups
__host__ __device__ inline int att_kstride(int D) {
  int ks = (D + 3) & ~3;
  while (ks % 32 != 8) ks += 4;
  return ks;
}
struct AttLayout {
  int WPS, WCS, KS, Up;
  size_t o_wcd, o_h, o_hw, o_qp, o_q, o_score, o_logit, o_bphi, o_bcd, o_red, o_part, o_bop, o_xchg, o_k, total;
};
__host__ __device__ inline size_t att_bop_bytes(int U) { return (size_t)((U + 15) / 16) * 512 + 16; }
__host__ __device__ inline AttLayout att_layout(int Hs, int E, int U, int D, int V, bool k_in, bool wreg, bool hybrid = false, bool split = false) {
  AttLayout a;
  a.WPS = Hs + 8;          // bf16 row strides: multiples of 8 keep every 16-byte chunk aligned
  a.WCS = Hs + E + 8;
  a.KS = att_kstride(D);
  a.Up = (U + 3) & ~3;
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o = (o + bytes + 15) & ~(size_t)15; return at; };
  take(wreg ? 0 : (size_t)D * a.WPS * 2);              // W_phi at offset 0 (not staged when the threads hold it in registers)
  a.o_wcd = take((size_t)V * a.WCS * 2);
  a.o_h = take((size_t)(((Hs + 63) & ~63) + ((E + 63) & ~63)) * 4);  // h, then ctx, each permuted (xpos) and padded to 64 floats
  a.o_hw = take((size_t)DEC_THREADS * 4);              // h in plain order, one 32-value segment per warp (per-warp query partials)
  a.o_qp = take((size_t)(DEC_THREADS / 32) * 64 * 4);  // [warp][64] partial sums of q
  a.o_q = take((size_t)a.KS * 4);
  a.o_score = take((size_t)a.Up * 4);
  a.o_logit = take(64 * 4);
  a.o_bphi = take((size_t)((D + 3) & ~3) * 4);
  a.o_bcd = take(64 * 4);
  a.o_red = take(64 * 4);
  a.o_part = take(4096 * 4);                           // context partial sums, or {mbarrier, TMEM slot, score operand}
  a.o_bop = hybrid ? take(att_bop_bytes(U)) : a.o_part; // hybrid context path: both at once
  // split attention: {2 mbarriers} + own partial [E + 4] + receive buffers [2 step parities][E + 4] floats
  a.o_xchg = split ? take(32 + (size_t)3 * (E + 4) * 4) : o;
  a.o_k = o;
  if (k_in) take((size_t)U * a.KS * 4);
  a.total = o;
  return a;
}

// Half of the encoder steps one CTA of a split pair holds: a whole number of 16-step UMMA K blocks
__host__ __device__ inline int att_split_half(int U) { return ((U + 1) / 2 + 15) / 16 * 16; }

template <int F16>
__device__ void attention_role(const DecParams& p, uint8_t* smem, int b, int rank) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARP = DEC_THREADS / 32;
  const bool split = p.att_split == 2;
  // Split attention (cluster of two CTAs per utterance): this CTA sees only the encoder steps [ub, ub + U) -- "U" below is the LOCAL
  // count; `Ulay` (the first half's size) sizes the shared-memory layout of both ranks.
  const int Utot = p.U;
  const int Ulay = split ? att_split_half(Utot) : Utot;
  const int ub = (split && rank) ? Ulay : 0;
  const int U = split ? (rank ? Utot - Ulay : Ulay) : Utot;
  const int Hs = p.Hs, E = p.E, D = p.D, V = p.V, KC = p.Hs + p.E;
  const int NT = E / 128;                                     // feature tiles
  const int ntm = p.ctx_tmem ? p.ctx_ntm : 0;                 // ... of which in tensor memory
  const bool hybrid = ntm > 0 && ntm * 128 < E;               // (E need not be a multiple of 128 when ntm = 0)
  const AttLayout L = att_layout(Hs, E, Ulay, D, V, p.k_in_smem != 0, p.wreg != 0, hybrid, split);
  const int KS = L.KS, WPS = L.WPS, WCS = L.WCS;
  const int gb = p.b0 + b;  // utterance index in the caller's tensors
  __nv_bfloat16* s_wphi = reinterpret_cast<__nv_bfloat16*>(smem);               // [D][WPS]
  __nv_bfloat16* s_wcd = reinterpret_cast<__nv_bfloat16*>(smem + L.o_wcd);      // [V][WCS]
  float* s_h = reinterpret_cast<float*>(smem + L.o_h);      // [Hs]
  float* s_ctx = s_h + ((Hs + 63) & ~63);                   // [E]
  float* s_hw = reinterpret_cast<float*>(smem + L.o_hw);    // [DEC_THREADS]
  float* s_qp = reinterpret_cast<float*>(smem + L.o_qp);    // [NWARP][64]
  float* s_q = reinterpret_cast<float*>(smem + L.o_q);      // [KS] (zero padded)
  float* s_score = reinterpret_cast<float*>(smem + L.o_score);  // [U]
  float* s_logit = reinterpret_cast<float*>(smem + L.o_logit);  // [V]
  float* s_bphi = reinterpret_cast<float*>(smem + L.o_bphi);
  float* s_bcd = reinterpret_cast<float*>(smem + L.o_bcd);
  float* s_red = reinterpret_cast<float*>(smem + L.o_red);      // [0,16): warp maxima, [16,32): warp sums
  float* s_part = reinterpret_cast<float*>(smem + L.o_part);
  float* s_k = reinterpret_cast<float*>(smem + L.o_k);          // [U][KS] when k_in_smem
  const int e_cc = ntm * 128;         // first feature of the CUDA-core context path (0: all of them; E: none)
  const int Ec = E - e_cc;
  const int ncg = Ec > 0 ? Ec / 8 : 1;  // 8-column groups of enc (CUDA-core context path)
  const int nrg = DEC_THREADS / ncg;  // row groups working in parallel
  // tensor-memory context path: the mbarrier, the TMEM slot and the score operand live in s_part's space (all features in
  // tensor memory: no partial sums needed) or in their own region (hybrid)
  float* s_tm = reinterpret_cast<float*>(smem + L.o_bop);
  uint64_t* ctx_bar = reinterpret_cast<uint64_t*>(s_tm);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_tm + 2);
  uint8_t* s_bop = reinterpret_cast<uint8_t*>(s_tm + 4);     // [2*nks core-K][2][8 rows][16 B]: row 0 = scores (bf16)
  const int nks = (U + 15) / 16;                              // UMMA K steps over the encoder axis
  const int CU = nks * 8;                                     // TMEM columns of one 128-feature tile of enc^T
  const int niss = ntm < 4 ? ntm : 4;  // warps issuing the context UMMAs, one chain of nks instructions per feature tile

  if (!p.wreg)
    for (int i = tid; i < D * Hs; i += DEC_THREADS) s_wphi[(size_t)(i / Hs) * WPS + (i % Hs)] = p.w_phi[i];
  // (prologue copies are vectorised: a segmented decode -- serving pipeline, <eos> early exit -- pays this prologue once per segment)
  if ((KC & 7) == 0) {
    const int rc8 = KC >> 3;  // 16-byte chunks per W_cd row; the padded row stride WCS keeps them aligned
    for (int i = tid; i < V * rc8; i += DEC_THREADS)
      *reinterpret_cast<uint4*>(s_wcd + (size_t)(i / rc8) * WCS + (i % rc8) * 8) = *reinterpret_cast<const uint4*>(p.w_cd + (size_t)(i / rc8) * KC + (i % rc8) * 8);
  } else {
    for (int i = tid; i < V * KC; i += DEC_THREADS) s_wcd[(size_t)(i / KC) * WCS + (i % KC)] = p.w_cd[i];
  }
  for (int i = tid; i < KS; i += DEC_THREADS) s_q[i] = 0.f;
  for (int i = tid; i < D; i += DEC_THREADS) s_bphi[i] = p.b_phi[i];
  for (int i = tid; i < V; i += DEC_THREADS) s_bcd[i] = p.b_cd[i];
  const float* psib = p.psi + ((size_t)gb * Utot + ub) * D;
  if (p.k_in_smem) {
    if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(psib) & 15) == 0)) {  // rows of D floats -> rows of KS floats (zero padded), 16 bytes at a time
      const int rd4 = D >> 2, rk4 = KS >> 2;
      for (int i = tid; i < U * rk4; i += DEC_THREADS) {
        const int u = i / rk4, c4 = i % rk4;
        reinterpret_cast<float4*>(s_k)[i] = c4 < rd4 ? *reinterpret_cast<const float4*>(psib + (size_t)u * D + 4 * c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    } else {
      for (int i = tid; i < U * KS; i += DEC_THREADS) {
        const int u = i / KS, d = i % KS;
        s_k[i] = d < D ? psib[(size_t)u * D + d] : 0.f;
      }
    }
  }
  const int ulen_tot = p.enc_lengths ? min(max(p.enc_lengths[gb], 1), Utot) : Utot;
  const int ulen = min(max(ulen_tot - ub, 0), U);  // (a split pair's second CTA may have nothing valid: its partial sums are zero)
  const __nv_bfloat16* encb = p.enc + ((size_t)b * Utot + ub) * E;
  // split attention: exchange area.  Each CTA writes its partial {context[E], max, sum} into its own `s_own` and into the PEER's
  // receive buffer of the step's parity (st.shared::cluster), one remote mbarrier arrive per warp.
  uint64_t* xbar = reinterpret_cast<uint64_t*>(smem + L.o_xchg);                 // [2]
  float* s_own = reinterpret_cast<float*>(smem + L.o_xchg + 32);                 // [E + 4]
  float* s_recv = s_own + (E + 4);                                               // [2][E + 4]
  const uint32_t peer = (uint32_t)(rank ^ 1);
  const int grp = (p.groups > 1) ? b / p.gsz : 0;  // (see lstm_role_ts: the LSTM CTAs serve the utterance groups alternately)
  uint32_t* ctx_ctr = counter(p, CTR_CTX, grp);
  uint32_t* word_ctr = counter(p, CTR_WORD, grp);
  uint32_t tmem = 0;
  if (p.ctx_tmem) {
    // enc[b]^T -> tensor memory, once: tile t holds features [128t, 128t+128) as TMEM lanes, encoder steps along the
    // columns (two bf16 per 32-bit column) = the A operand of  ctx^T[E,1] = enc^T[E,U] . score[U,1]
    if (tid == 0) {
      ptx::mbar_init(ctx_bar, (uint32_t)niss);
      if (split) {
        ptx::mbar_init(&xbar[0], NWARP);
        ptx::mbar_init(&xbar[1], NWARP);
      }
      ptx::fence_mbar_init();
    }
    if (warp == 0) ptx::tmem_alloc(tmem_slot, 512);
    for (int i = tid; i < nks * 512 / 16; i += DEC_THREADS) reinterpret_cast<uint4*>(s_bop)[i] = make_uint4(0, 0, 0, 0);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    tmem = *tmem_slot;
    const int qd = warp & 3;
    for (int t = warp >> 2; t < ntm; t += NWARP / 4) {
      const __nv_bfloat16* col = encb + t * 128 + qd * 32 + lane;
      // four K blocks (64 encoder steps, 64 two-byte loads) in flight per thread: this strided gather is latency-bound and is paid by
      // every segment of a segmented decode
      for (int ks0 = 0; ks0 < nks; ks0 += 4) {
        uint32_t v[4][8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int u0 = (ks0 + j) * 16 + 2 * i;
            const unsigned short lo = u0 < U ? *reinterpret_cast<const unsigned short*>(col + (size_t)u0 * E) : 0;
            const unsigned short hi = u0 + 1 < U ? *reinterpret_cast<const unsigned short*>(col + (size_t)(u0 + 1) * E) : 0;
            v[j][i] = (uint32_t)lo | ((uint32_t)hi << 16);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (ks0 + j < nks) ptx::tmem_st_32x32b_x8(tmem + ((uint32_t)(qd * 32) << 16) + t * CU + (ks0 + j) * 8, v[j]);
      }
    }
    ptx::tmem_st_wait();
    ptx::tc_fence_before();
  }
  __syncthreads();
  if (split) ptx::cluster_sync();  // the peer's exchange barriers are initialised before anything is sent to them
  ptx::tc_fence_after();

  const int hchunks = Hs >> 3, kchunks = KC >> 3;  // 16-byte chunks (8 bf16) of a W_phi row / W_cd row
  // W_phi in registers (D <= 64, Hs <= 512; otherwise the shared-memory copy): the query GEMV reads only h from shared memory (the
  // 64 KB of W_phi would otherwise be half of the step's shared-memory wavefronts).  Per-warp query partials: warp w owns
  // h[32w, 32w+32) -- the values it polls itself -- and lane l the outputs d = l and l + 32 (32 registers of W_phi), so a warp starts
  // its share of the GEMV the moment ITS OWN 32 values have arrived (the layer-1 CTAs finish up to ~0.5 us apart) instead of after a
  // CTA-wide barrier; the 16 partial sums per output are added after one barrier.
  const bool wreg = p.wreg != 0;
  uint4 wq[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = lane + 32 * (j >> 2), k = 32 * warp + 8 * (j & 3);
    wq[j] = (wreg && d < D && k < Hs) ? *reinterpret_cast<const uint4*>(p.w_phi + (size_t)d * Hs + k) : make_uint4(0, 0, 0, 0);
  }
  const int Dp = (D + 3) & ~3, Vp = (V + 1) & ~1;
  const int nd4 = (D + 3) >> 2;                    // float4 chunks of a psi row

  for (int s = 0; s < p.steps; ++s) {
    const int np = (s + 1) & 1;
    const bool last = (s == p.steps - 1);
    // ---- A: this step's top-layer h, polled straight out of the LSTM epilogue's flag-in-data slots
    if (wreg) {
      float hv = 0.f;
      if (tid < Hs) {
        hv = __uint_as_float(ll_wait(p.h_ll + (size_t)b * Hs + tid, (uint32_t)(s + 1)));
        s_h[xpos(tid)] = hv;  // permuted copy for the character distribution
      }
      s_hw[tid] = hv;
      __syncwarp();
      if (tid == 0) DEC_TRACE_ALL(0);
      if (tid == 0 && b == 0) { DEC_TRACE(2, 0); DEC_TRACE(3, 0); if (p.trace && s < 32) p.trace[(2 * 32 + s) * 8 + 7] = clock64(); }
      // ---- B: q = act(W_phi . h + b_phi)   (model/las_model.py:278): this warp's 32 columns of W_phi x its 32 values of h
      float a0 = 0.f, a1 = 0.f;
      const float4* hx = reinterpret_cast<const float4*>(s_hw + 32 * warp);  // same address in every lane: broadcast loads
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 x0 = hx[2 * j], x1 = hx[2 * j + 1];
        a0 = dot8(wq[j], x0, x1, a0, F16);
        a1 = dot8(wq[4 + j], x0, x1, a1, F16);
      }
      s_qp[warp * 64 + lane] = a0;
      s_qp[warp * 64 + 32 + lane] = a1;
      if (tid == 0 && b == 0) { DEC_TRACE(3, 1); DEC_TRACE(3, 2); }
      __syncthreads();
      if (tid < Dp) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < NWARP; ++w) acc += s_qp[w * 64 + tid];
        if (tid < D) {
          acc += s_bphi[tid];
          s_q[tid] = p.relu ? fmaxf(acc, 0.f) : acc;
        }
      }
    } else {
      if (tid < Hs) s_h[xpos(tid)] = __uint_as_float(ll_wait(p.h_ll + (size_t)b * Hs + tid, (uint32_t)(s + 1)));
      __syncthreads();
      if (tid == 0) DEC_TRACE_ALL(0);
      if (tid == 0 && b == 0) { DEC_TRACE(2, 0); DEC_TRACE(3, 0); if (p.trace && s < 32) p.trace[(2 * 32 + s) * 8 + 7] = clock64(); }

      // ---- B: q = act(W_phi . h + b_phi)   (model/las_model.py:278): 8 lanes per output, interleaved 16-byte chunks
      {
        const int part = tid & 7;
        for (int d = tid >> 3; d < Dp; d += DEC_THREADS / 8) {
          float acc = 0.f;
          if (d < D) {
            const uint4* wr = reinterpret_cast<const uint4*>(s_wphi + (size_t)d * WPS);
#pragma unroll 4
            for (int c = part; c < hchunks; c += 8) {
              const float4* xv = xchunk(s_h, c);
              acc = dot8(lds128(wr + c), xv[0], xv[8], acc, F16);
            }
          }
          if (tid == 0 && b == 0) DEC_TRACE(3, 1);
          acc += __shfl_xor_sync(0xffffffffu, acc, 1);
          acc += __shfl_xor_sync(0xffffffffu, acc, 2);
          acc += __shfl_xor_sync(0xffffffffu, acc, 4);
          if (tid == 0 && b == 0) DEC_TRACE(3, 2);
          if (part == 0 && d < D) {
            acc += s_bphi[d];
            s_q[d] = p.relu ? fmaxf(acc, 0.f) : acc;
          }
        }
      }
    }
    __syncthreads();
    if (tid == 0 && b == 0) { DEC_TRACE(2, 1); DEC_TRACE(3, 3); }

    // ---- C: energy[u] = <q, psi[b,u,:]>  (:289-291), two lanes per encoder step, then a softmax over the encoder
    //         steps (:292) with one exchange of warp maxima and one of warp sums
    float ev[ATT_MAXP];
    float lmax = -INFINITY;
    float m_loc = -INFINITY;  // this CTA's maximum energy (split attention: exchanged with the peer)
    {
      const int half = tid & 1;
#pragma unroll
      for (int ps = 0; ps < ATT_MAXP; ++ps) {
        ev[ps] = -INFINITY;
        if (ps * 256 < U) {
          const int u = ps * 256 + (tid >> 1);
          float acc = 0.f;
          if (u < ulen) {
            if (p.k_in_smem) {
              const float4* kr = reinterpret_cast<const float4*>(s_k + (size_t)u * KS);
              const float4* qv = reinterpret_cast<const float4*>(s_q);
              float acc2 = 0.f;
#pragma unroll 4
              for (int c = half; c < nd4; c += 2) {  // q and the psi rows are zero padded to KS
                const float4 kv = kr[c], q4 = qv[c];
                acc = fmaf(q4.x, kv.x, acc); acc2 = fmaf(q4.y, kv.y, acc2); acc = fmaf(q4.z, kv.z, acc); acc2 = fmaf(q4.w, kv.w, acc2);
              }
              acc += acc2;
            } else {
              const float* kr = psib + (size_t)u * D;
              for (int d = half; d < D; d += 2) acc = fmaf(s_q[d], kr[d], acc);
            }
          }
          acc += __shfl_xor_sync(0xffffffffu, acc, 1);
          if (u < ulen) ev[ps] = acc;
          lmax = fmaxf(lmax, ev[ps]);
        }
      }
      if (tid == 0 && b == 0) DEC_TRACE(3, 4);
      lmax = warp_max(lmax);
      if (lane == 0) s_red[warp] = lmax;
      __syncthreads();
      if (tid == 0 && b == 0) DEC_TRACE(3, 5);
      float m;
      {
        const float4* r4 = reinterpret_cast<const float4*>(s_red);
        const float4 a = r4[0], b4 = r4[1], c4 = r4[2], d4 = r4[3];
        m = fmaxf(fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)), fmaxf(fmaxf(b4.x, b4.y), fmaxf(b4.z, b4.w)));
        m = fmaxf(m, fmaxf(fmaxf(fmaxf(c4.x, c4.y), fmaxf(c4.z, c4.w)), fmaxf(fmaxf(d4.x, d4.y), fmaxf(d4.z, d4.w))));
      }
      m_loc = m;
      // p[u] = exp(e[u] - max) goes to the context reduction unnormalised (bf16 operand of the UMMA / fp32 for the
      // CUDA-core path); the sum arrives through the same barrier and the 1/sum scaling is applied to the context
      float lsum = 0.f;
#pragma unroll
      for (int ps = 0; ps < ATT_MAXP; ++ps) {
        ev[ps] = (ev[ps] == -INFINITY) ? 0.f : __expf(ev[ps] - m);
        if (half == 0) {
          lsum += ev[ps];
          const int u = ps * 256 + (tid >> 1);
          if (u < U) {
            if (ntm > 0) *reinterpret_cast<__nv_bfloat16*>(s_bop + (u >> 3) * 256 + (u & 7) * 2) = op_from_f32(ev[ps], F16);
            if (Ec > 0) s_score[u] = ev[ps];
          }
        }
      }
      lsum = warp_sum(lsum);
      if (lane == 0) s_red[16 + warp] = lsum;
    }
    if (p.ctx_tmem) ptx::fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0 && b == 0) { DEC_TRACE(3, 6); DEC_TRACE(2, 2); }
    if (tid == 0) DEC_TRACE_ALL(1);
    float inv, sum_loc;
    {
      const float4* r4 = reinterpret_cast<const float4*>(s_red + 16);
      const float4 a = r4[0], b4 = r4[1], c4 = r4[2], d4 = r4[3];
      sum_loc = ((a.x + a.y) + (a.z + a.w)) + ((b4.x + b4.y) + (b4.z + b4.w)) + ((c4.x + c4.y) + (c4.z + c4.w)) + ((d4.x + d4.y) + (d4.z + d4.w));
      inv = split ? 1.0f : 1.0f / sum_loc;  // split attention: the partial context stays unnormalised until the two halves are combined
    }

    // ---- D: context[e] = sum_u score[u] * enc[b,u,e]  (:293-297)
    if (warp < niss) {
      // scores (bf16) are row 0 of a 16-row K-major operand in shared memory:
      // D_t[128 features, 16] = enc^T tile (TMEM) . scores^T ; column 0 of each accumulator is the context.
      // One issuing warp per feature tile (up to four): a chain of N = 16 instructions is paced by its issuing thread (~27-58
      // cycles per instruction against ~8 in the pipe, tools/microbench_mma_insitu.cu), so independent chains issued from
      // different warps overlap.  Each issuer commits to ctx_bar (initialised with one arrival per issuer).
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const UmmaLayout lb{0, 256, 128, 0};
        const uint32_t idesc = umma_idesc_bf16(128, 16, F16);
        // Consecutive K steps are 512 bytes apart in the score operand and 8 columns apart in tensor memory, so both operands
        // advance by constants: 32 in the descriptor's 16-byte address field (which cannot carry out of its 14 bits: shared
        // memory ends below 256 KB) and 8 in the tensor-memory address.
        const uint64_t bd0 = umma_smem_desc(lb, ptx::smem_u32(s_bop), 0);
        for (int t = warp; t < ntm; t += niss) {
          uint64_t bd = bd0;
          uint32_t a = tmem + t * CU;
          const uint32_t dcol = tmem + ntm * CU + t * 16;
#pragma unroll 4
          for (int ks = 0; ks < nks; ++ks) {
            ptx::umma_bf16_ts(dcol, a, bd, idesc, ks != 0);
            a += 8;
            bd += 32;
          }
        }
        ptx::umma_commit(ctx_bar);
      }
      __syncwarp();
    }
    // The h half of the logits is evaluated together with the context half, AFTER the context has been published: the context UMMAs
    // (four issuing warps) finish in ~0.9 us, sooner than a GEMV squeezed in next to them, and the publish must not wait for it.
    const bool owner = !split || rank == 0;  // of a split pair only the first CTA publishes the context and evaluates the logits / feedback
    __nv_bfloat16* xr = p.xbuf[np] + (size_t)b * E;        // next LSTM input: context row
    __nv_bfloat16* wr_next = p.wbuf[np] + (size_t)b * DEC_VP;  // ... and dense word row (padded to 64)
    if (Ec > 0) {
      // CUDA-core part, features [e_cc, E): 16-byte bf16 loads of enc[b] (L2 resident), nrg row groups in parallel, 8 loads in
      // flight.  In the hybrid case this runs while the tensor pipe reduces the features below e_cc.
      const int rg = tid / ncg, cg = tid % ncg;
      float acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.f;
      if (rg < nrg) {
        const uint4* col = reinterpret_cast<const uint4*>(encb + e_cc + cg * 8);
        const int rstride = E / 8;  // uint4 per row
        for (int u = rg; u < ulen; u += 8 * nrg) {
          uint4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int uu = u + j * nrg;
            v[j] = (uu < ulen) ? __ldg(col + (size_t)uu * rstride) : make_uint4(0, 0, 0, 0);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int uu = u + j * nrg;
            const float a = (uu < ulen) ? s_score[uu] : 0.f;  // unnormalised exp(e - max)
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v[j]);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float2 f = op2_to_f32(h2[i], F16);
              acc[2 * i] = fmaf(a, f.x, acc[2 * i]);
              acc[2 * i + 1] = fmaf(a, f.y, acc[2 * i + 1]);
            }
          }
        }
        float4* dst = reinterpret_cast<float4*>(s_part + (size_t)rg * Ec + cg * 8);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
      }
    }
    if (ntm > 0) {
      ptx::mbar_wait(ctx_bar, (uint32_t)(s & 1));
      ptx::tc_fence_after();
      if (tid == 0 && b == 0 && !hybrid) DEC_TRACE(2, 3);
      const int qd = warp & 3;
      for (int t = warp >> 2; t < ntm; t += NWARP / 4) {
        const uint32_t r = ptx::tmem_ld_32x32b_x1(tmem + ((uint32_t)(qd * 32) << 16) + ntm * CU + t * 16);
        ptx::tmem_ld_wait();
        const int e = t * 128 + qd * 32 + lane;
        const float cv = __uint_as_float(r) * inv;
        if (split) {  // partial context: own copy + the peer's receive buffer of this step's parity
          s_own[e] = cv;
          asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ptx::mapa(ptx::smem_u32(s_recv + (size_t)(s & 1) * (E + 4) + e), peer)), "f"(cv) : "memory");
        } else {
          s_ctx[xpos(e)] = cv;
          if (last && p.ctx_out) p.ctx_out[(size_t)gb * E + e] = cv;
        }
      }
      ptx::tc_fence_before();
      if (split) {
        if (tid == 0) {  // this half's softmax statistics travel with warp 0's arrive
          s_own[E] = m_loc;
          s_own[E + 1] = sum_loc;
          const uint32_t dst = ptx::mapa(ptx::smem_u32(s_recv + (size_t)(s & 1) * (E + 4) + E), peer);
          asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(dst), "f"(m_loc) : "memory");
          asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(dst + 4), "f"(sum_loc) : "memory");
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_remote(ptx::mapa(ptx::smem_u32(&xbar[s & 1]), peer));  // release.cluster: cumulative over the warp's stores
      }
    }
    float att_scale = inv;  // factor that turns exp(e - local max) into the attention weight
    if (split) {
      // combine the two halves: M = max(m0, m1), w_r = exp(m_r - M), S = s0 w0 + s1 w1, context = (c0 w0 + c1 w1) / S
      ptx::mbar_wait_cluster(&xbar[s & 1], (uint32_t)((s >> 1) & 1));
      __syncthreads();  // own partial complete as well
      const float* rv = s_recv + (size_t)(s & 1) * (E + 4);
      const float m_peer = rv[E], s_peer = rv[E + 1];
      const float M = fmaxf(m_loc, m_peer);
      const float w_own = (m_loc == -INFINITY) ? 0.f : __expf(m_loc - M), w_peer = (m_peer == -INFINITY) ? 0.f : __expf(m_peer - M);
      const float rS = 1.0f / (sum_loc * w_own + s_peer * w_peer);
      att_scale = w_own * rS;
      for (int e = tid; e < E; e += DEC_THREADS) {
        const float cv = (s_own[e] * w_own + rv[e] * w_peer) * rS;
        s_ctx[xpos(e)] = cv;
        if (rank == 0 && last && p.ctx_out) p.ctx_out[(size_t)gb * E + e] = cv;
      }
    }
    if (Ec > 0) {
      __syncthreads();
      if (tid == 0 && b == 0) DEC_TRACE(2, 3);
      for (int ee = tid; ee < Ec; ee += DEC_THREADS) {
        float acc = 0.f;
        for (int rg = 0; rg < nrg; ++rg) acc += s_part[(size_t)rg * Ec + ee];
        acc *= inv;
        s_ctx[xpos(e_cc + ee)] = acc;
        if (last && p.ctx_out) p.ctx_out[(size_t)gb * E + e_cc + ee] = acc;
      }
    }
    __syncthreads();
    // publish the context row (bf16) with 16-byte stores from the first E/8 threads -- few, sector-filling writes keep the
    // release short -- then release: layer 0 starts its context GEMM while the character distribution is evaluated here
    if (owner) {
      const int npub = E >> 3, nsync = (npub + 31) & ~31;
      if (tid < nsync) {
        if (tid < npub) {
          const float4* xv = xchunk(s_ctx, tid);
          const float4 lo = xv[0], hi = xv[8];
          const __nv_bfloat162 p0 = op2_from_f32(lo.x, lo.y, F16), p1 = op2_from_f32(lo.z, lo.w, F16);
          const __nv_bfloat162 p2 = op2_from_f32(hi.x, hi.y, F16), p3 = op2_from_f32(hi.z, hi.w, F16);
          *reinterpret_cast<uint4*>(xr + 8 * tid) =
              make_uint4(*reinterpret_cast<const uint32_t*>(&p0), *reinterpret_cast<const uint32_t*>(&p1),
                         *reinterpret_cast<const uint32_t*>(&p2), *reinterpret_cast<const uint32_t*>(&p3));
        }
        if (nsync > 32) asm volatile("bar.sync 2, %0;" ::"r"(nsync) : "memory");
        else __syncwarp();
        if (tid == 0) {
          red_release_add(ctx_ctr, 1u);
          DEC_TRACE_ALL(3);
          if (b == 0) DEC_TRACE(2, 4);
        }
      }
    }

    if (p.attn && (tid & 1) == 0) {  // attention record (:292, returned to the caller): off the critical path, after the publish
#pragma unroll
      for (int ps = 0; ps < ATT_MAXP; ++ps) {
        const int u = ps * 256 + (tid >> 1);
        if (u < U) p.attn[((size_t)(p.s0 + s) * p.Bfull + gb) * Utot + ub + u] = ev[ps] * att_scale;
      }
    }

    // ---- E: logits = W_cd . [h || context] + b_cd, 16 lanes per output  (:181).  Warp 0 has just issued the release of the context
    // (its thread 0 stalls ~0.4 us on it), so it takes no part: warps 1-15 hold the 30 output groups, synchronise among themselves
    // (named barrier, 480 threads) and warp 1 goes on to the feedback; warp 0 only waits for them before it touches the next step's h.
    constexpr int FW = 1;  // the warp that evaluates the feedback (phase F)
    if (!owner) continue;
    if (warp != 0) {
      const int part = tid & 15;
      for (int v = (tid - 32) >> 4; v < Vp; v += (DEC_THREADS - 32) / 16) {
        float acc = 0.f;
        if (v < V) {
          const uint4* wr = reinterpret_cast<const uint4*>(s_wcd + (size_t)v * WCS);
#pragma unroll 4
          for (int c = part; c < kchunks - hchunks; c += 16) {
            const float4* xv = xchunk(s_ctx, c);
            acc = dot8(lds128(wr + hchunks + c), xv[0], xv[8], acc, F16);
          }
#pragma unroll 4
          for (int c = part; c < hchunks; c += 16) {
            const float4* xv = xchunk(s_h, c);
            acc = dot8(lds128(wr + c), xv[0], xv[8], acc, F16);
          }
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
        acc += __shfl_xor_sync(0xffffffffu, acc, 8);
        if (part == 0 && v < V) s_logit[v] = acc + s_bcd[v];
      }
      asm volatile("bar.sync 4, %0;" ::"n"(DEC_THREADS - 32) : "memory");   // logits complete (warps 1-15)
      asm volatile("bar.arrive 5, %0;" ::"n"(DEC_THREADS) : "memory");      // ... and s_h / s_ctx no longer read: warp 0 may move on
    } else {
      asm volatile("bar.sync 5, %0;" ::"n"(DEC_THREADS) : "memory");
    }
    if (tid == FW * 32 && b == 0) DEC_TRACE(2, 5);

    // ---- F: warp FW: log_softmax (:182), argmax / teacher forcing (:216-227), the word fed back (:236).  The other
    //         warps go straight on to poll for the next step's h.
    if (warp == FW) {
      // Greedy feedback first: argmax(log_softmax(z)) = argmax(z), so the token leaves for layer 0 (whose epilogue needs it
      // ~2.5 us after the context was published) before the log-sum-exp, the log-prob stores and the loss term are done.
      const bool early_tok = p.word_gather && !p.gt_index && !p.gt_dense && p.decode_mode != LAS_DECODE_SAMPLE;
      float lm = -INFINITY;
      int li = 0x7fffffff;
      for (int v = lane; v < V; v += 32) {
        const float z = s_logit[v];
        if (z > lm) { lm = z; li = v; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, lm, o);
        const int oi = __shfl_xor_sync(0xffffffffu, li, o);
        if (ov > lm || (ov == lm && oi < li)) { lm = ov; li = oi; }
      }
      if (early_tok) {
        for (int i = lane; i < p.ncl; i += 32) ll_store(p.tok_ll + (size_t)i * p.B + b, ll_pack((uint32_t)li, (uint32_t)(s + 1)));
        if (lane == 0 && b == 0) DEC_TRACE(2, 6);
      }
      float ls = 0.f;
      for (int v = lane; v < V; v += 32) ls += __expf(s_logit[v] - lm);
      ls = warp_sum(ls);
      const float lse = lm + __logf(ls);
      for (int v = lane; v < V; v += 32) p.logp[((size_t)(p.s0 + s) * p.Bfull + gb) * V + v] = s_logit[v] - lse;
      int bi = li;  // ties -> lowest index, as torch.topk / argmax on the host
      if (p.nll_terms && lane == 0) {  // NLLLoss(ignore_index=0) term of this (step, utterance)
        const int sg = p.s0 + s;
        const int lab = (p.nll_labels && sg < p.nll_steps) ? p.nll_labels[(size_t)gb * p.nll_steps + sg] : 0;
        p.nll_terms[(size_t)sg * p.Bfull + gb] = (lab > 0 && lab < V) ? -(s_logit[lab] - lse) : 0.f;
      }
      if (p.decode_mode == LAS_DECODE_SAMPLE && !p.gt_index && !p.gt_dense) {
        // decode_mode 2 (:229-234): feed back (and report) a draw from Categorical(probs = log-probs); s_logit -> log-probs first
        __syncwarp();
        for (int v = lane; v < V; v += 32) s_logit[v] -= lse;
        __syncwarp();
        if (lane == 0) bi = las_sample_logp_as_probs(s_logit, V, las_uniform(p.sample_seed, (uint32_t)(p.s0 + s), (uint32_t)gb));
        bi = __shfl_sync(0xffffffffu, bi, 0);
        for (int v = lane; v < V; v += 32) s_logit[v] += lse;  // the raw-feedback branch below expects logits
        __syncwarp();
      }
      if (lane == 0 && p.tokens) p.tokens[(size_t)(p.s0 + s) * p.Bfull + gb] = bi;
      if (p.word_gather) {
        // the word is an index: layer 0's epilogue adds the matching column of W_word itself
        const int fed = p.gt_index ? p.gt_index[(size_t)gb * p.gt_steps + p.s0 + s] : bi;
        if (last && lane == 0 && p.tok_carry) p.tok_carry[b] = fed;
        if (!p.gt_index && !early_tok)
          for (int i = lane; i < p.ncl; i += 32) ll_store(p.tok_ll + (size_t)i * p.B + b, ll_pack((uint32_t)fed, (uint32_t)(s + 1)));
        if (last && p.word_out)
          for (int i = lane; i < V; i += 32) p.word_out[(size_t)gb * V + i] = (i == fed) ? 1.f : 0.f;
      } else {
        for (int i = lane; i < DEC_VP; i += 32) {
          float val = 0.f;
          if (i < V) {
            if (p.gt_dense) val = p.gt_dense[((size_t)gb * p.gt_steps + p.s0 + s) * V + i];
            else if (p.decode_mode == LAS_DECODE_RAW) val = s_logit[i] - lse;
            else val = (i == bi) ? 1.f : 0.f;
            if (last && p.word_out) p.word_out[(size_t)gb * V + i] = val;
          }
          wr_next[i] = op_from_f32(val, F16);
        }
        __syncwarp();
        if (lane == 0) red_release_add(word_ctr, 1u);
      }
      if (!early_tok && lane == 0 && b == 0) DEC_TRACE(2, 6);
    }
  }
  if (p.ctx_tmem) {
    ptx::tc_fence_before();
    __syncthreads();
    if (split) ptx::cluster_sync();  // no CTA leaves while its peer could still write into its receive buffers
    if (warp == 0) ptx::tmem_dealloc(tmem, 512);
  }
}

template <int F16>
__global__ void __launch_bounds__(DEC_THREADS, 1) speller_decode_persistent_kernel(const __grid_constant__ DecParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment (SWIZZLE_128B atoms) as an offset from the __shared__ symbol, so that the compiler keeps the
  // address space and emits LDS/STS instead of generic loads
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int n_lstm = p.sl * p.ncl;
  if (p.stop && *reinterpret_cast<const volatile int32_t*>(p.stop) != 0) return;  // written before this launch: every CTA sees the same value
  if ((int)blockIdx.x < n_lstm) lstm_role_ts<F16>(p, smem, blockIdx.x / p.ncl, blockIdx.x % p.ncl);
  else if (p.att_split == 2) attention_role<F16>(p, smem, (blockIdx.x - n_lstm) >> 1, (blockIdx.x - n_lstm) & 1);
  else attention_role<F16>(p, smem, blockIdx.x - n_lstm, 0);
}

// ---- pack kernels ------------------------------------------------------------------------------------------
// LSTM layer weights -> per-CTA swizzled atoms.  K order: [h part (Hs) | input part], each padded to 64-wide atoms.
__global__ void pack_dec_w_kernel(const float* w_ih, const float* w_hh, uint8_t* img, int l, int Hs, int E, int V, int ncl, int f16) {
  const int nh = (Hs + 63) / 64;
  const int nx = (l == 0) ? (DEC_VP + E + 63) / 64 : (Hs + 63) / 64;
  const int natoms = nh + nx;
  const int Kx = (l == 0) ? V + E : Hs;  // row length of w_ih
  const size_t n = (size_t)ncl * natoms * DEC_NW * 64;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int kk = (int)(i % 64);
    const int rr = (int)((i / 64) % DEC_NW);
    const int at = (int)((i / (64 * DEC_NW)) % natoms);
    const int nb = (int)(i / ((size_t)64 * DEC_NW * natoms));
    const int unit = nb * DEC_UNITS + (rr >> 2), gate = rr & 3;
    const size_t srow = (size_t)gate * Hs + unit;
    float val = 0.f;
    if (at < nh) {
      const int k = at * 64 + kk;
      if (k < Hs) val = w_hh[srow * Hs + k];
    } else {
      const int kx = (at - nh) * 64 + kk;
      if (l == 0) {
        if (kx < DEC_VP) { if (kx < V) val = w_ih[srow * Kx + kx]; }
        else if (kx - DEC_VP < E) val = w_ih[srow * Kx + V + (kx - DEC_VP)];
      } else if (kx < Hs) {
        val = w_ih[srow * Kx + kx];
      }
    }
    const size_t off = ((size_t)nb * natoms + at) * WATOM_BYTES + (size_t)(rr >> 3) * 1024 + (rr & 7) * 128 + ((((kk >> 3) ^ (rr & 7)) & 7) << 4) +
                       (kk & 7) * 2;
    *reinterpret_cast<__nv_bfloat16*>(img + off) = op_from_f32(val, f16);
  }
}
__global__ void pack_dec_bias_kernel(const float* b_ih, const float* b_hh, float* dst, int Hs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 4 * Hs) return;
  const int nb = i / DEC_NW, rr = i % DEC_NW;
  const int unit = nb * DEC_UNITS + (rr >> 2), gate = rr & 3;
  dst[i] = b_ih[gate * Hs + unit] + b_hh[gate * Hs + unit];
}

// initial decoder input / state in the kernel's operand formats
__global__ void dec_init_kernel(DecParams p, const float* enc_f32, const float* word_in, const float* ctx_in, const float* h_in) {
  const int b = blockIdx.x, gb = p.b0 + blockIdx.x;
  __nv_bfloat16* xr = p.xbuf[0] + (size_t)b * p.E;
  __nv_bfloat16* wr = p.wbuf[0] + (size_t)b * DEC_VP;
  for (int i = threadIdx.x; i < DEC_VP + p.E; i += blockDim.x) {
    if (i < DEC_VP) wr[i] = op_from_f32((i < p.V) ? (word_in ? word_in[(size_t)gb * p.V + i] : (i == 0 ? 1.f : 0.f)) : 0.f, p.f16);  // <sos> = index 0
    else xr[i - DEC_VP] = op_from_f32(ctx_in ? ctx_in[(size_t)gb * p.E + (i - DEC_VP)] : enc_f32[(size_t)gb * p.U * p.E + (i - DEC_VP)], p.f16);  // enc[:,0,:]
  }
  for (int l = 0; l < p.sl; ++l)
    for (int i = threadIdx.x; i < p.Hs; i += blockDim.x)
      p.hbuf[l][0][(size_t)b * p.Hs + i] = op_from_f32(h_in ? h_in[((size_t)l * p.Bfull + gb) * p.Hs + i] : 0.f, p.f16);
}

// The packed image: Hs / 16 blocks of 16 units (a 32-unit LSTM CTA reads two of them)
struct Shape {
  int nblk, natoms[MAX_SL];
  size_t w_bytes[MAX_SL];
};
Shape shape_of(const las_speller_dims* d) {
  Shape s;
  s.nblk = d->Hs / DEC_UNITS;
  for (int l = 0; l < d->sl && l < MAX_SL; ++l) {
    const int nh = (d->Hs + 63) / 64;
    const int nx = (l == 0) ? (DEC_VP + d->E + 63) / 64 : (d->Hs + 63) / 64;
    s.natoms[l] = nh + nx;
    s.w_bytes[l] = (size_t)s.nblk * s.natoms[l] * WATOM_BYTES;
  }
  return s;
}
struct RingCfg {
  int box_rows, stage_bytes, nstages;
  size_t smem;
};
// shared memory of an LSTM CTA with `units` hidden units whose activation boxes have `rows` batch rows: the own-h (+ word) atoms of
// 4 * units gate rows (+ the 8 KB pad of the 16-unit form), the bias, the barriers, the epilogue's staging block [64 rows][units + 4] and one ring slot per atom of the larger
// streamed part (own h: ceil(Hs/64); context / lower h: ceil(E/64)) + the word slot, so that a whole step's critical input can be in
// flight at once
RingCfg ring_cfg(const las_speller_dims* d, int units, int rows) {
  const int nh = (d->Hs + 63) / 64, nc0 = (d->E + 63) / 64;
  RingCfg r;
  r.box_rows = rows;
  r.stage_bytes = rows * 128;
  r.nstages = (nh > nc0 ? nh : nc0) + 1;
  const size_t fixed = (size_t)(nh + 1) * units * 4 * 128 + (units == DEC_UNITS ? WATOM_BYTES : 0) + 4 * units * 4 + (DEC_MAX_STAGES + 4) * 8 + 64 + 64 * (units + 4) * 4;
  r.smem = fixed + (size_t)r.nstages * r.stage_bytes;
  return r;
}
// The form of the persistent decoder's LSTM CTAs for a launch of Bc utterances, decided here alone; the one reader of debug keys
// 19 and 30.  More than 32 utterances go through as two utterance groups of 32 rows (key 19 = 0: in lockstep, 64-row boxes).  A CTA
// can take 32 hidden units (128 gate rows: all lanes of its M = 128 MMAs) wherever one iteration serves at most 32 rows, so that the
// epilogue's eight warps still cover one group with four cells per thread -- half the LSTM CTAs of the 16-unit form.  It does so only
// for a launch that shares the chip with the next batch's listener (`beside`, fast_pipeline.cu), where the SMs it frees are what the
// listener runs on.  A decoder alone keeps 16 units: there the 32-unit form measured slower at Hs = 512 (DESIGN.md 4a).
struct LstmPlan {
  int groups, gsz, units, ncl;
};
LstmPlan lstm_plan(const las_speller_dims* d, int Bc, bool beside) {
  const DebugOptions& o = debug_options();
  LstmPlan lp;
  lp.groups = (Bc > 32 && o.dec_groups != 0) ? 2 : 1;
  lp.gsz = (lp.groups == 2 || Bc <= 32) ? 32 : 64;
  const bool wide = beside && lp.gsz <= 32 && ring_cfg(d, 32, lp.gsz).smem <= 224 * 1024;
  lp.units = o.dec_units ? o.dec_units : (wide ? 32 : 16);
  lp.ncl = (d->Hs + lp.units - 1) / lp.units;
  return lp;
}
// the launch group size the plan is made for when the batch is split into several launches (fast_speller_max_group)
int plan_rows(const las_speller_dims* d) { return d->B < 64 ? d->B : 64; }
bool att_wreg(const las_speller_dims* d) { return d->D <= DEC_THREADS / 8 && d->Hs <= 512; }
size_t att_smem(const las_speller_dims* d, bool k_in, bool hybrid = false, bool split = false) {
  return att_layout(d->Hs, d->E, split ? att_split_half(d->U) : d->U, d->D, d->V, k_in, att_wreg(d), hybrid, split).total + 64;
}
// Tensor-memory geometry of the context path for `U` encoder steps per CTA: feature tiles of enc^T that fit the 512 columns
int ctx_tiles_fit(int U, int E) {
  if (E % 128 != 0) return 0;
  const int nks = (U + 15) / 16, NT = E / 128;
  int ntm = 512 / (nks * 8 + 16);
  if (ntm > NT) ntm = NT;
  if (ntm == NT && att_bop_bytes(U) > 4096 * 4) ntm = 0;
  return ntm;
}
// The form of the persistent decoder's attention CTAs, decided here alone; the one reader of debug keys 2 and 11
struct AttPlan {
  int split, ntm;                // CTAs per utterance; 128-feature tiles of enc[b]^T in tensor memory (hybrid: 0 < ntm < E/128)
  bool hybrid, k_in_smem, wreg;
  size_t smem;                   // the attention CTA's dynamic shared memory
};
AttPlan att_plan(const las_speller_dims* d, int n_lstm) {
  const DebugOptions& o = debug_options();
  const int NT = d->E / 128;
  // Long encoders: when one CTA cannot hold all of enc[b]^T in tensor memory but half of the encoder steps fit (U <= 448 at E = 512),
  // a cluster of two CTAs attends each utterance (flash-decoding style partial softmax, combined through DSMEM) -- provided the LSTM
  // CTAs pair up (even count) and the chip has room for two attention CTAs per utterance.
  if (o.att_split && o.ctx_tmem && d->E % 128 == 0 && ctx_tiles_fit(d->U, d->E) != NT && ctx_tiles_fit(att_split_half(d->U), d->E) == NT &&
      n_lstm % 2 == 0 && n_lstm + 2 <= sm_count() && att_smem(d, true, false, true) <= 220 * 1024)
    return {2, NT, false, true, att_wreg(d), att_smem(d, true, false, true)};
  // all feature tiles of enc[b]^T in tensor memory when they fit its 512 columns (U <= 224 at E = 512); otherwise as many as fit,
  // the rest on the CUDA cores (hybrid; needs the score operand in its own shared-memory region), or none where that does not fit
  int ntm = o.ctx_tmem ? ctx_tiles_fit(d->U, d->E) : 0;
  if (ntm > 0 && ntm < NT && (512 % ((d->E - ntm * 128) / 8)) != 0) ntm = 0;
  bool hybrid = ntm > 0 && ntm < NT, k_in_smem = att_smem(d, true, hybrid) <= 220 * 1024;
  if (hybrid && att_smem(d, k_in_smem, true) > 220 * 1024) { ntm = 0; hybrid = false; k_in_smem = att_smem(d, true) <= 220 * 1024; }
  return {1, ntm, hybrid, k_in_smem, att_wreg(d), att_smem(d, k_in_smem, hybrid)};
}
int supported(const las_speller_dims* d) {
  LAS_REQUIRE(d->sl <= MAX_SL, "LAS_MODE_BF16 speller supports at most %d layers (sl=%d)", MAX_SL, d->sl);
  LAS_REQUIRE(d->Hs % 16 == 0 && d->Hs <= 512, "LAS_MODE_BF16 speller needs hidden_size %% 16 == 0 and <= 512 (Hs=%d); use LAS_MODE_FP32", d->Hs);
  LAS_REQUIRE(d->V <= DEC_VP, "LAS_MODE_BF16 speller supports vocabularies up to %d (V=%d)", DEC_VP, d->V);
  LAS_REQUIRE(d->E % 8 == 0 && d->E / 8 <= DEC_THREADS, "LAS_MODE_BF16 speller needs E %% 8 == 0 and E <= 4096 (E=%d)", d->E);
  LAS_REQUIRE(d->U <= ATT_MAXP * 256, "LAS_MODE_BF16 speller supports at most %d encoder steps (U=%d)", ATT_MAXP * 256, d->U);
  LAS_REQUIRE(att_smem(d, false) <= 220 * 1024 && ring_cfg(d, 16, 64).smem <= 224 * 1024 && ring_cfg(d, 16, 64).nstages <= DEC_MAX_STAGES,
              "LAS_MODE_BF16 speller: model does not fit shared memory (U=%d, Hs=%d)", d->U, d->Hs);
  return LAS_OK;
}

struct SpellerPackFast {
  uint8_t* w_img[MAX_SL];
  float* bias[MAX_SL];
  __nv_bfloat16* w_phi;
  __nv_bfloat16* w_cd;
  __nv_bfloat16* w_psi;
  size_t bytes;
};
SpellerPackFast pack_layout(const las_speller_dims* d, void* base) {
  SpellerPackFast p;
  const Shape s = shape_of(d);
  Carver cv(base);
  for (int l = 0; l < d->sl && l < MAX_SL; ++l) {
    p.w_img[l] = cv.take<uint8_t>(s.w_bytes[l]);
    p.bias[l] = cv.take<float>(4 * (size_t)d->Hs);
  }
  p.w_phi = cv.take<__nv_bfloat16>((size_t)d->D * d->Hs);
  p.w_cd = cv.take<__nv_bfloat16>((size_t)d->V * (d->Hs + d->E) + 8);
  p.w_psi = cv.take<__nv_bfloat16>((size_t)d->D * d->E);
  p.bytes = cv.total();
  return p;
}
struct SpellerWsFast {
  __nv_bfloat16* enc_bf16;
  __nv_bfloat16* hbuf[MAX_SL][2];
  __nv_bfloat16* xbuf[2];
  __nv_bfloat16* wbuf[2];
  uint8_t* flags;      // one block cleared per launch: counters, token slots, h slots
  size_t flag_bytes;
  uint32_t* sync;
  u64* tok_ll;
  u64* h_ll;
  float* c_carry;      // [sl, B, Hs] cell state between the segments of a segmented decode
  int32_t* tok_carry;  // [B] token fed back by the previous segment's last step
  int32_t* stop;       // <eos> early exit: [0] stop flag, [1] steps this launch group decoded, [2..66) per-utterance done flags
  size_t bytes;
};
SpellerWsFast ws_layout(const las_speller_dims* d, void* base) {
  SpellerWsFast w;
  Carver cv(base);
  w.enc_bf16 = cv.take<__nv_bfloat16>((size_t)d->B * d->U * d->E);
  for (int l = 0; l < MAX_SL; ++l)
    for (int k = 0; k < 2; ++k) w.hbuf[l][k] = cv.take<__nv_bfloat16>((size_t)d->B * d->Hs);
  for (int k = 0; k < 2; ++k) w.xbuf[k] = cv.take<__nv_bfloat16>((size_t)d->B * d->E);
  for (int k = 0; k < 2; ++k) w.wbuf[k] = cv.take<__nv_bfloat16>((size_t)d->B * DEC_VP);
  const size_t sync_bytes = sizeof(uint32_t) * 32 * N_CTR * 2 /* utterance groups */, tok_bytes = align_up(sizeof(u64) * (size_t)d->B * (d->Hs / DEC_UNITS), 256);
  w.flag_bytes = sync_bytes + tok_bytes + sizeof(u64) * (size_t)d->B * d->Hs;
  w.flags = cv.take<uint8_t>(w.flag_bytes);
  w.sync = reinterpret_cast<uint32_t*>(w.flags);
  w.tok_ll = reinterpret_cast<u64*>(w.flags ? w.flags + sync_bytes : nullptr);
  w.h_ll = reinterpret_cast<u64*>(w.flags ? w.flags + sync_bytes + tok_bytes : nullptr);
  w.c_carry = cv.take<float>((size_t)MAX_SL * d->B * d->Hs);
  w.tok_carry = cv.take<int32_t>((size_t)d->B);
  w.stop = cv.take<int32_t>(2 + 64);
  w.bytes = cv.total();
  return w;
}

}  // namespace

// Does the persistent decoder hold this model on chip?  (Otherwise las_api.cu runs the generic tensor-core path: speller_decode_f32 on
// the generic layout.)
bool fast_speller_fits(const las_speller_dims* d) {
  if (d->cell != LAS_CELL_LSTM || d->heads > 1 || d->no_mlp) return false;
  const bool ok = supported(d) == LAS_OK && d->sl * lstm_plan(d, plan_rows(d), false).ncl + 1 <= sm_count();
  return ok;
}

size_t fast_speller_packed_bytes(const las_speller_dims* d) { return pack_layout(d, nullptr).bytes; }
size_t fast_speller_workspace_bytes(const las_speller_dims* d) { return ws_layout(d, nullptr).bytes; }

int fast_speller_pack(const las_speller_weights* w, const las_speller_dims* d, void* packed_fast, bool f16, cudaStream_t st) {
  LAS_TRY(supported(d));
  const SpellerPackFast pk = pack_layout(d, packed_fast);
  const Shape s = shape_of(d);
  for (int l = 0; l < d->sl; ++l) {
    const las_lstm_weights& lw = w->rnn_host[l];
    pack_dec_w_kernel<<<592, 256, 0, st>>>(lw.w_ih, lw.w_hh, pk.w_img[l], l, d->Hs, d->E, d->V, s.nblk, f16);
    LAS_LAUNCH_OK("pack_dec_w_kernel");
    pack_dec_bias_kernel<<<(4 * d->Hs + 255) / 256, 256, 0, st>>>(lw.b_ih, lw.b_hh, pk.bias[l], d->Hs);
    LAS_LAUNCH_OK("pack_dec_bias_kernel");
  }
  LAS_TRY(launch_f32_to_bf16(w->w_phi, pk.w_phi, (size_t)d->D * d->Hs, f16, st));
  LAS_TRY(launch_f32_to_bf16(w->w_cd, pk.w_cd, (size_t)d->V * (d->Hs + d->E), f16, st));
  LAS_TRY(launch_f32_to_bf16(w->w_psi, pk.w_psi, (size_t)d->D * d->E, f16, st));
  return LAS_OK;
}

// One persistent launch: utterances [b0, b0 + Bc) of the batch, global steps [s_begin, s_begin + s_count).
//   first_seg: convert enc, compute psi, build the initial input / state (s_begin == 0);
//   last_seg:  hand the recurrent state back to the caller (io->h_state / c_state / word / context);
// between segments the state lives in the workspace: h / context / dense word in the parity-0 hand-off buffers (s_count is even
// for every segment but the last), c and the fed-back token in the carry buffers.
int fast_speller_decode_segment(const las_decode_io* io, const SpellerF32Inputs& f32, const void* packed_fast, const las_speller_dims* d,
                                int b0, int Bc, int s_begin, int s_count, bool first_seg, bool last_seg, int decode_mode, int relu,
                                void* ws_fast, bool f16, bool beside, cudaStream_t st) {
  const LstmPlan lp = lstm_plan(d, Bc, beside);
  const int n_lstm = d->sl * lp.ncl;
  LAS_REQUIRE(lp.units == 16 || lp.gsz <= 32, "32 hidden units per LSTM CTA need at most 32 rows per iteration (%d utterances in lockstep)", Bc);
  LAS_REQUIRE(last_seg || (s_count % 2 == 0), "decoder segments must have an even number of steps (%d)", s_count);
  LAS_REQUIRE(s_begin % 2 == 0, "decoder segments must start at an even step (%d)", s_begin);
  const SpellerPackFast pk = pack_layout(d, const_cast<void*>(packed_fast));
  const float* psi = io->psi ? io->psi : f32.psi;

  {
    las_speller_dims dc = *d;
    dc.B = Bc;
    const SpellerWsFast w = ws_layout(&dc, ws_fast);
    DecParams p;
    memset(&p, 0, sizeof(p));
    p.B = Bc; p.U = d->U; p.E = d->E; p.Hs = d->Hs; p.sl = d->sl; p.V = d->V; p.D = d->D;
    p.steps = s_count; p.s0 = s_begin; p.decode_mode = decode_mode; p.relu = relu; p.gt_steps = io->gt_steps; p.ncl = lp.ncl;
    const AttPlan ap = att_plan(d, n_lstm);
    p.att_split = ap.split; p.ctx_ntm = ap.ntm; p.ctx_tmem = ap.ntm > 0; p.k_in_smem = ap.k_in_smem; p.wreg = ap.wreg;
    const RingCfg rc = ring_cfg(d, lp.units, lp.gsz);
    LAS_REQUIRE(rc.smem <= 224 * 1024, "LAS_MODE_BF16 speller: %d-unit LSTM CTAs do not fit shared memory (Hs=%d)", lp.units, d->Hs);
    p.groups = lp.groups;
    p.gsz = lp.gsz;
    p.units = lp.units;
    p.nstages = rc.nstages;
    p.stage_bytes = rc.stage_bytes;
    // the LSTM CTAs fetch an activation part as one 3-D copy where its rows are whole 64-column atoms (E == Hs), else atom by atom
    const bool whole_atoms = d->Hs % 64 == 0;
    for (int l = 0; l < d->sl; ++l) {
      p.w_img[l] = pk.w_img[l];
      p.bias[l] = pk.bias[l];
      for (int k = 0; k < 2; ++k) {
        p.hbuf[l][k] = w.hbuf[l][k];
        if (whole_atoms) LAS_TRY(make_tmap_bf16_atoms(&p.tm_h3[l][k], w.hbuf[l][k], Bc, d->Hs / 64, d->Hs, rc.box_rows, d->Hs / 64));
        else LAS_TRY(make_tmap_bf16_box(&p.tm_h[l][k], w.hbuf[l][k], Bc, d->Hs, d->Hs, rc.box_rows));
      }
    }
    for (int k = 0; k < 2; ++k) {
      p.xbuf[k] = w.xbuf[k];
      p.wbuf[k] = w.wbuf[k];
      if (whole_atoms) LAS_TRY(make_tmap_bf16_atoms(&p.tm_x3[k], w.xbuf[k], Bc, d->E / 64, d->E, rc.box_rows, d->E / 64));
      else LAS_TRY(make_tmap_bf16_box(&p.tm_x[k], w.xbuf[k], Bc, d->E, d->E, rc.box_rows));
      LAS_TRY(make_tmap_bf16_box(&p.tm_w[k], w.wbuf[k], Bc, DEC_VP, DEC_VP, rc.box_rows));
    }
    const size_t so = (size_t)b0;  // batch offset into caller tensors
    p.Bfull = d->B;
    p.b0 = b0;
    if (first_seg) { p.c_init = io->c_state; p.c_init_rows = d->B; p.c_init_b0 = b0; }
    else { p.c_init = w.c_carry; p.c_init_rows = Bc; p.c_init_b0 = 0; }
    if (last_seg) { p.c_out = io->c_state; p.c_out_rows = d->B; p.c_out_b0 = b0; p.h_out = io->h_state; }
    else { p.c_out = w.c_carry; p.c_out_rows = Bc; p.c_out_b0 = 0; p.h_out = nullptr; }
    p.tok_init = first_seg ? nullptr : w.tok_carry;
    p.tok_carry = last_seg ? nullptr : w.tok_carry;
    p.stop = (io->early_exit && !first_seg) ? w.stop : nullptr;
    p.enc = w.enc_bf16;
    p.psi = psi;
    p.w_phi = pk.w_phi; p.b_phi = f32.b_phi; p.w_cd = pk.w_cd; p.b_cd = f32.b_cd;
    p.gt_dense = io->gt_dense;
    p.gt_index = io->gt_index;
    p.enc_lengths = io->enc_lengths;
    p.logp = io->logp; p.attn = io->attn; p.tokens = io->tokens;
    p.nll_labels = io->nll_labels; p.nll_terms = io->nll_terms; p.nll_steps = io->nll_steps;
    if (last_seg) { p.word_out = io->word; p.ctx_out = io->context; }
    p.sync = w.sync;
    p.h_ll = w.h_ll;
    p.tok_ll = w.tok_ll;
    p.f16 = f16;
    // the fed-back word is an index (greedy argmax / index teacher forcing) unless a dense vector is asked for
    p.word_gather = io->gt_dense ? 0 : (io->gt_index ? 1 : (decode_mode != LAS_DECODE_RAW ? 1 : 0));
    p.sample_seed = io->sample_seed;
    p.trace = first_seg ? debug_options().trace_at(TRACE_DEC) : nullptr;

    {
      ProfScope ps("speller.prepare", st);
      if (first_seg) LAS_TRY(launch_f32_to_bf16(io->enc + so * d->U * d->E, w.enc_bf16, (size_t)Bc * d->U * d->E, f16, st));
      LAS_CUDA_OK(cudaMemsetAsync(w.flags, 0, w.flag_bytes, st));
      if (first_seg) {
        dec_init_kernel<<<Bc, 256, 0, st>>>(p, io->enc, io->word, io->context, io->h_state);
        LAS_LAUNCH_OK("dec_init_kernel");
      }
    }
    if (!io->psi && first_seg) {
      // psi(enc) once per utterance (model/las_model.py:279 recomputes it every step): the same tcgen05 GEMM as the
      // listener's input projection, bf16 operands (the enc copy made above), fp32 accumulate + bias + relu
      ProfScope pp("speller.psi", st);
      LAS_TRY(launch_gemm_bf16_tc(w.enc_bf16, d->E, pk.w_psi, d->E, f32.b_psi, f32.psi + so * d->U * d->D, d->D, Bc * d->U, d->D, d->E, f16,
                                  st, relu != 0));
    }
    ProfScope ps("speller.steps", st);
    const size_t smem = (rc.smem > ap.smem ? rc.smem : ap.smem) + 1024;
    // the operand format is a template parameter: the conversions sit in the GEMV inner loops (a run-time branch there cost 20 %)
    auto kern = p.f16 ? speller_decode_persistent_kernel<1> : speller_decode_persistent_kernel<0>;
    LAS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_lstm + p.att_split * Bc);
    cfg.blockDim = dim3(DEC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (p.att_split == 2) {  // pairs of consecutive CTAs form clusters (the LSTM CTAs' pairing is not used)
      at[1].id = cudaLaunchAttributeClusterDimension;
      at[1].val.clusterDim.x = 2;
      at[1].val.clusterDim.y = 1;
      at[1].val.clusterDim.z = 1;
      cfg.numAttrs = 2;
    }
    LAS_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p));
    count_launch();
  }
  return LAS_OK;
}

int fast_speller_max_group(const las_speller_dims* d) {
  // utterances per persistent launch: one attention CTA each (two for split attention), and at most 64 (activation slots hold
  // 64 batch rows)
  const int n_lstm = d->sl * lstm_plan(d, plan_rows(d), false).ncl;
  const int n = (sm_count() - n_lstm) / att_plan(d, n_lstm).split;
  return n < 64 ? n : 64;
}

int fast_speller_ctas(const las_speller_dims* d, bool beside) {
  const int n_lstm = d->sl * lstm_plan(d, d->B, beside).ncl;
  return n_lstm + att_plan(d, n_lstm).split * d->B;
}

// Segment lengths: `seg` steps each (even), the remainder in the last one.  seg <= 0: one segment.
static int next_segment(int s_begin, int steps, int seg) {
  if (seg <= 0 || s_begin + seg >= steps) return steps - s_begin;
  return seg;
}

int fast_speller_decode(const las_decode_io* io, const SpellerF32Inputs& f32, const void* packed_fast, const las_speller_dims* d, int steps,
                        int decode_mode, int relu, void* ws_fast, bool f16, cudaStream_t st) {
  LAS_TRY(supported(d));
  const int n_lstm = d->sl * lstm_plan(d, plan_rows(d), false).ncl;
  const int nsm = sm_count();
  LAS_REQUIRE(n_lstm + 1 <= nsm, "LAS_MODE_BF16 speller: %d LSTM CTAs do not fit %d SMs", n_lstm, nsm);
  const int max_b = fast_speller_max_group(d);
  const bool eos = io->early_exit != 0;
  LAS_REQUIRE(!eos || io->tokens, "<eos> early exit needs io->tokens");
  int seg = io->segment_steps > 0 ? (io->segment_steps + 1) & ~1 : 0;
  if (eos && seg == 0) seg = 32;
  if (eos && io->steps_done) LAS_CUDA_OK(cudaMemsetAsync(io->steps_done, 0, sizeof(int32_t), st));
  for (int b0 = 0; b0 < d->B; b0 += max_b) {
    const int Bc = (d->B - b0) < max_b ? (d->B - b0) : max_b;
    las_speller_dims dc = *d;
    dc.B = Bc;
    int32_t* const stop = ws_layout(&dc, ws_fast).stop;  // <eos> bookkeeping of the launch group: stop, group_steps, done[64]
    if (eos) LAS_CUDA_OK(cudaMemsetAsync(stop, 0, sizeof(int32_t) * (2 + 64), st));
    for (int sb = 0; sb < steps;) {
      const int n = next_segment(sb, steps, seg);
      LAS_TRY(fast_speller_decode_segment(io, f32, packed_fast, d, b0, Bc, sb, n, sb == 0, sb + n == steps, decode_mode, relu, ws_fast, f16, false, st));
      if (eos) LAS_TRY(launch_eos_check(io->tokens, d->B, b0, Bc, sb, sb + n, io->eos_token, stop, st));
      sb += n;
    }
    if (eos)
      LAS_TRY(launch_eos_fill(stop, steps, d->B, b0, Bc, d->V, d->U, 1, io->eos_token, io->logp, io->attn, io->tokens, io->nll_terms, io->steps_done, st));
  }
  return LAS_OK;
}

}  // namespace las
