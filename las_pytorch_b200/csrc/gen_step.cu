// Generic tensor-core decoder step, fused (LAS_MODE_BF16 / LAS_MODE_F16 beyond what the persistent decoder keeps on chip: the
// reference's shipped config/librispeech-config.yaml:13-34 with its 1024-wide speller cells, GRU / RNN cells, use_mlp_in_attention
// False).  One decoder step (model/las_model.py:178-238) is `layers` launches of gen_cell_step_kernel + one of attend_cluster_kernel:
//
//   gen_cell_step_kernel   one stacked-cell layer: pre[r, b] = W[r, :] . [x_b | h_prev_b]  (tcgen05, weights streamed from L2 through a
//                          TMA ring, fp32 accumulation in tensor memory) + bias -> cell update in fp32 -> h as fp32 (attention, state
//                          output) AND as 16-bit operand rows of the GEMMs that consume it next (this layer's next step, the next
//                          layer's current step): no pre-activation round trip, no operand-building kernel.
//   attend_cluster_kernel  phi, energies, masked softmax, context, character distribution, feedback for one utterance by a cluster of
//                          up to 8 CTAs: the encoder steps are cut into 8 fixed slices (flash-decoding style partial softmax / partial
//                          context per slice, combined in slice order through distributed shared memory), phi's and the character
//                          MLP's rows are dealt to the CTAs.  The slices, and every summation order, are the same for every cluster
//                          size, so an utterance's result does not depend on the batch it is decoded in.
//
// Launches are chained with programmatic dependent launch: a kernel's prologue, and for the cell kernel the K blocks that multiply the
// layer's OWN previous state (written a whole step earlier), run under the tail of the kernel in front of it.
#include <cuda.h>
#include <string.h>

#include "attend_tail.cuh"
#include "las_fast.cuh"
#include "umma.cuh"

namespace las {

namespace {

__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
// =========================================================================================================
// gen_cell_step_kernel.  CTA c owns 64 / G consecutive cells and all G gate rows of each (LSTM: i,f,g,o; GRU: r,z,n_x,n_h; RNN: 1),
// i.e. 64 rows of the packed [R, Kp] weights (kernels_f32.cu gen_pack_w_kernel; Kp is a multiple of 64).  The weights are the A
// operand (M = 64), the activations [B, Kp] the B operand (N = B rounded up to 16, rows beyond B are TMA zero fill).
//   warp 0 (one thread)  TMA producer.  One ring stage = GS_KBS 64-column K blocks, fetched by TWO copies: a 4-D box {64 k, 64/G
//                        cells, G gates, GS_KBS blocks} of the weights and a 3-D box {64 k, N, GS_KBS} of the activations (per-copy cost
//                        dominates small boxes: one 16-row box per gate and block ran at 0.42 us per block, 5x slower)
//   warp 1 (one thread)  tcgen05.mma issuer; tensor-memory allocation
//   all warps            epilogue: lanes 0-63 -> shared memory (warps 4, 5), then one (utterance, cell) per thread
// Stages [st_first, n_stages) multiply only the layer's own previous state and are issued first, before griddepcontrol.wait.
// =========================================================================================================
constexpr int GS_ROWS = 64, GS_THREADS = 256, GS_WBYTES = GS_ROWS * 128, GS_KBS = 2;

struct GenStepArgs {
  const float* bias;     // [R]
  float* c;              // [B, H] (LSTM)
  const float* h_prev;   // [B, H] row stride h_ld (GRU)
  long long h_ld;
  float* h_out;          // [B, H] row stride hout_ld
  long long hout_ld;
  __nv_bfloat16* o1;     // nullable: operand rows that receive h (this layer's next step), already offset to the h columns
  long long o1_ld;
  __nv_bfloat16* o2;     // nullable: the next layer's x columns
  long long o2_ld;
  int B, H, G, cell, Kp, NB, stages, f16, st_first;
  int early;         // trigger the dependent launch at once (last layer: the attention kernel's prologue reads only constants)
  int region;        // activations in their own region (two copies per launch) instead of riding in the ring stages
  long long* trace;  // nullable (tools/gen_step_probe.py): clock64 stamps of CTA 0
};

__global__ void __launch_bounds__(GS_THREADS, 1)
gen_cell_step_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_ai,
                     const __grid_constant__ CUtensorMap tm_ad, const GenStepArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* const ring = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int a_bytes = p.NB * 128;                          // one K block of the activations
  // ring stage: [w block 0][w block 1] and, unless the activations have their own region, [a block 0][a block 1]
  const int stage_bytes = p.region ? GS_KBS * GS_WBYTES : GS_KBS * (GS_WBYTES + a_bytes);
  const int k_blocks = p.Kp / 64, n_stages = (k_blocks + GS_KBS - 1) / GS_KBS;
  uint8_t* const acts = ring + (size_t)p.stages * stage_bytes;
  uint64_t* const full = reinterpret_cast<uint64_t*>(acts + (p.region ? (size_t)n_stages * GS_KBS * a_bytes : 0));
  uint64_t* const empty = full + p.stages;
  uint64_t* const done = empty + p.stages;
  uint64_t* const afull = done + 1;  // [2]: independent / dependent activations (region form)
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(afull + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long* const tr = (p.trace && blockIdx.x == 0) ? p.trace : nullptr;
  if (tr && tid == 0) { tr[0] = clock64(); tr[9] = gtime(); }
  if (p.early) griddep_launch();
  const int cells = GS_ROWS / p.G, cell0 = blockIdx.x * cells;
  uint32_t ncols = 32;
  while ((int)ncols < p.NB) ncols <<= 1;

  if (tid == 0) {
    ptx::prefetch_tensormap(&tm_w);
    ptx::prefetch_tensormap(p.region ? &tm_ai : &tm_a);
    if (p.region) ptx::prefetch_tensormap(&tm_ad);
    ptx::mbar_init(&afull[0], 1);
    ptx::mbar_init(&afull[1], 1);
    for (int i = 0; i < p.stages; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    ptx::mbar_init(done, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc(tmem_slot, ncols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (tr && tid == 0) tr[1] = clock64();

  // Operands of this thread's first (utterance, cell) of the epilogue: the cell state / previous h were written a whole step ago and
  // the biases never change, so their loads are issued here, long before the accumulators are ready.
  const int H = p.H;
  const int b_first = tid / cells, j_first = tid % cells;
  const bool first_ok = tid < p.B * cells && cell0 + j_first < H;
  float bias_r[4] = {0.f, 0.f, 0.f, 0.f}, c_first = 0.f, hp_first = 0.f;
  if (first_ok) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
      if (g < p.G) bias_r[g] = p.bias[g * H + cell0 + j_first];
    if (p.cell == LAS_CELL_LSTM) c_first = p.c[(size_t)b_first * H + cell0 + j_first];
    if (p.cell == LAS_CELL_GRU && p.h_prev) hp_first = p.h_prev[(long long)b_first * p.h_ld + cell0 + j_first];
  }

  // Both role threads run ALONE on their warps, so every instruction they execute costs its full latency: the loops below keep shared
  // memory addresses as 32-bit values, advance them by constants and avoid divisions (with generic pointers, i % stages and a
  // descriptor built per instruction one producer iteration took 0.35 us and one MMA 57 cycles of issue time).
  const int n_indep = n_stages - p.st_first;
  const uint32_t ring_a = ptx::smem_u32(ring), full_a = ptx::smem_u32(full), empty_a = ptx::smem_u32(empty);
  const uint32_t stage_b = (uint32_t)stage_bytes, ring_end = ring_a + (uint32_t)p.stages * stage_b;
  // (The role warps stay converged and issue through elect_one(): under `if (lane == 0)` the compiler wraps every TMA / MMA
  // instruction in an elect-and-branch loop -- 93 cycles per MMA instead of ~40.)
  if (warp == 0) {
    const uint64_t tw = reinterpret_cast<uint64_t>(&tm_w), ta = reinterpret_cast<uint64_t>(&tm_a);
    uint32_t dst = ring_a, boff = 0, par = 1;  // slot address, barrier offset, parity of the `empty` wait
    auto advance = [&]() {
      dst += stage_b;
      boff += 8;
      if (dst == ring_end) { dst = ring_a; boff = 0; par ^= 1; }
    };
    auto wait_empty = [&]() {
      uint32_t ok;
      do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(empty_a + boff), "r"(par) : "memory");
      } while (!ok);
    };
    // one stage: arm its barrier, weights, and (ring form, when `with_acts`) its activation blocks
    auto load_stage = [&](int kb, bool with_acts) {
      if (ptx::elect_one()) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full_a + boff), "r"(stage_b) : "memory");
        asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                     ::"r"(dst), "l"(tw), "r"(full_a + boff), "r"(0), "r"(cell0), "r"(0), "r"(kb) : "memory");
        if (with_acts)
          asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                       ::"r"(dst + GS_KBS * GS_WBYTES), "l"(ta), "r"(full_a + boff), "r"(0), "r"(0), "r"(kb) : "memory");
      }
    };
    // Region form: ALL activation blocks of a part in one copy (a small copy completes ~0.35 us after the one in front of it).
    auto load_region = [&](const CUtensorMap* tm, int part, int blk0, int nblk) {
      if (ptx::elect_one()) {
        const uint32_t bar = ptx::smem_u32(&afull[part]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(nblk * a_bytes)) : "memory");
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                     ::"r"(ptx::smem_u32(acts) + (uint32_t)(blk0 * a_bytes)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(0), "r"(0), "r"(blk0)
                     : "memory");
      }
    };
    // 1. the independent stages (K blocks that multiply the layer's own previous state)
    int kb = GS_KBS * p.st_first;
    if (p.region && n_indep > 0) load_region(&tm_ai, 0, kb, GS_KBS * n_indep);
    for (int i = 0; i < n_indep; ++i, kb += GS_KBS) {
      wait_empty();
      load_stage(kb, !p.region);
      advance();
    }
    // 2. the WEIGHTS of the dependent stages do not depend on the previous launch either.  The first `stages` of them go into slots
    // whose previous occupant is an independent stage (consumed without the dependency), so waiting for those slots is safe.
    const uint32_t dst0 = dst, boff0 = boff;
    int j = 0;
    kb = 0;
    for (; j < p.st_first && j < p.stages; ++j, kb += GS_KBS) {
      wait_empty();
      load_stage(kb, false);
      advance();
    }
    if (tr && lane == 0) tr[2] = clock64();
    griddep_wait();
    griddep_launch();
    if (tr && lane == 0) { tr[3] = clock64(); tr[10] = gtime(); }
    // 3. their activations, then the remaining stages whole
    if (p.region) {
      if (p.st_first > 0) load_region(&tm_ad, 1, 0, GS_KBS * p.st_first);
    } else {
      uint32_t d = dst0, bo = boff0;
      for (int k = 0, kk = 0; k < j; ++k, kk += GS_KBS) {
        if (ptx::elect_one())
          asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                       ::"r"(d + GS_KBS * GS_WBYTES), "l"(ta), "r"(full_a + bo), "r"(0), "r"(0), "r"(kk) : "memory");
        d += stage_b;
        bo += 8;
        if (d == ring_end) { d = ring_a; bo = 0; }
      }
    }
    for (; j < p.st_first; ++j, kb += GS_KBS) {
      wait_empty();
      load_stage(kb, !p.region);
      advance();
    }
  } else if (warp == 1) {
    const UmmaLayout lw{1, 0, 1024, 0};
    const uint32_t idesc = umma_idesc_bf16(64, (uint32_t)p.NB, p.f16);
    const uint64_t wdesc0 = umma_smem_desc(lw, ring_a, 0),
                   adesc0 = umma_smem_desc(lw, p.region ? ptx::smem_u32(acts) : ring_a + GS_KBS * GS_WBYTES, 0);
    const uint32_t a16 = (uint32_t)a_bytes >> 4, stage16 = stage_b >> 4, end16 = ((uint32_t)p.stages * stage_b) >> 4;
    uint32_t off16 = 0, boff = 0, par = 0, accum = 0;
    int kb = GS_KBS * p.st_first;
    for (int i = 0; i < n_stages; ++i) {
      if (i == n_indep) kb = 0;
      if (p.region && (i == 0 || i == n_indep)) ptx::mbar_wait(&afull[i == n_indep ? 1 : 0], 0);
      uint32_t ok;
      do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(full_a + boff), "r"(par) : "memory");
      } while (!ok);
      ptx::tc_fence_after();
      if (tr && lane == 0 && i == n_indep) tr[7] = clock64();
      if (ptx::elect_one()) {
        uint64_t wd = wdesc0 + off16, ad = p.region ? adesc0 + (uint32_t)kb * a16 : adesc0 + off16;
#pragma unroll
        for (int jb = 0; jb < GS_KBS; ++jb) {
          if (kb + jb < k_blocks) {  // (a block beyond Kp is zero fill)
#pragma unroll
            for (int k = 0; k < 4; ++k) ptx::umma_bf16(tmem, wd + 2 * k, ad + 2 * k, idesc, (accum | jb | k) != 0);
          }
          wd += GS_WBYTES >> 4;
          ad += a16;
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty_a + boff) : "memory");
      }
      accum = 1;
      kb += GS_KBS;
      off16 += stage16;
      boff += 8;
      if (off16 == end16) { off16 = 0; boff = 0; par ^= 1; }
    }
    if (tr && lane == 0) tr[8] = clock64();
    if (ptx::elect_one()) ptx::umma_commit(done);
    ptx::mbar_wait(done, 0);
  }
  __syncthreads();  // (the other warps sleep here instead of polling the barrier)
  ptx::tc_fence_after();
  if (tr && tid == 64) tr[4] = clock64();
  griddep_wait();  // (already satisfied: the dependent stages were loaded after the producer's wait)

  // accumulator rows 0-63 -> shared memory (the ring is dead: every copy has landed and every MMA has read its operands).  M = 64:
  // row i sits in tensor-memory lane (i / 16) * 32 + i % 16, so warps 4-7 each read their lane quadrant and keep lanes 0-15.
  float* const pre = reinterpret_cast<float*>(ring);
  const int ldp = p.NB + 1;
  if (warp >= 4) {
    const int row = (warp - 4) * 16 + lane;
    for (int c0 = 0; c0 < p.NB; c0 += 16) {
      uint32_t v[16];
      ptx::tmem_ld_32x32b_x16(tmem + ((uint32_t)((warp - 4) * 32) << 16) + (uint32_t)c0, v);
      ptx::tmem_ld_wait();
      if (lane < 16) {
#pragma unroll
        for (int j = 0; j < 16; ++j) pre[row * ldp + c0 + j] = __uint_as_float(v[j]);
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (tr && tid == 64) tr[5] = clock64();

  for (int i = tid; i < p.B * cells; i += GS_THREADS) {
    const int b = i / cells, j = i % cells, cell = cell0 + j;
    if (cell >= H) continue;
    const bool pre_loaded = i == tid;  // (first item: operands already in registers)
    auto P = [&](int g) { return pre[(g * cells + j) * ldp + b] + (pre_loaded ? bias_r[g] : p.bias[g * H + cell]); };
    float h;
    if (p.cell == LAS_CELL_LSTM) {
      const float ig = sigmoid_precise(P(0)), fg = sigmoid_precise(P(1)), gg = tanhf(P(2)), og = sigmoid_precise(P(3));
      const float cn = fg * (pre_loaded ? c_first : p.c[(size_t)b * H + cell]) + ig * gg;
      p.c[(size_t)b * H + cell] = cn;
      h = og * tanhf(cn);
    } else if (p.cell == LAS_CELL_GRU) {
      const float hp = pre_loaded ? hp_first : (p.h_prev ? p.h_prev[(long long)b * p.h_ld + cell] : 0.f);
      const float rg = sigmoid_precise(P(0)), zg = sigmoid_precise(P(1));
      const float ng = tanhf(P(2) + rg * P(3));
      h = (1.0f - zg) * ng + zg * hp;
    } else {
      h = tanhf(P(0));
    }
    p.h_out[(long long)b * p.hout_ld + cell] = h;
    const __nv_bfloat16 ho = op_from_f32(h, p.f16);
    if (p.o1) p.o1[(long long)b * p.o1_ld + cell] = ho;
    if (p.o2) p.o2[(long long)b * p.o2_ld + cell] = ho;
  }
  __syncthreads();
  if (tr && tid == 64) { tr[6] = clock64(); tr[11] = gtime(); }
  if (warp == 1) ptx::tmem_dealloc(tmem, ncols);
}

// =========================================================================================================
// attend_cluster_kernel (heads == 1, E % 4 == 0).  Cluster of C in {1,2,4,8} CTAs per utterance, rank r:
//   q        rows [r*D/C ..) of phi, stored into every peer's shared memory                                 -- cluster barrier 1
//   slices   encoder steps in AC_SLICES fixed slices; rank r owns slices [r*8/C, (r+1)*8/C): energies, slice maximum m_i,
//            p = exp(e - m_i), slice sum s_i, partial context part_i[E] = sum_u p[u] enc[b,u,:]; {part_i, m_i, s_i} go to every peer
//            as ONE bulk copy per peer, completing on the peer's mbarrier (pulling them with ld.shared::cluster took 4 us)
//   combine  M = max m_i, w_i = exp(m_i - M), S = sum s_i w_i (slice order), context = (sum_i w_i part_i) / S in every CTA (each
//            needs the whole context for its rows of the character MLP); scores of the own slices
//   logits   rows v = r, r+C, .. of the character MLP as four K segments each, summed in segment order, sent to rank 0  -- barrier 2
//   rank 0   log-softmax, NLL term, token, fed-back word (attend_tail)
// Dot products read 16-byte vectors with four of them in flight per lane where the row is aligned for it.
// =========================================================================================================
constexpr int AC_SLICES = 8, AC_SEGS = 4;

// lanes of one warp: sum_k w[k] * x[k] over [0, n), x in shared memory; vec: n % 4 == 0 and both 16-byte aligned
// (One out-of-line copy each: the kernel runs once per launch, so its code size is paid in instruction fetches every decoder step.
// Generic loads: the row may be in global or in shared memory.)
__device__ __noinline__ float warp_dot(const float* w, const float* x, int n, int lane, bool vec) {
  float acc = 0.f;
  if (vec) {
    const float4* w4 = reinterpret_cast<const float4*>(w);
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const int n4 = n >> 2;
    int i = lane;
    for (; i + 96 < n4; i += 128) {
      const float4 a0 = w4[i], a1 = w4[i + 32], a2 = w4[i + 64], a3 = w4[i + 96];
      const float4 b0 = x4[i], b1 = x4[i + 32], b2 = x4[i + 64], b3 = x4[i + 96];
      acc = fmaf(a0.x, b0.x, acc); acc = fmaf(a0.y, b0.y, acc); acc = fmaf(a0.z, b0.z, acc); acc = fmaf(a0.w, b0.w, acc);
      acc = fmaf(a1.x, b1.x, acc); acc = fmaf(a1.y, b1.y, acc); acc = fmaf(a1.z, b1.z, acc); acc = fmaf(a1.w, b1.w, acc);
      acc = fmaf(a2.x, b2.x, acc); acc = fmaf(a2.y, b2.y, acc); acc = fmaf(a2.z, b2.z, acc); acc = fmaf(a2.w, b2.w, acc);
      acc = fmaf(a3.x, b3.x, acc); acc = fmaf(a3.y, b3.y, acc); acc = fmaf(a3.z, b3.z, acc); acc = fmaf(a3.w, b3.w, acc);
    }
    for (; i < n4; i += 32) {
      const float4 a0 = w4[i];
      const float4 b0 = x4[i];
      acc = fmaf(a0.x, b0.x, acc); acc = fmaf(a0.y, b0.y, acc); acc = fmaf(a0.z, b0.z, acc); acc = fmaf(a0.w, b0.w, acc);
    }
  } else {
#pragma unroll 1
    for (int k = lane; k < n; k += 32) acc = fmaf(w[k], x[k], acc);
  }
  return warp_sum(acc);
}
__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// kShared: several decoder rows per utterance (a.rows_per_utt > 1, beam search); the one-row form keeps the division out of the prologue
template <bool kShared>
__global__ void __launch_bounds__(AC_THREADS, 1) attend_cluster_kernel(const AttendArgs a, const int C) {
  extern __shared__ __align__(16) float sm[];
  const int nown = AC_SLICES / C;
  const int EP = a.E + 4;                               // one slice's record: part[E], m, s, 2 pad
  const int Hs4 = (a.Hs + 3) & ~3, D4 = (a.D + 3) & ~3, U4 = (a.U + 3) & ~3, V4 = (a.V + 3) & ~3;
  float* s_state = sm;                                  // Hs | E contiguous (Hs % 4 == 0): the character MLP's input vector
  float* s_ctx = s_state + ((a.Hs & 3) ? Hs4 : a.Hs);
  float* s_q = s_ctx + a.E;                             // D
  float* s_p = s_q + D4;                                // U (own slices only)
  float* s_w = s_p + U4;                                // AC_SLICES weights, 1/S
  float* s_logit = s_w + 12;                            // V (rank 0 collects)
  float* s_lpart = s_logit + V4;                        // rows per CTA * AC_SEGS
  float* s_red = s_lpart + (((a.V + C - 1) / C) * AC_SEGS + 3 & ~3);  // 32
  float* s_bias = s_red + 32;                           // D4 + V4: b_phi, b_cd (fetched before the dependency resolves)
  float* s_all = s_bias + D4 + V4;                      // AC_SLICES * EP: every slice's record (own ones computed here)
  uint64_t* xbar = reinterpret_cast<uint64_t*>(s_all + AC_SLICES * EP);
  const int ngroups = (a.E * 2 <= 4 * AC_THREADS) ? ((a.E * 4 <= 4 * AC_THREADS) ? 4 : 2) : 1;  // row groups of the context loop
  const int dq = (a.D + C - 1) / C, KC = a.Hs + a.E;
  const int us = (a.U + AC_SLICES - 1) / AC_SLICES;
  float* s_tmp = reinterpret_cast<float*>(xbar + 2);    // (ngroups - 1) * E: the other row groups' sums of the slice being reduced
  const int r = (C > 1) ? (int)ptx::cluster_ctarank() : 0;
  const int b = blockIdx.x / C;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = AC_THREADS >> 5;
  const uint32_t rec_bytes = (uint32_t)(nown * EP * 4);

  long long* const tr = (a.trace && blockIdx.x == 0 && tid == 0) ? a.trace : nullptr;
  if (tr) tr[0] = clock64();
  if (tid == 0 && C > 1) {
    ptx::mbar_init(xbar, 1);
    ptx::fence_mbar_init();
    ptx::mbar_arrive_expect_tx(xbar, (uint32_t)(C - 1) * rec_bytes);
  }
  // (biases and the utterance's length do not depend on the launch in front of this one)
  const int u_begin = min(a.U, r * nown * us), u_end = min(a.U, (r + 1) * nown * us);
  const int bu = kShared ? b / a.rows_per_utt : b;  // the utterance whose encoder features row b attends over
  const float* psib = a.psi + (size_t)bu * a.U * a.D;
  const float* encb = a.enc + (size_t)bu * a.U * a.E;
  {
    if (a.w_phi) for (int d = tid; d < a.D; d += AC_THREADS) s_bias[d] = a.b_phi[d];
    if (a.w_cd) for (int v = tid; v < a.V; v += AC_THREADS) s_bias[D4 + v] = a.b_cd[v];
  }
  const int ulen = a.enc_lengths ? min(max(a.enc_lengths[bu], 1), a.U) : a.U;
  griddep_wait();
  griddep_launch();
  if (tr) { tr[1] = clock64(); tr[10] = gtime(); }

  for (int k = tid; k < a.Hs; k += AC_THREADS) s_state[k] = a.state[(size_t)b * a.state_ld + k];
  __syncthreads();

  // ---- q = act(W_phi . state + b_phi)   (model/las_model.py:278; :283-285 without the MLP)
  if (!a.w_phi) {
    for (int d = tid; d < a.D; d += AC_THREADS) s_q[d] = s_state[d];
  } else {
    const int d_end = min(a.D, (r + 1) * dq);
    const bool vec = (a.Hs & 3) == 0 && aligned16(a.w_phi);
    for (int d = r * dq + wid; d < d_end; d += nw) {
      float acc = warp_dot(a.w_phi + (size_t)d * a.Hs, s_state, a.Hs, lane, vec) + s_bias[d];
      if (a.relu) acc = fmaxf(acc, 0.f);
      if (C == 1) {
        if (lane == 0) s_q[d] = acc;
      } else if (lane < C) {
        st_cluster_f32(ptx::mapa(ptx::smem_u32(&s_q[d]), (uint32_t)lane), acc);
      }
    }
  }
  if (C > 1) ptx::cluster_sync(); else __syncthreads();
  if (tr) tr[2] = clock64();

  // ---- energies of the own slices   (:289-291): eight lanes per encoder step where D allows, else a warp
  if ((a.D & 31) == 0 && a.D <= 256 && aligned16(psib)) {
    const int sub = lane >> 3, l8 = lane & 7, nv = a.D >> 5;  // float4 per lane
    const float4* q4 = reinterpret_cast<const float4*>(s_q);
    for (int u0 = u_begin + wid * 4; u0 < u_end; u0 += nw * 4) {
      const int u = u0 + sub;
      float acc = 0.f;
      if (u < u_end) {
        const float4* p4 = reinterpret_cast<const float4*>(psib + (size_t)u * a.D);
        for (int j = 0; j < nv; ++j) {
          const float4 x = p4[l8 + 8 * j], qq = q4[l8 + 8 * j];
          acc = fmaf(qq.x, x.x, acc); acc = fmaf(qq.y, x.y, acc); acc = fmaf(qq.z, x.z, acc); acc = fmaf(qq.w, x.w, acc);
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      if (l8 == 0 && u < u_end) s_p[u] = (u < ulen) ? acc : -INFINITY;
    }
  } else {
    for (int u = u_begin + wid; u < u_end; u += nw) {
      const float acc = warp_dot(psib + (size_t)u * a.D, s_q, a.D, lane, false);
      if (lane == 0) s_p[u] = (u < ulen) ? acc : -INFINITY;
    }
  }
  __syncthreads();
  // slice maximum, exponentials, slice sum: one warp per own slice
  for (int li = wid; li < nown; li += nw) {
    const int i = r * nown + li;
    const int s0 = min(a.U, i * us), s1 = min(a.U, (i + 1) * us);
    float m = -INFINITY;
    for (int u = s0 + lane; u < s1; u += 32) m = fmaxf(m, s_p[u]);
    m = warp_max(m);
    float sum = 0.f;
    for (int u = s0 + lane; u < s1; u += 32) {
      const float e = (m == -INFINITY) ? 0.f : expf(s_p[u] - m);
      s_p[u] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    if (lane == 0) {
      s_all[i * EP + a.E] = m;
      s_all[i * EP + a.E + 1] = sum;
    }
  }
  __syncthreads();
  if (tr) tr[3] = clock64();
  // ---- partial contexts of the own slices   (:293-297).  Four features per thread; the threads form `ngroups` row groups (a function of
  // E only) that take the slice's encoder steps round robin, each ascending; the groups' sums are added in group order.
  {
    const int cols4 = a.E >> 2, grp = tid / cols4, e = 4 * (tid % cols4);
    for (int li = 0; li < nown; ++li) {
      const int i = r * nown + li;
      const int s0 = min(a.U, i * us), s1 = min(a.U, (i + 1) * us);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      if (grp < ngroups) {
        int u = s0 + grp;
#pragma unroll 1
        for (; u < s1; u += 8 * ngroups) {  // eight encoder steps in flight
          float4 x[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (u + j * ngroups < s1) x[j] = __ldg(reinterpret_cast<const float4*>(encb + (size_t)(u + j * ngroups) * a.E + e));
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (u + j * ngroups < s1) {
              const float pj = s_p[u + j * ngroups];
              acc.x = fmaf(pj, x[j].x, acc.x); acc.y = fmaf(pj, x[j].y, acc.y); acc.z = fmaf(pj, x[j].z, acc.z); acc.w = fmaf(pj, x[j].w, acc.w);
            }
          }
        }
        if (grp > 0) *reinterpret_cast<float4*>(&s_tmp[(grp - 1) * a.E + e]) = acc;
      }
      if (ngroups > 1) __syncthreads();
      if (grp == 0) {
        for (int g = 1; g < ngroups; ++g) {
          const float4 o = *reinterpret_cast<const float4*>(&s_tmp[(g - 1) * a.E + e]);
          acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        *reinterpret_cast<float4*>(&s_all[i * EP + e]) = acc;
      }
      if (ngroups > 1 && li + 1 < nown) __syncthreads();
    }
  }
  if (tr) tr[4] = clock64();
  // ---- own records to every peer: one bulk copy each, then wait for the peers' records
  if (C > 1) {
    ptx::fence_proxy_async_smem();
    __syncthreads();
    if (tid < C && tid != r) {
      const uint32_t src = ptx::smem_u32(&s_all[r * nown * EP]);
      ptx::bulk_copy_to_cluster(ptx::mapa(src, (uint32_t)tid), src, rec_bytes, ptx::mapa(ptx::smem_u32(xbar), (uint32_t)tid));
    }
    ptx::mbar_wait_cluster(xbar, 0);
  } else {
    __syncthreads();
  }
  if (tr) tr[5] = clock64();

  // ---- combine   (softmax :292 over all slices)
  if (tid < 32) {
    float M = -INFINITY;
    for (int i = 0; i < AC_SLICES; ++i) M = fmaxf(M, s_all[i * EP + a.E]);
    float S = 0.f;
    for (int i = 0; i < AC_SLICES; ++i) {
      const float mi = s_all[i * EP + a.E];
      const float w = (mi == -INFINITY) ? 0.f : expf(mi - M);
      if (tid == 0) s_w[i] = w;
      S = fmaf(s_all[i * EP + a.E + 1], w, S);
    }
    if (tid == 0) s_w[AC_SLICES] = 1.0f / S;
  }
  __syncthreads();
  const float inv = s_w[AC_SLICES];
  for (int e = 4 * tid; e < a.E; e += 4 * AC_THREADS) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < AC_SLICES; ++i) {
      const float4 x = *reinterpret_cast<const float4*>(&s_all[i * EP + e]);
      const float w = s_w[i];
      acc.x = fmaf(w, x.x, acc.x); acc.y = fmaf(w, x.y, acc.y); acc.z = fmaf(w, x.z, acc.z); acc.w = fmaf(w, x.w, acc.w);
    }
    acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    *reinterpret_cast<float4*>(&s_ctx[e]) = acc;
    if (r == 0) {
      float* co = a.ctx_out + (size_t)b * a.ctx_ld + e;
      co[0] = acc.x; co[1] = acc.y; co[2] = acc.z; co[3] = acc.w;
      if (a.op_out) {
        __nv_bfloat16* oo = a.op_out + (size_t)b * a.op_ld + a.V + e;
        oo[0] = op_from_f32(acc.x, a.op_f16); oo[1] = op_from_f32(acc.y, a.op_f16);
        oo[2] = op_from_f32(acc.z, a.op_f16); oo[3] = op_from_f32(acc.w, a.op_f16);
      }
    }
  }
  if (a.score_out) {
    for (int u = u_begin + tid; u < u_end; u += AC_THREADS) a.score_out[(size_t)b * a.U + u] = s_p[u] * s_w[u / us] * inv;
  }
  __syncthreads();
  if (tr) tr[6] = clock64();
  if (!a.w_cd) {
    if (C > 1) ptx::cluster_sync();  // nobody leaves while a copy out of its shared memory may still be in flight
    return;
  }

  // ---- logits = W_cd . [state || context] + b_cd   (:181): rows r, r+C, ..; AC_SEGS K segments per row
  const int rows_own = (a.V > r) ? (a.V - r + C - 1) / C : 0;
  const int seg_len = (((KC + AC_SEGS - 1) / AC_SEGS) + 3) & ~3;
  const bool vec_cd = (a.Hs & 3) == 0 && (KC & 3) == 0 && aligned16(a.w_cd);
  for (int item = wid; item < rows_own * AC_SEGS; item += nw) {
    const int lr = item / AC_SEGS, sg = item % AC_SEGS, v = r + lr * C;
    const int k0 = min(KC, sg * seg_len), k1 = min(KC, k0 + seg_len);
    float acc;
    if ((a.Hs & 3) == 0) {
      acc = warp_dot(a.w_cd + (size_t)v * KC + k0, s_state + k0, k1 - k0, lane, vec_cd);
    } else {  // state and context are not contiguous in shared memory
      const float* wr = a.w_cd + (size_t)v * KC;
      acc = 0.f;
      for (int k = k0 + lane; k < k1; k += 32) acc = fmaf(wr[k], k < a.Hs ? s_state[k] : s_ctx[k - a.Hs], acc);
      acc = warp_sum(acc);
    }
    if (lane == 0) s_lpart[item] = acc;
  }
  __syncthreads();
  for (int lr = tid; lr < rows_own; lr += AC_THREADS) {
    const int v = r + lr * C;
    float acc = s_bias[D4 + v];
    for (int sg = 0; sg < AC_SEGS; ++sg) acc += s_lpart[lr * AC_SEGS + sg];
    if (C == 1) s_logit[v] = acc;
    else st_cluster_f32(ptx::mapa(ptx::smem_u32(&s_logit[v]), 0u), acc);
  }
  if (tr) tr[7] = clock64();
  if (C > 1) ptx::cluster_sync(); else __syncthreads();
  if (r != 0) return;
  if (tr) tr[8] = clock64();
  attend_tail(a, b, s_logit, s_red);
  if (tr) { tr[9] = clock64(); tr[11] = gtime(); }
}

}  // namespace

// Activations in their own shared-memory region (one copy per part and launch) while all K blocks of them fit 72 KB
static bool gen_region(int nb, int Kp) { return (size_t)((Kp / 64 + GS_KBS - 1) / GS_KBS) * GS_KBS * nb * 128 <= 72 * 1024; }

int gen_step_make_maps(GenStepMaps* m, const __nv_bfloat16* w, const __nv_bfloat16* act0, const __nv_bfloat16* act1, int H, int G, int B, int Kxp,
                       int Kp) {
  const int nb = (B + 15) & ~15;
  LAS_REQUIRE(nb <= 256 && Kp % 64 == 0, "fused generic decoder step: at most 256 utterances per launch, K a multiple of 64 (B=%d K=%d)", B, Kp);
  const int cells = GS_ROWS / G;
  const int n_stages = (Kp / 64 + GS_KBS - 1) / GS_KBS, first = (Kxp + 64 * GS_KBS - 1) / (64 * GS_KBS);
  const int st_first = first < n_stages ? first : n_stages;
  {  // weights [G*H, Kp] as {64 k, H cells, G gates, Kp/64 blocks}
    const unsigned long long dims[4] = {64, (unsigned long long)H, (unsigned long long)G, (unsigned long long)(Kp / 64)};
    const unsigned long long strides[3] = {(unsigned long long)Kp * 2, (unsigned long long)H * Kp * 2, 128};
    const unsigned box[4] = {64, (unsigned)cells, (unsigned)G, (unsigned)GS_KBS};
    LAS_TRY(make_tmap_bf16_nd(&m->w, w, 4, dims, strides, box));
  }
  for (int q = 0; q < 2; ++q) {  // activations [B, Kp] as {64 k, B, Kp/64 blocks}: per-stage box, and one box per part (region form)
    const unsigned long long dims[3] = {64, (unsigned long long)B, (unsigned long long)(Kp / 64)};
    const unsigned long long strides[2] = {(unsigned long long)Kp * 2, 128};
    const unsigned box[3] = {64, (unsigned)nb, (unsigned)GS_KBS};
    LAS_TRY(make_tmap_bf16_nd(&m->a[q], q ? act1 : act0, 3, dims, strides, box));
    const int nd = GS_KBS * st_first, ni = GS_KBS * (n_stages - st_first);
    const bool region = gen_region(nb, Kp);
    const unsigned box_d[3] = {64, (unsigned)nb, (unsigned)((region && nd > 0) ? nd : 1)};
    const unsigned box_i[3] = {64, (unsigned)nb, (unsigned)((region && ni > 0) ? ni : 1)};
    LAS_TRY(make_tmap_bf16_nd(&m->a_dep[q], q ? act1 : act0, 3, dims, strides, box_d));
    LAS_TRY(make_tmap_bf16_nd(&m->a_ind[q], q ? act1 : act0, 3, dims, strides, box_i));
  }
  return LAS_OK;
}

int launch_gen_cell_step(const GenStepMaps& m, int parity, const float* bias, float* c, const float* h_prev, long long h_ld, float* h_out,
                         long long hout_ld, __nv_bfloat16* o1, long long o1_ld, __nv_bfloat16* o2, long long o2_ld, int B, int H, int cell,
                         int Kxp, int Kp, bool pdl, bool f16, cudaStream_t st, int trace_slot) {
  GenStepArgs p;
  memset(&p, 0, sizeof(p));
  p.bias = bias; p.c = c; p.h_prev = h_prev; p.h_ld = h_ld; p.h_out = h_out; p.hout_ld = hout_ld;
  p.o1 = o1; p.o1_ld = o1_ld; p.o2 = o2; p.o2_ld = o2_ld;
  p.B = B; p.H = H; p.G = (cell == LAS_CELL_RNN) ? 1 : 4; p.cell = cell; p.Kp = Kp;
  p.NB = (B + 15) & ~15;
  p.region = gen_region(p.NB, Kp) ? 1 : 0;
  const size_t region_bytes = p.region ? (size_t)((Kp / 64 + GS_KBS - 1) / GS_KBS) * GS_KBS * p.NB * 128 : 0;
  p.stages = (int)((200 * 1024 - region_bytes) / (GS_KBS * (GS_WBYTES + (p.region ? 0 : p.NB * 128))));  // ring + region <= 200 KB
  if (p.stages > 10) p.stages = 10;
  p.f16 = f16;
  p.early = (o2 == nullptr) ? 1 : 0;
  const int n_stages = (Kp / 64 + GS_KBS - 1) / GS_KBS, first = (Kxp + 64 * GS_KBS - 1) / (64 * GS_KBS);
  p.st_first = first < n_stages ? first : n_stages;
  p.trace = debug_options().trace_at(TRACE_GEN + TRACE_GEN_SLOT * (1 + trace_slot));
  const int cells = GS_ROWS / p.G;
  const size_t smem = 1024 + (size_t)p.stages * GS_KBS * (GS_WBYTES + (p.region ? 0 : p.NB * 128)) + region_bytes + 8 * (2 * p.stages + 3) + 16;
  LAS_CUDA_OK(cudaFuncSetAttribute(gen_cell_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)((H + cells - 1) / cells));
  cfg.blockDim = dim3(GS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  LAS_CUDA_OK(cudaLaunchKernelEx(&cfg, gen_cell_step_kernel, m.w, m.a[parity & 1], m.a_ind[parity & 1], m.a_dep[parity & 1], p));
  LAS_LAUNCH_OK("gen_cell_step_kernel");
  return LAS_OK;
}

int launch_attend_cluster(const AttendArgs& a, int C, bool pdl, cudaStream_t st) {
  LAS_REQUIRE(a.heads == 1 && a.E % 4 == 0 && a.E <= 4 * AC_THREADS && (reinterpret_cast<uintptr_t>(a.enc) & 15) == 0 && (C == 1 || C == 2 || C == 4 || C == 8),
              "attend_cluster_kernel: heads == 1, E %% 4 == 0, E <= %d, aligned enc, C = 1 / 2 / 4 / 8 (heads=%d E=%d C=%d)", 4 * AC_THREADS, a.heads, a.E, C);
  auto r4 = [](size_t n) { return (n + 3) & ~(size_t)3; };
  size_t floats = r4(a.Hs) + a.E + r4(a.D) + r4(a.U) + 12 + r4(a.V) + r4((size_t)((a.V + C - 1) / C) * AC_SEGS) + 32 + r4(a.D) + r4(a.V) +
                  (size_t)AC_SLICES * (a.E + 4) + 4 /* barrier */ + (size_t)3 * a.E /* row-group sums */;
  const size_t smem = sizeof(float) * floats + 16;
  LAS_REQUIRE(smem <= 200 * 1024, "attention step needs %zu bytes of shared memory (U=%d E=%d)", smem, a.U, a.E);
  const bool shared = a.rows_per_utt > 1;
  LAS_CUDA_OK(cudaFuncSetAttribute(shared ? attend_cluster_kernel<true> : attend_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(a.B * C));
  cfg.blockDim = dim3(AC_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (C > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = (unsigned)C;
    at[n].val.clusterDim.y = 1;
    at[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = at;
  cfg.numAttrs = n;
  AttendArgs at2 = a;
  at2.trace = debug_options().trace_at(TRACE_GEN);
  LAS_CUDA_OK(cudaLaunchKernelEx(&cfg, shared ? attend_cluster_kernel<true> : attend_cluster_kernel<false>, at2, C));
  LAS_LAUNCH_OK("attend_cluster_kernel");
  return LAS_OK;
}

}  // namespace las
