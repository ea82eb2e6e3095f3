// LAS_MODE_BF16 listener: tcgen05 input-projection GEMM (fast_gemm.cu) + cluster-resident LSTM recurrence.
//
// Recurrence kernel (SURVEY.md row a4; the h.W_hh^T + gates half of the nn.LSTM call at model/las_model.py:90):
//   * one thread-block CLUSTER per (direction, batch chunk of Bc utterances); forward and backward directions and
//     all batch chunks run concurrently in one launch;
//   * the cluster's CS CTAs split the hidden units 32 per CTA; each CTA keeps its [4 gates x 32 units, H] slice of
//     W_hh (bf16) resident in tensor memory for the whole sequence, as the A operand of a "swap-AB" UMMA:
//         D[128 gate rows, Bc] (TMEM, fp32) = W_slice[128, H] . h_{t-1}^T[H, Bc]
//   * h_{t-1} (bf16, the B operand) lives in every CTA's shared memory; after the gate math each CTA pushes its
//     32-unit slice of h_t into all CS CTAs' buffers with st.shared::cluster (DSMEM) and arrives on their mbarriers;
//   * c_t and the gate math stay fp32 in registers; the input projection P (from the GEMM, biases included) is
//     prefetched one step ahead.
// Gate rows are ordered unit-major / gate-minor (row = 4*unit + gate), so the four gates of a unit sit in four
// adjacent lanes of one warp after tcgen05.ld and are exchanged with warp shuffles.  The GEMM's weight rows are
// permuted the same way at pack time, so P[b,t] holds (i,f,g,o) of a unit as one float4.
#include <cuda.h>

#include "las_fast.cuh"
#include "las_kernels.cuh"
#include "umma.cuh"

namespace las {

int make_tmap_x_core(CUtensorMap* tm, const void* x_bf16, int B, int Tl, int Kx, int box_b);  // fast_gemm.cu

namespace {

// Warps: 4*EPW epilogue warps (TMEM lane quadrant = warp % 4, batch slice = warp / 4), then the MMA issuer, then the warp that
// watches the input-projection GEMM's tile flags (when it runs concurrently).  EPW = 2 up to 32 utterances per cluster; the
// 64-utterance chunk (serving pipeline: one cluster per direction next to the decoder) uses EPW = 4 so that a thread still
// owns only 4 cells.
template <int BC> struct RecCfg { static constexpr int EPW = BC >= 64 ? 4 : 2; static constexpr int THREADS = (4 * EPW + 2) * 32; };

struct RecParams {
  const float* P;               // [Tl*Bp, NP] fp32, time-major: row = t*Bp + b; column = dir*4Hp + r*128 + jj*4 + gate
  const uint32_t* gemm_flags;   // nullable [m_tiles * n_tiles]: the GEMM's per-tile completion counters (4 = tile stored)
  int Bp, n_tiles;              // padded batch (rows per time step of P); column tiles of the GEMM
  const uint8_t* whh_img;       // [2][CS] images of the W_hh slices (128 x Hp bf16, INTERLEAVE layout), copied to tensor memory
  float* out_f32;               // nullable [B, Tl, 2H]
  __nv_bfloat16* out_bf16;      // nullable [B, Tl, 2H]
  const int32_t* lengths;       // nullable [B]: valid steps of this layer (length-mask extension)
  int B, Tl, H, Hp, CS, nchunks;
  long long* trace;             // nullable test hook: [64 steps][8] clock64 stamps from CTA 0
  // Fused input projection (layer 0, template FX): the K = 2F projection X.W_ih^T is never materialised.  Each step's folded frames
  // x_t [BC, Kx] arrive by TMA straight in the B-operand layout, W_ih's slice sits in tensor memory next to W_hh's, and the Kx/16
  // extra MMAs of step s are issued while the CTA still waits for h_{s-1}.
  CUtensorMap tm_x;             // {8 k, B, Kx/8, Tl} view of the bf16 input [B, Tl, Kx]: a box {8, BC, Kx/8, 1} lands as [Kx/8][BC][8]
  const __nv_bfloat16* wih_img; // [2][CS][128][Kx] bf16, rows in gate-row order (= the GEMM's packed W_ih)
  const float* bias;            // [2][CS][128] b_ih + b_hh in gate-row order
  int Kx;
  int f16;                      // GEMM operand format: 0 = bf16, 1 = IEEE fp16
  int* resident;                // nullable: every CTA adds 1 once it is running (the serving pipeline launches the decoder, which takes
                                // all but a few SMs, only after this kernel's clusters have been placed)
};

#define REC_TRACE(slot) do { if (p.trace && blockIdx.x == 0 && s < 64) p.trace[s * 8 + (slot)] = clock64(); } while (0)

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(tanh_fast(0.5f * x), 0.5f, 0.5f); }
__device__ __forceinline__ float sel4(float a0, float a1, float a2, float a3, int i) {
  return i == 0 ? a0 : (i == 1 ? a1 : (i == 2 ? a2 : a3));
}

// W_hh slice operand: 128 rows x Hp, INTERLEAVE: K-adjacent core matrices 2048 B apart, 8-row groups 128 B apart
__host__ __device__ inline UmmaLayout whh_layout() { return UmmaLayout{0, 2048, 128, 0}; }
// h operand: Bc rows x Hp, INTERLEAVE: [coreK][coreN][8 rows][16 B]
__host__ __device__ inline UmmaLayout h_layout(int Bc) { return UmmaLayout{0, (uint32_t)Bc * 16u, 128, 0}; }

__host__ __device__ inline uint32_t rec_tmem_cols(int Hp, int BC, int Kx = 0) {
  // Kx > 0 (fused input projection): W_ih slice behind W_hh, and two accumulator sets (step s+1's input part is issued while the
  // epilogue still reads step s's)
  uint32_t need = (uint32_t)BC * (Kx > 0 ? 2u : 1u) + (uint32_t)Hp / 2 + (uint32_t)Kx / 2, c = 32;
  while (c < need) c <<= 1;
  return c;
}

constexpr int XSLOTS = 4;  // ring of x_t tiles (fused input projection)

template <int BC, bool FX>
__global__ void __launch_bounds__(RecCfg<BC>::THREADS, 1) lstm_recurrence_cluster_kernel(const __grid_constant__ RecParams p) {
  constexpr int EPW = RecCfg<BC>::EPW;
  constexpr int REC_MMA_WARP = 4 * EPW, REC_POLL_WARP = 4 * EPW + 1, REC_EPI_THREADS = 4 * EPW * 32;
  constexpr int HB = BC / EPW;  // batch columns per epilogue warp (EPW warps share a TMEM lane quadrant)
  constexpr int NB = HB / 4;    // cells per epilogue thread
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);  // offset from the __shared__ symbol keeps the address space
  const int Hp = p.Hp;
  const uint32_t a_bytes = 128u * Hp * 2u, h_bytes = (uint32_t)BC * Hp * 2u;
  uint8_t* sH0 = base;                                        // two h buffers of h_bytes each
  uint8_t* sStage = sH0 + 2 * h_bytes;                        // [2 parities] x (4 coreK x BC x 16 bytes)
  const uint32_t x_bytes = FX ? (uint32_t)BC * p.Kx * 2u : 0u;  // one x_t tile: [Kx/8][BC][8] bf16
  uint8_t* sX = sStage + 2 * 4 * BC * 16;                     // XSLOTS tiles (FX)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sX + XSLOTS * x_bytes);
  uint64_t* h_full = bars;        // [2]
  uint64_t* mma_done = bars + 2;  // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  int* s_ready = reinterpret_cast<int*>(bars + 4);  // steps (in processing order) whose P rows are known to be stored
  uint64_t* x_full = bars + 5;    // [XSLOTS]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t r = ptx::cluster_ctarank();
  const int CS = p.CS;
  const int cluster_id = blockIdx.x / CS;
  const int dir = cluster_id / p.nchunks, chunk = cluster_id % p.nchunks;
  const int b_base = chunk * BC;
  const uint32_t tcols = rec_tmem_cols(Hp, BC, FX ? p.Kx : 0);
  const uint8_t* w_img = p.whh_img + ((size_t)dir * CS + r) * a_bytes;

  // ---- one-time setup: barriers, TMEM, resident W_hh slice
  if (threadIdx.x == 0) {
    if (p.resident) atomicAdd(p.resident, 1);
    *s_ready = p.gemm_flags ? 0 : p.Tl;
    ptx::mbar_init(&h_full[0], 1);  // one local arrive.expect_tx per phase; the peers' bulk copies complete the bytes
    ptx::mbar_init(&h_full[1], 1);
    ptx::mbar_init(mma_done, 1);
    if (FX)
      for (int i = 0; i < XSLOTS; ++i) ptx::mbar_init(&x_full[i], 1);
    ptx::fence_mbar_init();
    // arm the first use of each h buffer (steps 1 and 2) before any peer can send
    if (p.Tl > 1) ptx::mbar_arrive_expect_tx(&h_full[1], h_bytes);
    if (p.Tl > 2) ptx::mbar_arrive_expect_tx(&h_full[0], h_bytes);
  }
  if (warp == REC_MMA_WARP) ptx::tmem_alloc(tmem_slot, tcols);
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // TMEM map: A operand (W_hh slice, lane = gate row, 2 bf16 per column) in columns [0, Hp/2), accumulator behind it
  const uint32_t x_col = (uint32_t)Hp / 2;                       // W_ih slice (FX): Kx/2 columns
  const uint32_t d_col = x_col + (FX ? (uint32_t)p.Kx / 2 : 0u);
  if (FX && warp < 4) {
    const __nv_bfloat16* wx = p.wih_img + ((size_t)(dir * CS + r) * 128 + threadIdx.x) * p.Kx;  // this lane's gate row
    for (int k0 = 0; k0 < p.Kx; k0 += 16) {
      const uint4 q0 = *reinterpret_cast<const uint4*>(wx + k0), q1 = *reinterpret_cast<const uint4*>(wx + k0 + 8);
      const uint32_t v[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
      ptx::tmem_st_32x32b_x8(tmem + ((uint32_t)(warp * 32) << 16) + x_col + k0 / 2, v);
    }
    ptx::tmem_st_wait();
  }
  if (warp < 4) {
    const UmmaLayout la = whh_layout();
    const int row = threadIdx.x;
    for (int k0 = 0; k0 < Hp; k0 += 16) {
      const uint4 q0 = *reinterpret_cast<const uint4*>(w_img + umma_offset(la, row, k0));
      const uint4 q1 = *reinterpret_cast<const uint4*>(w_img + umma_offset(la, row, k0 + 8));
      const uint32_t v[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
      ptx::tmem_st_32x32b_x8(tmem + ((uint32_t)(warp * 32) << 16) + k0 / 2, v);
    }
    ptx::tmem_st_wait();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();  // every CTA's barriers are initialised (and armed) before anyone sends
  ptx::tc_fence_after();
  const int Tl = p.Tl;

  if (warp == REC_MMA_WARP) {
    // ================================ MMA issuer ================================
    // The whole warp walks the loop with warp-uniform values (descriptors end up in uniform registers); only the
    // tcgen05 / mbarrier-arrive instructions are predicated on one elected lane.
    const UmmaLayout lb = h_layout(BC);
    const uint32_t idesc = umma_idesc_bf16(128, BC, p.f16);
    const uint32_t h0_addr = ptx::smem_u32(sH0);
    const uint32_t x0_addr = ptx::smem_u32(sX);
    // x_t tile of processing step `st` -> ring slot st % XSLOTS (all CTAs of the cluster read the same tile; it stays in L2)
    auto load_x = [&](int st) {
      const int t = dir ? Tl - 1 - st : st;
      uint64_t* bar = &x_full[st % XSLOTS];
      ptx::mbar_arrive_expect_tx(bar, x_bytes);
      asm volatile(
          "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
              x0_addr + (uint32_t)(st % XSLOTS) * x_bytes),
          "l"(reinterpret_cast<uint64_t>(&p.tm_x)), "r"(ptx::smem_u32(bar)), "r"(0), "r"(b_base), "r"(0), "r"(t)
          : "memory");
    };
    if (FX) {
      if (ptx::elect_one())
        for (int st = 0; st < XSLOTS - 1 && st < Tl; ++st) load_x(st);
    } else {
      if (ptx::elect_one()) ptx::mbar_arrive(mma_done);  // step 0: h_{-1} = 0, nothing to multiply
    }
    __syncwarp();
    for (int s = FX ? 0 : 1; s < Tl; ++s) {
      const uint32_t acc = tmem + d_col + (FX ? (uint32_t)(s & 1) * BC : 0u);
      if (FX) {
        // input part of step s: x_t . W_ih^T into a fresh accumulator, issued before h_{s-1} is here
        ptx::mbar_wait(&x_full[s % XSLOTS], (uint32_t)((s / XSLOTS) & 1));
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const UmmaLayout lx = h_layout(BC);
          const uint32_t xa = x0_addr + (uint32_t)(s % XSLOTS) * x_bytes;
#pragma unroll 1
          for (int ki = 0; ki < p.Kx / 16; ++ki)
            ptx::umma_bf16_ts(acc, tmem + x_col + ki * 8, umma_smem_desc(lx, xa, ki * 16), idesc, ki > 0);
          if (s == 0) ptx::umma_commit(mma_done);
        }
        __syncwarp();
        if (s == 0) {
          if (ptx::elect_one() && XSLOTS - 1 < Tl) load_x(XSLOTS - 1);
          __syncwarp();
          continue;
        }
      }
      ptx::mbar_wait(&h_full[s & 1], (uint32_t)((((s + 1) >> 1) - 1) & 1));
      if (lane == 0) REC_TRACE(0);
      ptx::tc_fence_after();
      const uint32_t b_addr = h0_addr + (uint32_t)(s & 1) * h_bytes;
      if (ptx::elect_one()) {
        if (s + 2 < Tl) ptx::mbar_arrive_expect_tx(&h_full[s & 1], h_bytes);  // re-arm for step s+2
        // Lean issue loop, one accumulator chain: the issuing thread's own instructions between two tcgen05.mma pace the chain (~40
        // cycles per instruction with the descriptor rebuilt each time, ~27 in tools/microbench_mma_insitu.cu's lean loop).  Consecutive
        // K steps are 8 tensor-memory columns and two core-matrix columns (2 * BC * 16 bytes) apart, so both operands advance by
        // constants (the descriptor's 14-bit address field cannot carry: shared memory ends below 256 KB).  Every chunk size BC
        // accumulates in this one order, so an utterance's result does not depend on how its batch is sharded.
        uint64_t bd = umma_smem_desc(lb, b_addr, 0);
        uint32_t a = tmem;
        ptx::umma_bf16_ts(acc, a, bd, idesc, FX ? 1u : 0u);
#pragma unroll 4
        for (int ki = 1; ki < Hp / 16; ++ki) {
          a += 8;
          bd += 2 * BC;
          ptx::umma_bf16_ts(acc, a, bd, idesc, 1u);
        }
        ptx::umma_commit(mma_done);
        // the MMAs of step s-1 are complete (h_s could not have arrived otherwise): its x slot takes the tile of step s + XSLOTS - 1
        if (FX && s + XSLOTS - 1 < Tl) load_x(s + XSLOTS - 1);
      }
      __syncwarp();
      if (lane == 0) REC_TRACE(1);
    }
  } else if (warp == REC_POLL_WARP) {
    // ================================ GEMM progress watcher ================================
    // One lane follows the tile flags of the column tile this CTA reads, in the order the recurrence consumes time steps, and
    // publishes how many steps are covered.  Each flag counts the GEMM's four epilogue warps.
    if (p.gemm_flags && lane == 0) {
      const int n_tile = (dir * 4 * Hp + (int)r * 128) >> 8;  // 256-column tiles of the GEMM
      int ready = 0;
      while (ready < Tl) {
        const int t = dir ? Tl - 1 - ready : ready;
        const long long m_tile = ((long long)t * p.Bp + b_base) >> 7;  // the chunk's 16 rows of a time step share one 128-row tile
        const uint32_t* f = p.gemm_flags + m_tile * p.n_tiles + n_tile;
        uint32_t v;
        ptx::SpinGuard guard;
        for (;;) {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
          if (v >= 4u) break;
          guard.tick();
        }
        do {  // every further step whose rows lie in the same tile
          ++ready;
        } while (ready < Tl && ((((long long)(dir ? Tl - 1 - ready : ready)) * p.Bp + b_base) >> 7) == m_tile);
        asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(ptx::smem_u32(s_ready)), "r"(ready) : "memory");
      }
    }
  } else {
    // ================================ gate math + h exchange ================================
    const int tid = threadIdx.x;
    const int wq = warp & 3, hb = warp >> 2;     // TMEM lane quadrant; batch half [hb*HB, hb*HB + HB) of the chunk
    const int row = wq * 32 + lane;              // TMEM lane = gate row = 4*jj + g
    const int jj = row >> 2, g = row & 3;
    const bool bit0 = (g & 1) != 0, bit1 = (g & 2) != 0;
    const int j = (int)r * 32 + jj;        // hidden unit
    const int NP = 8 * Hp;
    const float* pcol = FX ? nullptr : p.P + (size_t)dir * 4 * Hp + (size_t)r * 128 + jj * 4;
    // fused input projection: the accumulator already holds x_t.W_ih^T + h.W_hh^T; only the bias (i,f,g,o of this unit) is added
    const float4 bias4 = FX ? *reinterpret_cast<const float4*>(p.bias + (size_t)dir * 4 * Hp + (size_t)r * 128 + jj * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    float c[NB];
    float4 pnext[NB];
    int len[NB];  // valid steps of this thread's utterances: past them the cell keeps its state and emits h = 0
#pragma unroll
    for (int m = 0; m < NB; ++m) {
      c[m] = 0.f;
      const int b = b_base + hb * HB + 4 * m + g;
      len[m] = (p.lengths && b < p.B) ? p.lengths[b] : Tl;
    }
    // P rows may still be in flight from the concurrently running input-projection GEMM: `s_ready` (maintained by the
    // watcher warp) counts the steps, in processing order, whose rows are stored
    auto wait_ready = [&](int steps) {
      if (p.gemm_flags) {
        int v;
        do {
          asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"(ptx::smem_u32(s_ready)) : "memory");
        } while (v < steps);
      }
    };
    // P rows are loaded into registers one step ahead and pulled into L2 two steps ahead.  Steps run in blocks of 8 with the
    // readiness check between the blocks (20 steps ahead), so that the check (inline asm with a memory clobber) never sits
    // inside the step body, where it would pin the schedule of the P loads (measured: +8 % per step).
    wait_ready(Tl < 20 ? Tl : 20);
    {
      const int t0 = dir ? Tl - 1 : 0;
#pragma unroll
      for (int m = 0; m < NB; ++m) {
        const int b = b_base + hb * HB + 4 * m + g;
        pnext[m] = (!FX && b < p.B) ? *reinterpret_cast<const float4*>(pcol + ((size_t)t0 * p.Bp + b) * NP) : bias4;
      }
    }
    const uint32_t stage0 = ptx::smem_u32(sStage);
    const uint32_t h0_addr = ptx::smem_u32(sH0);
    const int dst_per_warp = (CS + 4 * EPW - 1) / (4 * EPW);  // destination CTAs each warp serves
    for (int s0 = 0; s0 < Tl; s0 += 8) {
    wait_ready(s0 + 20 < Tl ? s0 + 20 : Tl);
    const int s_end = s0 + 8 < Tl ? s0 + 8 : Tl;
    for (int s = s0; s < s_end; ++s) {
      const int t = dir ? Tl - 1 - s : s;
      float4 pc[NB];
#pragma unroll
      for (int m = 0; m < NB; ++m) pc[m] = pnext[m];
      if (!FX && s + 1 < Tl) {
        const int tn = dir ? t - 1 : t + 1;
#pragma unroll
        for (int m = 0; m < NB; ++m) {
          const int b = b_base + hb * HB + 4 * m + g;
          if (b < p.B) pnext[m] = *reinterpret_cast<const float4*>(pcol + ((size_t)tn * p.Bp + b) * NP);
        }
        if (s + 2 < Tl) {  // pull the step after that into L2 so the register prefetch above never sees DRAM latency
          const int tnn = dir ? t - 2 : t + 2;
#pragma unroll
          for (int m = 0; m < NB; ++m) {
            const int b = b_base + hb * HB + 4 * m + g;
            if (b < p.B) asm volatile("prefetch.global.L2 [%0];" ::"l"(pcol + ((size_t)tnn * p.Bp + b) * NP));
          }
        }
      }
      ptx::mbar_wait(mma_done, (uint32_t)(s & 1));
      if (tid == 0) REC_TRACE(2);
      uint32_t v[HB];
      if (FX || s > 0) {
        ptx::tc_fence_after();
        constexpr int LDW = HB < 16 ? HB : 16;  // columns per tcgen05.ld
#pragma unroll
        for (int c0 = 0; c0 < HB; c0 += LDW) {
          const uint32_t addr = tmem + ((uint32_t)(wq * 32) << 16) + d_col + (FX ? (uint32_t)(s & 1) * BC : 0u) + hb * HB + c0;
          if constexpr (LDW == 16) ptx::tmem_ld_32x32b_x16(addr, *reinterpret_cast<uint32_t(*)[16]>(v + c0));
          else ptx::tmem_ld_32x32b_x8(addr, *reinterpret_cast<uint32_t(*)[8]>(v + c0));
          ptx::tmem_ld_wait();
        }
        ptx::tc_fence_before();
      } else {
#pragma unroll
        for (int i = 0; i < HB; ++i) v[i] = 0u;
      }
      if (tid == 0) REC_TRACE(3);
      float hval[NB];
#pragma unroll
      for (int m = 0; m < NB; ++m) {
        // 4x4 transpose inside the 4-lane group (two butterfly stages, branch-free): lane g starts with its gate's
        // pre-activations for batches 4m..4m+3 and ends with all four gates (i,f,g,o) of batch 4m+g.
        float v0 = __uint_as_float(v[4 * m]), v1 = __uint_as_float(v[4 * m + 1]), v2 = __uint_as_float(v[4 * m + 2]),
              v3 = __uint_as_float(v[4 * m + 3]);
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
        const float a_i = v0 + pc[m].x, a_f = v1 + pc[m].y, a_g = v2 + pc[m].z, a_o = v3 + pc[m].w;
        const float cn = sigmoid_fast(a_f) * c[m] + sigmoid_fast(a_i) * tanh_fast(a_g);
        const bool on = t < len[m];
        c[m] = on ? cn : c[m];
        hval[m] = on ? sigmoid_fast(a_o) * tanh_fast(cn) : 0.f;
      }
      if (tid == 0) REC_TRACE(4);
      // ---- h_t slice -> every CTA of the cluster (B operand of step s+1)
      if (s + 1 < Tl) {
        // stage the CTA's 32-unit slice as 4 core-matrix columns (coreK = 4r + warp): [coreK][coreN][8 rows][8 k] bf16.
        // Double-buffered by step parity: the bulk copies issued at step s have landed in every peer before any CTA
        // can reach the epilogue of step s+2 (each peer needs them to finish its own step s+1).
        const uint32_t sb = stage0 + (uint32_t)(s & 1) * (4u * BC * 16u);
#pragma unroll
        for (int m = 0; m < NB; ++m) {
          const int bl = hb * HB + 4 * m + g;  // batch row within the chunk
          const uint32_t off = (uint32_t)wq * (BC * 16u) + (uint32_t)(bl >> 3) * 128u + (uint32_t)(bl & 7) * 16u + (uint32_t)(jj & 7) * 2u;
          const __nv_bfloat16 hb = op_from_f32(hval[m], p.f16);
          asm volatile("st.shared.b16 [%0], %1;" ::"r"(sb + off), "h"(*reinterpret_cast<const unsigned short*>(&hb)) : "memory");
        }
        ptx::fence_proxy_async_smem();  // generic-proxy staging writes -> visible to the bulk-copy (async proxy) reads
        asm volatile("bar.sync 1, %0;" ::"n"(REC_EPI_THREADS) : "memory");
        if (tid == 0) REC_TRACE(6);
        const int d = warp * dst_per_warp + lane;
        if (lane < dst_per_warp && d < CS) {
          // one DSMEM bulk copy of the whole slice per destination CTA; completes its bytes on that CTA's h_full barrier
          const uint32_t nb = (uint32_t)((s + 1) & 1);
          const uint32_t dst_rank = (r + d) % CS;
          const uint32_t dst_off = h0_addr + nb * h_bytes + ((uint32_t)(4 * r) * BC) * 16u;
          ptx::bulk_copy_to_cluster(ptx::mapa(dst_off, dst_rank), sb, 4u * BC * 16u, ptx::mapa(ptx::smem_u32(&h_full[nb]), dst_rank));
        }
        if (tid == 0) REC_TRACE(7);
      }
      // ---- outputs to global (off the critical path: after the exchange has been issued)
      if (j < p.H) {
#pragma unroll
        for (int m = 0; m < NB; ++m) {
          const int b = b_base + hb * HB + 4 * m + g;
          if (b < p.B) {
            const size_t o = ((size_t)b * Tl + t) * 2 * p.H + (size_t)dir * p.H + j;
            if (p.out_f32) p.out_f32[o] = hval[m];
            if (p.out_bf16) p.out_bf16[o] = op_from_f32(hval[m], p.f16);
          }
        }
      }
      if (tid == 0) REC_TRACE(5);
    }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();  // no CTA leaves while a peer could still address its shared memory
  if (warp == REC_MMA_WARP) ptx::tmem_dealloc(tmem, tcols);
}

// ---- pack kernels ------------------------------------------------------------------------------------------
// W_ih rows permuted to the recurrence's gate-row order, converted to bf16: dst [8Hp, K]
__global__ void pack_wih_kernel(const float* w_fwd, const float* w_rev, __nv_bfloat16* dst, int H, int Hp, int K, int f16) {
  const size_t n = (size_t)8 * Hp * K;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    const int row = (int)(i / K);
    const int dir = row / (4 * Hp), rem = row % (4 * Hp);
    const int unit = rem >> 2, gate = rem & 3;  // rem = r*128 + jj*4 + gate with unit = r*32 + jj
    const float* w = dir ? w_rev : w_fwd;
    dst[i] = op_from_f32(unit < H ? w[(size_t)(gate * H + unit) * K + k] : 0.f, f16);
  }
}
__global__ void pack_bias_kernel(const float* bi_f, const float* bh_f, const float* bi_r, const float* bh_r, float* dst, int H, int Hp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 8 * Hp) return;
  const int dir = i / (4 * Hp), rem = i % (4 * Hp);
  const int unit = rem >> 2, gate = rem & 3;
  const float* bi = dir ? bi_r : bi_f;
  const float* bh = dir ? bh_r : bh_f;
  dst[i] = unit < H ? bi[gate * H + unit] + bh[gate * H + unit] : 0.f;
}
// W_hh -> per (dir, rank) shared-memory images of the 128 x Hp A operand
__global__ void pack_whh_kernel(const float* w_fwd, const float* w_rev, uint8_t* img, int H, int Hp, int CS, int f16) {
  const size_t per = (size_t)128 * Hp;
  const size_t n = 2 * (size_t)CS * per;
  const UmmaLayout la = whh_layout();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % Hp);
    const int row = (int)((i / Hp) % 128);
    const int rk = (int)((i / per) % CS);
    const int dir = (int)(i / (per * CS));
    const int unit = rk * 32 + (row >> 2), gate = row & 3;
    const float* w = dir ? w_rev : w_fwd;
    const float val = (unit < H && k < H) ? w[(size_t)(gate * H + unit) * H + k] : 0.f;
    *reinterpret_cast<__nv_bfloat16*>(img + ((size_t)dir * CS + rk) * per * 2 + umma_offset(la, row, k)) = op_from_f32(val, f16);
  }
}

// Side stream on which a layer's input-projection GEMM runs while the recurrence consumes its tiles on the caller's
// stream.  One per host thread and device, created on first use and kept (entry points stay re-entrant: nothing here is
// shared between threads).
struct SideStream {
  int dev = -1;
  cudaStream_t s = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
thread_local SideStream g_side;
int side_stream(SideStream** out) {
  int dev = -1;
  LAS_CUDA_OK(cudaGetDevice(&dev));
  if (g_side.s == nullptr || g_side.dev != dev) {
    if (g_side.s) {
      cudaStreamDestroy(g_side.s);
      cudaEventDestroy(g_side.fork);
      cudaEventDestroy(g_side.join);
      g_side = SideStream();
    }
    LAS_CUDA_OK(cudaStreamCreateWithFlags(&g_side.s, cudaStreamNonBlocking));
    LAS_CUDA_OK(cudaEventCreateWithFlags(&g_side.fork, cudaEventDisableTiming));
    LAS_CUDA_OK(cudaEventCreateWithFlags(&g_side.join, cudaEventDisableTiming));
    g_side.dev = dev;
  }
  *out = &g_side;
  return LAS_OK;
}

struct Geo {
  int Hp, CS;
  bool ok;
};
Geo geometry(int H) {
  Geo g;
  g.CS = (H + 31) / 32;
  g.Hp = g.CS * 32;
  g.ok = (g.CS == 1 || g.CS == 2 || g.CS == 4 || g.CS == 8 || g.CS == 16) && (H <= 32 || H % 32 == 0);
  return g;
}
int pick_bc(int B, int CS) {
  // batch chunk per cluster (the UMMA N): multiples of 16; grow it only when the clusters would not fit the chip
  const int max_clusters = sm_count() / CS > 0 ? sm_count() / CS : 1;
  int bc = 16;
  while (bc < 64 && 2 * ((B + bc - 1) / bc) > max_clusters) bc *= 2;
  return bc;
}

struct ListenerPackFast {
  __nv_bfloat16* wih[16];
  float* bias[16];
  uint8_t* whh[16];
  size_t bytes;
};
ListenerPackFast pack_layout(const las_listener_dims* d, void* base) {
  ListenerPackFast p;
  const Geo g = geometry(d->H);
  Carver cv(base);
  for (int l = 0; l < d->L; ++l) {
    const size_t K = (l == 0) ? 2 * (size_t)d->F : 4 * (size_t)d->H;
    p.wih[l] = cv.take<__nv_bfloat16>(8 * (size_t)g.Hp * K);
    p.bias[l] = cv.take<float>(8 * (size_t)g.Hp);
    p.whh[l] = cv.take<uint8_t>(2 * (size_t)g.CS * 128 * g.Hp * 2);
  }
  p.bytes = cv.total();
  return p;
}
struct ListenerWsFast {
  __nv_bfloat16* xb;
  float* P;
  __nv_bfloat16* act[2];
  int32_t* len;  // [L][B]
  uint32_t* flags;  // per-tile completion counters of the layer's input-projection GEMM
  size_t n_flags;
  size_t bytes;
};
ListenerWsFast ws_layout(const las_listener_dims* d, void* base) {
  ListenerWsFast w;
  const Geo g = geometry(d->H);
  Carver cv(base);
  const size_t M0 = (size_t)d->B * (d->T / 2);
  const size_t M0p = (size_t)listener_padded_batch(d->B) * (d->T / 2);  // P is time-major with the batch padded per time step
  w.xb = cv.take<__nv_bfloat16>((size_t)d->B * d->T * d->F);
  w.P = cv.take<float>(M0p * 8 * g.Hp);
  w.n_flags = (M0p / 128 + 1) * ((size_t)(8 * g.Hp + 255) / 256);
  w.flags = cv.take<uint32_t>(w.n_flags);
  w.act[0] = cv.take<__nv_bfloat16>(M0 * 2 * d->H);
  w.act[1] = cv.take<__nv_bfloat16>(M0 / 2 * 2 * d->H + 64);
  w.len = cv.take<int32_t>((size_t)d->L * d->B);
  w.bytes = cv.total();
  return w;
}

int shape_ok(const las_listener_dims* d) {
  const Geo g = geometry(d->H);
  LAS_REQUIRE(g.ok, "LAS_MODE_BF16 listener supports hidden sizes <= 32 or 64/128/256/512 (H=%d); use LAS_MODE_FP32", d->H);
  LAS_REQUIRE((2 * d->F) % 8 == 0 && (4 * d->H) % 8 == 0,
              "LAS_MODE_BF16 needs 16-byte aligned bf16 rows for TMA: 2F (%d) and 4H (%d) must be multiples of 8", 2 * d->F, 4 * d->H);
  return LAS_OK;
}

template <int BC, bool FX>
int launch_rec(const RecParams& p, cudaStream_t st, bool exclusive_sm) {
  size_t smem = 1024 + 2u * BC * p.Hp * 2 + 2 * 4 * BC * 16 + (FX ? XSLOTS * (size_t)BC * p.Kx * 2 : 0) + 128;
  // While the GEMM runs concurrently, a GEMM CTA (197 KB of shared memory, all 512 TMEM columns) must never land on an SM that
  // hosts a recurrence CTA (it would wait for tensor memory held by a CTA that waits for the GEMM's tiles): ask for enough
  // shared memory that the two cannot be co-resident.
  if (exclusive_sm && smem < 48 * 1024) smem = 48 * 1024;
  LAS_CUDA_OK(cudaFuncSetAttribute(lstm_recurrence_cluster_kernel<BC, FX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (p.CS > 8) LAS_CUDA_OK(cudaFuncSetAttribute(lstm_recurrence_cluster_kernel<BC, FX>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(p.CS * 2 * p.nchunks);
  cfg.blockDim = dim3(p.gemm_flags ? RecCfg<BC>::THREADS : RecCfg<BC>::THREADS - 32);  // the watcher warp exists only next to a concurrent GEMM
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = p.CS;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  LAS_CUDA_OK(cudaLaunchKernelEx(&cfg, lstm_recurrence_cluster_kernel<BC, FX>, p));
  count_launch();
  return LAS_OK;
}

}  // namespace

// Does the cluster-resident recurrence cover this model?  (Otherwise las_api.cu runs the generic path: tensor-core input projection,
// fp32 recurrent kernel.)
bool fast_listener_fits(const las_listener_dims* d) {
  const Geo g = geometry(d->H);
  return d->cell == LAS_CELL_LSTM && g.ok && (2 * d->F) % 8 == 0 && (4 * d->H) % 8 == 0;
}
size_t fast_listener_packed_bytes(const las_listener_dims* d) { return pack_layout(d, nullptr).bytes; }
size_t fast_listener_workspace_bytes(const las_listener_dims* d) { return ws_layout(d, nullptr).bytes; }

int fast_listener_pack(const las_lstm_weights* w, const las_listener_dims* d, void* packed, bool f16, cudaStream_t st) {
  LAS_TRY(shape_ok(d));
  const Geo g = geometry(d->H);
  const ListenerPackFast pk = pack_layout(d, packed);
  for (int l = 0; l < d->L; ++l) {
    const int K = (l == 0) ? 2 * d->F : 4 * d->H;
    const las_lstm_weights &f = w[2 * l], &r = w[2 * l + 1];
    LAS_REQUIRE(f.w_ih && f.w_hh && f.b_ih && f.b_hh && r.w_ih && r.w_hh && r.b_ih && r.b_hh, "null weight pointer in layer %d", l);
    pack_wih_kernel<<<592, 256, 0, st>>>(f.w_ih, r.w_ih, pk.wih[l], d->H, g.Hp, K, f16);
    LAS_LAUNCH_OK("pack_wih_kernel");
    pack_bias_kernel<<<(8 * g.Hp + 255) / 256, 256, 0, st>>>(f.b_ih, f.b_hh, r.b_ih, r.b_hh, pk.bias[l], d->H, g.Hp);
    LAS_LAUNCH_OK("pack_bias_kernel");
    pack_whh_kernel<<<592, 256, 0, st>>>(f.w_hh, r.w_hh, pk.whh[l], d->H, g.Hp, g.CS, f16);
    LAS_LAUNCH_OK("pack_whh_kernel");
  }
  return LAS_OK;
}

// One stage of the listener: stage 0 = input cast, 1 + 2l = layer l's input-projection GEMM, 2 + 2l = layer l's recurrence.
// fast_listener_forward chains them (GEMM concurrent with the recurrence where possible); the serving pipeline (fast_pipeline.cu)
// issues them one by one between / next to the decoder's segments.
struct LayerGeom {
  const __nv_bfloat16* in;
  int Tl, K, NP;
};
static LayerGeom layer_geom(const las_listener_dims* d, const Geo& g, const ListenerWsFast& w, int l) {
  LayerGeom q;
  q.in = (l == 0) ? w.xb : w.act[(l - 1) & 1];
  q.Tl = d->T >> (l + 1);
  q.K = (l == 0) ? 2 * d->F : 4 * d->H;
  q.NP = 8 * g.Hp;
  return q;
}
static RecParams rec_params(const las_listener_dims* d, const Geo& g, const ListenerPackFast& pk, const ListenerWsFast& w, int l, float* enc,
                            const int32_t* len_l, int bc, bool f16) {
  const LayerGeom q = layer_geom(d, g, w, l);
  const bool last = (l == d->L - 1);
  RecParams rp;
  rp.P = w.P;
  rp.gemm_flags = nullptr;
  rp.Bp = listener_padded_batch(d->B);
  rp.n_tiles = (q.NP + 255) / 256;
  rp.whh_img = pk.whh[l];
  rp.out_f32 = last ? enc : nullptr;
  rp.out_bf16 = last ? nullptr : w.act[l & 1];
  rp.lengths = len_l;
  rp.B = d->B; rp.Tl = q.Tl; rp.H = d->H; rp.Hp = g.Hp; rp.CS = g.CS;
  rp.trace = (l == 0) ? debug_options().trace_at(TRACE_REC) : nullptr;
  rp.nchunks = (d->B + bc - 1) / bc;
  rp.resident = nullptr;
  rp.f16 = f16;
  rp.Kx = 0;
  rp.wih_img = nullptr;
  rp.bias = nullptr;
  memset(&rp.tm_x, 0, sizeof(rp.tm_x));
  return rp;
}
// switch layer 0's recurrence to the fused input projection
static int rec_fuse(RecParams& rp, const las_listener_dims* d, const ListenerPackFast& pk, const ListenerWsFast& w, int bc) {
  rp.Kx = 2 * d->F;
  rp.wih_img = pk.wih[0];
  rp.bias = pk.bias[0];
  rp.P = nullptr;
  return make_tmap_x_core(&rp.tm_x, w.xb, d->B, d->T / 2, rp.Kx, bc);
}
static int launch_rec_bc(const RecParams& rp, int bc, cudaStream_t st, bool exclusive) {
  if (rp.Kx > 0) {  // fused input projection (layer 0)
    if (bc == 16) return launch_rec<16, true>(rp, st, exclusive);
    if (bc == 32) return launch_rec<32, true>(rp, st, exclusive);
    return launch_rec<64, true>(rp, st, exclusive);
  }
  if (bc == 16) return launch_rec<16, false>(rp, st, exclusive);
  if (bc == 32) return launch_rec<32, false>(rp, st, exclusive);
  return launch_rec<64, false>(rp, st, exclusive);
}

// layer l's input projection can be fused when K = 2F splits into 16-wide MMA steps
static bool fuse_x(const las_listener_dims* d, int l) { return l == 0 && (2 * d->F) % 16 == 0 && 2 * d->F <= 256; }

// CTAs the recurrence of this model occupies with batch chunk `bc`
int fast_listener_rec_ctas(const las_listener_dims* d, int bc) {
  const Geo g = geometry(d->H);
  return 2 * ((d->B + bc - 1) / bc) * g.CS;
}

int fast_listener_stage(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d, float* enc,
                        int32_t* enc_lengths, void* ws, int stage, int bc, int* resident, int max_ctas, bool f16, cudaStream_t st) {
  LAS_TRY(shape_ok(d));
  const Geo g = geometry(d->H);
  const ListenerPackFast pk = pack_layout(d, const_cast<void*>(packed));
  const ListenerWsFast w = ws_layout(d, ws);
  char nm[48];
  if (stage == 0) {
    ProfScope ps("listener.cast_bf16", st);
    return launch_f32_to_bf16(x, w.xb, (size_t)d->B * d->T * d->F, f16, st);
  }
  const int l = (stage - 1) / 2;
  const LayerGeom q = layer_geom(d, g, w, l);
  if ((stage - 1) % 2 == 0) {
    if (x_lengths) LAS_TRY(launch_pyramid_lengths(l == 0 ? x_lengths : w.len + (size_t)(l - 1) * d->B, w.len + (size_t)l * d->B, d->B, q.Tl, st));
    if (fuse_x(d, l)) return LAS_OK;  // the recurrence does the projection itself
    snprintf(nm, sizeof(nm), "listener.L%d.input_gemm", l);
    ProfScope ps(nm, st);
    return launch_gemm_listener(q.in, d->B, q.Tl, q.K, pk.wih[l], pk.bias[l], w.P, q.NP, nullptr, max_ctas, f16, st);
  }
  RecParams rp = rec_params(d, g, pk, w, l, enc, x_lengths ? w.len + (size_t)l * d->B : nullptr, bc, f16);
  rp.resident = resident;
  if (fuse_x(d, l)) LAS_TRY(rec_fuse(rp, d, pk, w, bc));
  snprintf(nm, sizeof(nm), "listener.L%d.recurrence", l);
  {
    ProfScope ps(nm, st);
    LAS_TRY(launch_rec_bc(rp, bc, st, true));
  }
  if (l == d->L - 1 && x_lengths && enc_lengths)
    LAS_CUDA_OK(cudaMemcpyAsync(enc_lengths, w.len + (size_t)(d->L - 1) * d->B, sizeof(int32_t) * d->B, cudaMemcpyDeviceToDevice, st));
  return LAS_OK;
}

// events / side stream of the calling thread (fast_pipeline.cu)
int fast_side_stream(cudaStream_t* s) {
  SideStream* side = nullptr;
  LAS_TRY(side_stream(&side));
  *s = side->s;
  return LAS_OK;
}

int fast_listener_forward(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d, float* enc,
                          int32_t* enc_lengths, void* ws, bool f16, cudaStream_t st) {
  LAS_TRY(shape_ok(d));
  const Geo g = geometry(d->H);
  const ListenerPackFast pk = pack_layout(d, const_cast<void*>(packed));
  const ListenerWsFast w = ws_layout(d, ws);
  const int B = d->B;
  LAS_TRY(fast_listener_stage(x, x_lengths, packed, d, enc, enc_lengths, ws, 0, 0, nullptr, 0, f16, st));
  for (int l = 0; l < d->L; ++l) {
    const LayerGeom q = layer_geom(d, g, w, l);
    const int32_t* len_l = nullptr;
    if (x_lengths) {
      LAS_TRY(launch_pyramid_lengths(l == 0 ? x_lengths : w.len + (size_t)(l - 1) * B, w.len + (size_t)l * B, B, q.Tl, st));
      len_l = w.len + (size_t)l * B;
    }
    const int bc = debug_options().rec_force_bc ? debug_options().rec_force_bc : pick_bc(B, g.CS);
    RecParams rp = rec_params(d, g, pk, w, l, enc, len_l, bc, f16);
    // The GEMM emits its tiles in the recurrence's consumption order and flags each one, so it can run next to the recurrence
    // (which occupies 2 * nchunks * CS SMs) on the remaining SMs instead of in front of it.  Needs the two directions' columns
    // to fall on separate column tiles and enough free SMs to be worth it.
    if (fuse_x(d, l)) {
      // layer 0: K = 2F = 80 makes the projection's [B*T/2, 8H] fp32 output (419 MB at c3) the cost, not its flops (SURVEY.md
      // 7.2.3): it is never materialised, the recurrence multiplies x_t itself
      LAS_TRY(rec_fuse(rp, d, pk, w, bc));
      ProfScope ps("listener.L0.recurrence", st);
      LAS_TRY(launch_rec_bc(rp, bc, st, false));
      continue;
    }
    const int rec_ctas = 2 * rp.nchunks * g.CS;
    const int gemm_ctas = sm_count() - rec_ctas - 4;
    const bool overlap = debug_options().rec_overlap && ((q.NP / 2) % 256 == 0) && gemm_ctas >= 32;
    SideStream* side = nullptr;
    if (overlap) LAS_TRY(side_stream(&side));
    if (overlap) rp.gemm_flags = w.flags;
    char nm[48];
    if (overlap) LAS_CUDA_OK(cudaMemsetAsync(w.flags, 0, sizeof(uint32_t) * w.n_flags, st));
    {
      // pyramid fold = reading [B, Tin, Fin] as [B, Tl, 2*Fin] (model/las_model.py:86-87): only the tensor map changes.
      // The output is time-major (row = t*Bp + b).
      cudaStream_t gs = st;
      if (overlap) {
        LAS_CUDA_OK(cudaEventRecord(side->fork, st));
        LAS_CUDA_OK(cudaStreamWaitEvent(side->s, side->fork, 0));
        gs = side->s;
      }
      snprintf(nm, sizeof(nm), overlap ? "listener.L%d.input_gemm.overlapped" : "listener.L%d.input_gemm", l);
      ProfScope ps(nm, gs);
      LAS_TRY(launch_gemm_listener(q.in, B, q.Tl, q.K, pk.wih[l], pk.bias[l], w.P, q.NP, overlap ? w.flags : nullptr, overlap ? gemm_ctas : 0, f16, gs));
    }
    {
      snprintf(nm, sizeof(nm), "listener.L%d.recurrence", l);
      ProfScope ps(nm, st);
      LAS_TRY(launch_rec_bc(rp, bc, st, overlap));
    }
    if (overlap) {  // the GEMM kernel has delivered every tile by now; join so that P / flags can be reused by the next layer
      LAS_CUDA_OK(cudaEventRecord(side->join, side->s));
      LAS_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
    }
  }
  if (x_lengths && enc_lengths)
    LAS_CUDA_OK(cudaMemcpyAsync(enc_lengths, w.len + (size_t)(d->L - 1) * B, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, st));
  return LAS_OK;
}

}  // namespace las
