// Listener input projection on the 5th-gen tensor cores (SURVEY.md row a3):
//     P[M, N] = A[M, K] . W[N, K]^T + bias[N]        A, W bf16 (K-major), P fp32, fp32 accumulation in TMEM
// Replaces the x.W_ih^T half of the nn.LSTM call at model/las_model.py:90 for all timesteps and both directions
// at once (N = 8H).  The pyramid fold (:86-87) costs nothing: [B, 2Tl, Fin] and [B*Tl, 2Fin] are the same memory,
// so the fold is just the tensor map's shape.
//
// Structure (one CTA per SM, persistent over 128x256 output tiles):
//   warp 0     TMA producer: cp.async.bulk.tensor 2-D loads of A (128x64) and W (256x64) tiles, SWIZZLE_128B,
//              4-stage mbarrier ring; K / M / N tails are TMA out-of-bounds zero fill
//   warp 1     TMEM allocator + single-thread tcgen05.mma issuer (M=128, N=256, K=16 per instruction),
//              tcgen05.commit releases smem stages and publishes finished accumulators
//   warps 2-5  epilogue: tcgen05.ld accumulator rows -> +bias -> a 32x32 fp32 block per warp in shared memory (128-byte rows,
//              chunk-swizzled: conflict-free) -> one TMA store per block (full 128-byte lines; M / N tails clipped by the
//              tensor map); two 256-column accumulators in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//              Row-per-thread st.global.v4 stores (32 partial lines per instruction) are the other epilogue: slower when the
//              GEMM has the chip to itself (K=80: 172 vs 148 us, K=1024: 129 vs 104 us), but the one used when the GEMM runs next to
//              the listener's recurrence with tile flags: there the bulk stores slow the recurrence by ~5 % (1.70 vs 1.66 ms per
//              listener pass, profiles/r01_gemm_epilogue_ab.log), and the GEMM is hidden behind the recurrence anyway.
#include <cuda.h>
#include <string.h>

#include "las_fast.cuh"
#include "umma.cuh"

namespace las {

namespace {

constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4;
constexpr int A_TILE_BYTES = BM * BK * 2, B_TILE_BYTES = BN * BK * 2;
constexpr int GEMM_THREADS = 192;

constexpr int EPI_BLOCK_BYTES = 32 * 32 * 4;  // one epilogue warp's staging block: 32 rows x 32 fp32
struct __align__(1024) GemmSmem {
  uint8_t a[STAGES][A_TILE_BYTES];
  uint8_t b[STAGES][B_TILE_BYTES];
  uint8_t epi[4][2][EPI_BLOCK_BYTES];  // [epilogue warp][double buffer]: source of the TMA stores (1024-byte aligned blocks)
  uint64_t full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
};

// Tile schedule / A-operand addressing.  mode 0: A is a plain [M, K] matrix, tiles in natural order.  mode 1 (listener):
// A is the 3-D view {K, b, t} of the layer input, output row r = t*Bp + b; tile i of the schedule is
//   (m = i / n_tiles,               n = i % n_tiles)   for the forward direction's column tiles  (n <  nfwd)
//   (m = m_tiles - 1 - i / n_tiles, n = i % n_tiles)   for the backward direction's             (n >= nfwd)
// i.e. the recurrence's consumption order: early time steps for the forward LSTM, late ones for the backward LSTM.
struct GemmSched {
  int mode, Bp, nfwd;
  int f16;          // operand format of A and W: 0 = bf16, 1 = IEEE fp16
  uint32_t* flags;  // nullable: [m_tiles * n_tiles] counters, +1 per epilogue warp that has stored its rows of the tile
};
__device__ __forceinline__ void sched_tile(const GemmSched& sc, int i, int m_tiles, int n_tiles, int& m, int& n) {
  n = i % n_tiles;
  m = i / n_tiles;
  if (sc.mode == 1 && n >= sc.nfwd) m = m_tiles - 1 - m;
}

__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                    const __grid_constant__ CUtensorMap tm_c, const float* __restrict__ bias, float* __restrict__ C, long long ldc,
                    int M, int N, int K, int relu, int tma_store, const GemmSched sc) {
  extern __shared__ uint8_t smem_raw[];
  GemmSmem& s = *reinterpret_cast<GemmSmem*>(smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u));  // offset from the __shared__ symbol keeps the address space
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (M + BM - 1) / BM, n_tiles = (N + BN - 1) / BN, k_blocks = (K + BK - 1) / BK;
  const int num_tiles = m_tiles * n_tiles;

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tm_a);
    ptx::prefetch_tensormap(&tm_b);
    if (tma_store) ptx::prefetch_tensormap(&tm_c);
    for (int i = 0; i < STAGES; ++i) {
      ptx::mbar_init(&s.full[i], 1);
      ptx::mbar_init(&s.empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&s.tmem_full[i], 1);
      ptx::mbar_init(&s.tmem_empty[i], 128);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc(&s.tmem_base, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = s.tmem_base;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int mt, nt;
        sched_tile(sc, tile, m_tiles, n_tiles, mt, nt);
        const int m0 = mt * BM, n0 = nt * BN;
        for (int kb = 0; kb < k_blocks; ++kb) {
          ptx::mbar_wait(&s.empty[stage], phase ^ 1);
          ptx::mbar_arrive_expect_tx(&s.full[stage], A_TILE_BYTES + B_TILE_BYTES);
          if (sc.mode == 1) ptx::tma_load_3d(s.a[stage], &tm_a, &s.full[stage], kb * BK, m0 % sc.Bp, m0 / sc.Bp);  // rows = (t, b) pairs
          else ptx::tma_load_2d(s.a[stage], &tm_a, &s.full[stage], kb * BK, m0);
          ptx::tma_load_2d(s.b[stage], &tm_b, &s.full[stage], kb * BK, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const UmmaLayout la{1, 0, 1024, A_TILE_BYTES}, lb{1, 0, 1024, B_TILE_BYTES};
      const uint32_t idesc = umma_idesc_bf16(BM, BN, sc.f16);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        ptx::mbar_wait(&s.tmem_empty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < k_blocks; ++kb) {
          ptx::mbar_wait(&s.full[stage], phase);
          ptx::tc_fence_after();
          const uint32_t a_addr = ptx::smem_u32(s.a[stage]), b_addr = ptx::smem_u32(s.b[stage]);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            ptx::umma_bf16(d_tmem, umma_smem_desc(la, a_addr, k * 16), umma_smem_desc(lb, b_addr, k * 16), idesc, (kb | k) != 0);
          ptx::umma_commit(&s.empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        ptx::umma_commit(&s.tmem_full[acc]);
      }
    }
  } else {
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const bool vec_ok = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
    int it = 0;
    if (tma_store) {
      // ---- TMA-store epilogue.  Bulk groups: one per 32-column block, 8 per tile.
      uint8_t* const blk0 = s.epi[q][0];
      const uint32_t sw = (uint32_t)(lane & 7);
      uint32_t nblk = 0;                 // blocks issued so far by this warp (buffer = nblk & 1)
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        int mt, nt;
        sched_tile(sc, tile, m_tiles, n_tiles, mt, nt);
        const int m0 = mt * BM, n0 = nt * BN;
        ptx::mbar_wait(&s.tmem_full[acc], acc_phase);
        ptx::tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          const int col0 = n0 + c0;
          if (col0 >= N) break;  // warp-uniform: this and the following blocks lie beyond the last column
          uint32_t v[32];
          ptx::tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + c0, v);
          ptx::tmem_ld_wait();
          uint8_t* dst = blk0 + (nblk & 1) * EPI_BLOCK_BYTES;
          if (nblk >= 2) {  // the store issued from this buffer two blocks ago must have read it
            if (lane == 0) ptx::tma_store_wait_read<1>();
            __syncwarp();
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 bv;
            if (col0 + 4 * j + 3 < N) bv = *reinterpret_cast<const float4*>(bias + col0 + 4 * j);
            else {
              bv.x = col0 + 4 * j < N ? bias[col0 + 4 * j] : 0.f;
              bv.y = col0 + 4 * j + 1 < N ? bias[col0 + 4 * j + 1] : 0.f;
              bv.z = col0 + 4 * j + 2 < N ? bias[col0 + 4 * j + 2] : 0.f;
              bv.w = 0.f;
            }
            float4 o;
            o.x = __uint_as_float(v[4 * j]) + bv.x;
            o.y = __uint_as_float(v[4 * j + 1]) + bv.y;
            o.z = __uint_as_float(v[4 * j + 2]) + bv.z;
            o.w = __uint_as_float(v[4 * j + 3]) + bv.w;
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            // row `lane`, 16-byte chunk j at the SWIZZLE_128B position: the 8 lanes of a quarter warp fill all 32 banks
            *reinterpret_cast<float4*>(dst + lane * 128 + (((uint32_t)j ^ sw) << 4)) = o;
          }
          ptx::fence_proxy_async_smem();  // generic-proxy writes above -> the bulk store's async-proxy reads
          __syncwarp();
          if (lane == 0) {
            if (m0 + q * 32 < M) ptx::tma_store_2d(&tm_c, dst, col0, m0 + q * 32);  // rows >= M / columns >= N are clipped
            ptx::tma_store_commit();
          }
          ++nblk;
        }
        ptx::tc_fence_before();
        ptx::mbar_arrive(&s.tmem_empty[acc]);
      }
      if (lane == 0) ptx::tma_store_wait<0>();  // every store has read its buffer and landed before the CTA retires
      __syncwarp();
    } else
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      int mt, nt;
      sched_tile(sc, tile, m_tiles, n_tiles, mt, nt);
      const int m0 = mt * BM, n0 = nt * BN;
      ptx::mbar_wait(&s.tmem_full[acc], acc_phase);
      ptx::tc_fence_after();
      const int row = m0 + q * 32 + lane;
      float* crow = C + (long long)row * ldc;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + c0, v);
        ptx::tmem_ld_wait();
        const int col0 = n0 + c0;
        if (row < M && col0 < N) {
          if (vec_ok && col0 + 32 <= N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bv = *reinterpret_cast<const float4*>(bias + col0 + j);
              float4 o;
              o.x = __uint_as_float(v[j]) + bv.x;
              o.y = __uint_as_float(v[j + 1]) + bv.y;
              o.z = __uint_as_float(v[j + 2]) + bv.z;
              o.w = __uint_as_float(v[j + 3]) + bv.w;
              if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              *reinterpret_cast<float4*>(crow + col0 + j) = o;
            }
          } else {
            for (int j = 0; j < 32; ++j)
              if (col0 + j < N) {
                const float o = __uint_as_float(v[j]) + bias[col0 + j];
                crow[col0 + j] = relu ? fmaxf(o, 0.f) : o;
              }
          }
        }
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(&s.tmem_empty[acc]);
      if (sc.flags) {  // this warp's 32 rows of the tile are stored: publish (the release is cumulative over the warp barrier)
        __syncwarp();
        if (lane == 0) asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(sc.flags + (size_t)mt * n_tiles + nt), "r"(1u) : "memory");
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 512);
}

// ---- host: tensor maps ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  LAS_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
  *out = reinterpret_cast<EncodeTiledFn>(fn);
  return LAS_OK;
}

// row-major bf16 matrix [rows, cols] with row pitch `ld` elements; box = {64 cols, box_rows}, 128-byte swizzle
int make_tmap_bf16(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows) {
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  LAS_REQUIRE((ld * 2) % 16 == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0,
              "TMA needs 16-byte aligned rows (ld=%lld elements)", ld);
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", (int)r, rows, cols, ld);
  return LAS_OK;
}

// row-major fp32 matrix [rows, cols] with row pitch `ld` elements; box = {32 cols, 32 rows}, 128-byte swizzle (TMA store target)
int make_tmap_f32_store(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld) {
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled (fp32 output) failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", (int)r, rows, cols, ld);
  return LAS_OK;
}
// TMA can address the output when the base and the row pitch are 16-byte aligned; otherwise the kernel stores rows directly.
// Narrow outputs (psi: N = 64, two blocks per tile) are a little faster with direct stores (14.3 vs 16.4 us), so they keep them.
bool tma_store_ok(const float* C, long long ldc, int N, const uint32_t* flags) {
  return (reinterpret_cast<uintptr_t>(C) & 15) == 0 && (ldc * 4) % 16 == 0 && N >= 128 && !flags && !debug_options().gemm_direct_store;
}

}  // namespace

int make_tmap_bf16_box(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows) {
  return make_tmap_bf16(tm, base, rows, cols, ld, box_rows);
}

// General 16-bit tensor map, 128-byte swizzle: dims / box innermost first (dims[0] = box[0] = 64 elements), strides in bytes for
// dimensions 1..rank-1.
int make_tmap_bf16_nd(CUtensorMap* tm, const void* base, int rank, const unsigned long long* dims, const unsigned long long* strides,
                      const unsigned* box) {
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  LAS_REQUIRE(rank >= 2 && rank <= 5 && (reinterpret_cast<uintptr_t>(base) & 15) == 0, "bad tensor map request (rank=%d)", rank);
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], estr[5] = {1, 1, 1, 1, 1};
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    if (i) {
      LAS_REQUIRE(strides[i - 1] % 16 == 0, "TMA needs 16-byte aligned strides (dimension %d: %llu bytes)", i, strides[i - 1]);
      gstr[i - 1] = strides[i - 1];
    }
  }
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled (rank %d) failed with CUresult %d", rank, (int)r);
  return LAS_OK;
}

// The same row-major bf16 matrix [rows, 64*atoms] seen as {64 k, rows, atoms}: one copy of box {64, box_rows, box_atoms}
// lands as box_atoms consecutive 128-byte-swizzled [box_rows x 64] atoms, i.e. what box_atoms 2-D copies would write.
int make_tmap_bf16_atoms(CUtensorMap* tm, const void* base, long long rows, int atoms, long long ld, int box_rows, int box_atoms) {
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  LAS_REQUIRE((ld * 2) % 16 == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0 && (long long)atoms * 64 <= ld,
              "TMA atom view needs 16-byte aligned rows of at least %d elements (ld=%lld)", atoms * 64, ld);
  cuuint64_t gdim[3] = {64, (cuuint64_t)rows, (cuuint64_t)atoms};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 2, 128};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, (cuuint32_t)box_atoms};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled (atom view) failed with CUresult %d (rows=%lld atoms=%d ld=%lld)", (int)r, rows, atoms, ld);
  return LAS_OK;
}

// bf16 [B, Tl, Kx] (row pitch Kx, utterance pitch Tl*Kx) seen as {8 k, B, Kx/8, Tl}: one copy of box {8, box_b, Kx/8, 1} lands as
// [Kx/8][box_b][8] -- the no-swizzle K-major UMMA operand layout (core matrices of 8 rows x 16 bytes, 8-row groups 128 bytes apart,
// K-adjacent core matrices box_b*16 bytes apart) -- for the time step given by the last coordinate.  Rows beyond B read as zeros.
int make_tmap_x_core(CUtensorMap* tm, const void* x_bf16, int B, int Tl, int Kx, int box_b) {
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  LAS_REQUIRE(Kx % 8 == 0 && (reinterpret_cast<uintptr_t>(x_bf16) & 15) == 0 && box_b <= 256, "TMA core-matrix view needs K %% 8 == 0 (K=%d)", Kx);
  cuuint64_t gdim[4] = {8, (cuuint64_t)B, (cuuint64_t)(Kx / 8), (cuuint64_t)Tl};
  cuuint64_t gstr[3] = {(cuuint64_t)Tl * Kx * 2, 16, (cuuint64_t)Kx * 2};
  cuuint32_t box[4] = {8, (cuuint32_t)box_b, (cuuint32_t)(Kx / 8), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x_bf16), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled (core-matrix view) failed with CUresult %d (B=%d Tl=%d K=%d)", (int)r, B, Tl, Kx);
  return LAS_OK;
}

int launch_gemm_bf16_tc(const __nv_bfloat16* A, long long lda, const __nv_bfloat16* W, long long ldw, const float* bias, float* C,
                        long long ldc, int M, int N, int K, bool f16, cudaStream_t st, bool relu) {
  LAS_REQUIRE(M > 0 && N > 0 && K > 0, "bad GEMM shape %dx%dx%d", M, N, K);
  CUtensorMap tm_a, tm_b;
  LAS_TRY(make_tmap_bf16(&tm_a, A, M, K, lda, BM));
  LAS_TRY(make_tmap_bf16(&tm_b, W, N, K, ldw, BN));
  CUtensorMap tm_c;
  memset(&tm_c, 0, sizeof(tm_c));
  const bool ts = tma_store_ok(C, ldc, N, nullptr);
  if (ts) LAS_TRY(make_tmap_f32_store(&tm_c, C, M, N, ldc));
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int grid = tiles < sm_count() ? tiles : sm_count();
  const size_t smem = sizeof(GemmSmem) + 1024;
  // per launch, not cached: the attribute belongs to the current device's context and a host thread may serve several devices
  LAS_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gemm_bf16_tc_kernel<<<grid, GEMM_THREADS, smem, st>>>(tm_a, tm_b, tm_c, bias, C, ldc, M, N, K, relu ? 1 : 0, ts ? 1 : 0, GemmSched{0, 0, 0, f16, nullptr});
  LAS_LAUNCH_OK("gemm_bf16_tc_kernel");
  return LAS_OK;
}

int listener_padded_batch(int B) {
  if (B > 128) return (B + 127) / 128 * 128;
  int bp = 1;
  while (bp < B) bp <<= 1;
  return bp;
}

int launch_gemm_listener(const __nv_bfloat16* A, int B, int Tl, int K, const __nv_bfloat16* W, const float* bias, float* C, int N,
                         uint32_t* flags, int max_ctas, bool f16, cudaStream_t st) {
  LAS_REQUIRE(B > 0 && Tl > 0 && N > 0 && K > 0, "bad listener GEMM shape B=%d Tl=%d N=%d K=%d", B, Tl, N, K);
  const int Bp = listener_padded_batch(B);
  const int M = Tl * Bp;
  EncodeTiledFn enc;
  LAS_TRY(get_encode_fn(&enc));
  LAS_REQUIRE((K * 2) % 16 == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0, "TMA needs 16-byte aligned rows (K=%d)", K);
  // A as {k, b, t}: element (k, b, t) at A + (b*Tl + t)*K + k.  One 128-row tile = {64 k, min(Bp,128) b, 128/Bp t}: rows beyond B
  // (padding) and time steps beyond Tl are out of bounds and read as zeros.
  CUtensorMap tm_a, tm_b;
  {
    cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)B, (cuuint64_t)Tl};
    cuuint64_t gstr[2] = {(cuuint64_t)Tl * K * 2, (cuuint64_t)K * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)(Bp < 128 ? Bp : 128), (cuuint32_t)(Bp < 128 ? 128 / Bp : 1)};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(&tm_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(A), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(LAS_ECUDA, "cuTensorMapEncodeTiled (3-D listener input) failed with CUresult %d (B=%d Tl=%d K=%d)", (int)r, B, Tl, K);
  }
  LAS_TRY(make_tmap_bf16(&tm_b, W, N, K, K, BN));
  CUtensorMap tm_c;
  memset(&tm_c, 0, sizeof(tm_c));
  const bool ts = tma_store_ok(C, N, N, flags);
  if (ts) LAS_TRY(make_tmap_f32_store(&tm_c, C, M, N, N));
  const int n_tiles = (N + BN - 1) / BN;
  const int tiles = ((M + BM - 1) / BM) * n_tiles;
  int grid = tiles < sm_count() ? tiles : sm_count();
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  const size_t smem = sizeof(GemmSmem) + 1024;
  // per launch, not cached: the attribute belongs to the current device's context and a host thread may serve several devices
  LAS_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // forward-direction columns are the first half of N; when the halves do not fall on tile boundaries every column tile
  // serves both directions and the natural (front-first) order is kept
  const int nfwd = ((N / 2) % BN == 0) ? (N / 2) / BN : n_tiles;
  gemm_bf16_tc_kernel<<<grid, GEMM_THREADS, smem, st>>>(tm_a, tm_b, tm_c, bias, C, (long long)N, M, N, K, 0, ts ? 1 : 0, GemmSched{1, Bp, nfwd, f16, flags});
  LAS_LAUNCH_OK("gemm_bf16_tc_kernel");
  return LAS_OK;
}

// =========================================================================================================
// UMMA probe (test hook): one CTA stages A[M=128,K] and B[N,K] into shared memory with the layout helpers of
// umma.cuh, runs the K/16 tcgen05.mma chain and dumps the TMEM accumulator.  tests/ use it to pin the descriptor
// conventions every other tensor-core kernel here relies on.
// =========================================================================================================
__global__ void __launch_bounds__(128, 1)
umma_probe_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ B, float* __restrict__ D, int N, int K,
                  UmmaLayout la, UmmaLayout lb, uint32_t a_bytes, int variant) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);  // offset from the __shared__ symbol keeps the address space
  uint8_t* sa = base;
  uint8_t* sb = base + a_bytes;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    ptx::mbar_init(&bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 0) ptx::tmem_alloc(&tmem_slot, 256);
  const bool a_tmem = (variant & 2) != 0;  // A operand staged in tensor memory (columns 128..) instead of smem
  if (!a_tmem) {
    for (int i = threadIdx.x; i < 128 * K; i += blockDim.x) {
      const int r = i / K, k = i % K;
      *reinterpret_cast<__nv_bfloat16*>(sa + umma_offset(la, r, k)) = A[i];
    }
  }
  for (int i = threadIdx.x; i < N * K; i += blockDim.x) {
    const int r = i / K, k = i % K;
    *reinterpret_cast<__nv_bfloat16*>(sb + umma_offset(lb, r, k)) = B[i];
  }
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (a_tmem) {
    const int row = warp * 32 + lane;
    for (int k0 = 0; k0 < K; k0 += 16) {
      uint32_t v[8];
      const uint4 q0 = *reinterpret_cast<const uint4*>(A + (size_t)row * K + k0);
      const uint4 q1 = *reinterpret_cast<const uint4*>(A + (size_t)row * K + k0 + 8);
      v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w; v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
      ptx::tmem_st_32x32b_x8(tmem + ((uint32_t)(warp * 32) << 16) + 128 + k0 / 2, v);
    }
    ptx::tmem_st_wait();
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
  }
  if (threadIdx.x == 0) {
    const uint32_t idesc = umma_idesc_bf16(128, N);
    auto swap_fields = [](uint64_t d) {  // hypothesis test: LBO / SBO meanings swapped
      const uint64_t l = (d >> 16) & 0x3FFF, s2 = (d >> 32) & 0x3FFF;
      d &= ~((0x3FFFull << 16) | (0x3FFFull << 32));
      return d | (s2 << 16) | (l << 32);
    };
    for (int k0 = 0; k0 < K; k0 += 16) {
      uint64_t da = umma_smem_desc(la, ptx::smem_u32(sa), k0), db = umma_smem_desc(lb, ptx::smem_u32(sb), k0);
      if (variant & 1) {
        if (!la.sw128) da = swap_fields(da);
        if (!lb.sw128) db = swap_fields(db);
      }
      if (a_tmem) ptx::umma_bf16_ts(tmem, tmem + 128 + k0 / 2, db, idesc, k0 != 0);
      else ptx::umma_bf16(tmem, da, db, idesc, k0 != 0);
    }
    ptx::umma_commit(&bar);
  }
  ptx::mbar_wait(&bar, 0);
  ptx::tc_fence_after();
  const int row = warp * 32 + lane;
  for (int c0 = 0; c0 < N; c0 += 8) {
    uint32_t v[8];
    ptx::tmem_ld_32x32b_x8(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) D[(size_t)row * N + c0 + j] = __uint_as_float(v[j]);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem, 256);
}

int launch_umma_probe(const void* A, const void* B, float* D, int N, int K, int a_sw128, int b_sw128, int variant, cudaStream_t st) {
  LAS_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0, "probe needs N in [16,256], multiple of 16 (N=%d)", N);
  LAS_REQUIRE(K >= 16 && K % 16 == 0 && K <= 256, "probe needs K in [16,256], multiple of 16 (K=%d)", K);
  LAS_REQUIRE(!(a_sw128 || b_sw128) || K % 64 == 0, "SW128 probe needs K %% 64 == 0");
  LAS_REQUIRE(!(variant & 2) || N <= 128, "A-in-TMEM probe needs N <= 128");
  UmmaLayout la, lb;
  if (a_sw128) la = UmmaLayout{1, 0, 1024, 128u * 128u};
  else la = UmmaLayout{0, (128u / 8) * 128u, 128, 0};
  if (b_sw128) lb = UmmaLayout{1, 0, 1024, (uint32_t)N * 128u};
  else lb = UmmaLayout{0, ((uint32_t)N / 8) * 128u, 128, 0};
  const uint32_t a_bytes = 128u * K * 2, b_bytes = (uint32_t)N * K * 2;
  const size_t smem = (size_t)a_bytes + b_bytes + 2048;
  LAS_CUDA_OK(cudaFuncSetAttribute(umma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  umma_probe_kernel<<<1, 128, smem, st>>>(static_cast<const __nv_bfloat16*>(A), static_cast<const __nv_bfloat16*>(B), D, N, K, la, lb,
                                          (a_bytes + 1023) & ~1023u, variant);
  LAS_LAUNCH_OK("umma_probe_kernel");
  return LAS_OK;
}

// fp32 -> 16-bit GEMM operand (bf16 or fp16, round to nearest even), dense
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n, int f16) {
  for (size_t i = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4; i < n; i += (size_t)gridDim.x * blockDim.x * 4) {
    if (i + 3 < n) {
      const float4 v = *reinterpret_cast<const float4*>(src + i);
      *reinterpret_cast<__nv_bfloat162*>(dst + i) = op2_from_f32(v.x, v.y, f16);
      *reinterpret_cast<__nv_bfloat162*>(dst + i + 2) = op2_from_f32(v.z, v.w, f16);
    } else {
      for (size_t j = i; j < n; ++j) dst[j] = op_from_f32(src[j], f16);
    }
  }
}
int launch_f32_to_bf16(const float* src, __nv_bfloat16* dst, size_t n, bool f16, cudaStream_t st) {
  if (n == 0) return LAS_OK;
  LAS_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0, "unaligned cast buffers");
  const size_t blocks = (n / 4 + 255) / 256;
  f32_to_bf16_kernel<<<(unsigned)(blocks < 2368 ? (blocks ? blocks : 1) : 2368), 256, 0, st>>>(src, dst, n, f16);
  LAS_LAUNCH_OK("f32_to_bf16_kernel");
  return LAS_OK;
}

}  // namespace las
