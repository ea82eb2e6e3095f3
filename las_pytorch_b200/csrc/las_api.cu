// extern "C" entry points of include/las_b200.h: argument validation, buffer carving, kernel sequencing.
#include "las_kernels.cuh"
#include "las_fast.cuh"

#include <math.h>
#include <string.h>

namespace las {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

char* err_buf() { return g_err; }
int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void count_launch(int n) { g_launches += n; }

static DebugOptions g_debug;  // written by las_debug_set_option / las_debug_set_trace only
const DebugOptions& debug_options() { return g_debug; }

// tensor-core modes (same kernels; they differ in the 16-bit operand format)
static inline bool tc_mode(int mode) { return mode == LAS_MODE_BF16 || mode == LAS_MODE_F16; }

// ---- profiling registry (thread-local) ------------------------------------------------------------------
struct ProfRec {
  char name[48];
  cudaEvent_t e0, e1;
  int64_t launches0, launches1;
};
static thread_local bool g_prof_on = false;
static thread_local bool g_prof_starts = false;
static thread_local ProfRec g_prof[4096];
static thread_local int g_prof_n = 0;

ProfScope::ProfScope(const char* name, cudaStream_t stream) : st(stream) {
  if (!g_prof_on || g_prof_n >= 4096) return;
  ProfRec& r = g_prof[g_prof_n];
  if (cudaEventCreate(&r.e0) != cudaSuccess || cudaEventCreate(&r.e1) != cudaSuccess) return;
  snprintf(r.name, sizeof(r.name), "%s", name);
  r.launches0 = g_launches;
  cudaEventRecord(r.e0, st);
  slot = g_prof_n++;
}
ProfScope::~ProfScope() {
  if (slot < 0) return;
  g_prof[slot].launches1 = g_launches;
  cudaEventRecord(g_prof[slot].e1, st);
}

int sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 148;
  return n;
}

static int device_ok() {
  int dev = 0, major = 0;
  LAS_CUDA_OK(cudaGetDevice(&dev));
  LAS_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10)
    return fail(LAS_EDEVICE, "device %d has compute capability %d.x; this library is built for sm_100a only (no fallback)",
                dev, major);
  return LAS_OK;
}

__global__ void bias_sum_kernel(float* out, const float* a, const float* b, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}

// ---------------------------------------------------------------------------------------------------------
// Listener, fp32 mode.  Packed layout per layer: Wcat [8H, K] (fwd rows then reverse rows), bias [8H]
// (= b_ih + b_hh), Whh [2][4H, H].
// ---------------------------------------------------------------------------------------------------------
struct ListenerPackF32 {
  float* wcat[16];
  float* bias[16];
  float* whh[16];
  float* bhh[16];  // GRU / RNN: b_hh kept apart from the input projection's bias (the GRU's n gate needs it inside r * (...))
  size_t bytes;
};
static inline int n_gates(int cell) { return cell == LAS_CELL_LSTM ? 4 : (cell == LAS_CELL_GRU ? 3 : 1); }
static int listener_check(const las_listener_dims* d) {
  LAS_REQUIRE(d != nullptr, "dims is NULL");
  LAS_REQUIRE(d->cell >= LAS_CELL_LSTM && d->cell <= LAS_CELL_RNN, "unknown recurrent cell %d", d->cell);
  LAS_REQUIRE(d->B > 0 && d->T > 0 && d->F > 0 && d->H > 0, "listener dims must be positive (B=%d T=%d F=%d H=%d)", d->B, d->T, d->F, d->H);
  LAS_REQUIRE(d->L >= 1 && d->L <= 16, "Listener should have at least 1 layer (L=%d)", d->L);
  LAS_REQUIRE(d->T % (1 << d->L) == 0,
              "timestep %d is not divisible by 2^%d: the pyramid fold (model/las_model.py:86-87) needs an even length at every layer",
              d->T, d->L);
  return LAS_OK;
}
static ListenerPackF32 listener_pack_layout_f32(const las_listener_dims* d, void* base) {
  ListenerPackF32 p;
  Carver cv(base);
  for (int l = 0; l < d->L; ++l) {
    const size_t K = (l == 0) ? 2 * (size_t)d->F : 4 * (size_t)d->H;
    const size_t GH2 = 2 * (size_t)n_gates(d->cell) * d->H;  // both directions' gate rows
    p.wcat[l] = cv.take<float>(GH2 * K);
    p.bias[l] = cv.take<float>(GH2);
    p.whh[l] = cv.take<float>(GH2 * d->H);
    p.bhh[l] = cv.take<float>(GH2);
  }
  p.bytes = cv.total();
  return p;
}

struct ListenerWsF32 {
  float* P;
  float* act[2];
  float* c;
  int32_t* len;  // [L][B] valid steps per layer (length-mask extension)
  size_t bytes;
};
static ListenerWsF32 listener_ws_layout_f32(const las_listener_dims* d, void* base) {
  ListenerWsF32 w;
  Carver cv(base);
  const size_t M0 = (size_t)d->B * (d->T / 2);
  w.P = cv.take<float>(M0 * 2 * n_gates(d->cell) * d->H);
  w.act[0] = cv.take<float>(M0 * 2 * d->H);
  w.act[1] = cv.take<float>(M0 / 2 * 2 * d->H + 16);
  w.c = cv.take<float>(2 * (size_t)d->B * d->H);
  w.len = cv.take<int32_t>((size_t)d->L * d->B);
  w.bytes = cv.total();
  return w;
}

// LAS_MODE_BF16 for GRU / RNN cells and hidden sizes the cluster-resident recurrence does not cover: the input projection (the one
// dense contraction of a layer) runs as a tcgen05 GEMM over bf16 copies of the layer input and of W_ih, the recurrence on the fp32
// cell kernel.  The bf16 weights follow the fp32 pack, the bf16 activations the fp32 workspace.
struct ListenerGen {
  __nv_bfloat16* w[16];  // pack: [2*G*H, K] per layer;  workspace: w[0] = bf16 copy of the current layer's input
  size_t bytes;
};
static bool listener_gen_ok(const las_listener_dims* d) { return (2 * d->F) % 8 == 0 && (4 * d->H) % 8 == 0; }
static ListenerGen listener_pack_layout_gen(const las_listener_dims* d, void* base) {
  ListenerGen p;
  Carver cv(base);
  for (int l = 0; l < d->L; ++l) {
    const size_t K = (l == 0) ? 2 * (size_t)d->F : 4 * (size_t)d->H;
    p.w[l] = cv.take<__nv_bfloat16>(2 * (size_t)n_gates(d->cell) * d->H * K);
  }
  p.bytes = cv.total();
  return p;
}
static ListenerGen listener_ws_layout_gen(const las_listener_dims* d, void* base) {
  ListenerGen p;
  Carver cv(base);
  const size_t n0 = (size_t)d->B * d->T * d->F, n1 = (size_t)d->B * (d->T / 2) * 2 * d->H;
  p.w[0] = cv.take<__nv_bfloat16>(n0 > n1 ? n0 : n1);
  p.bytes = cv.total();
  return p;
}

// The kernels that run a model, and with them the layout of its pack and workspace
enum class Path {
  F32,   // fp32 kernels on the fp32 layouts
  GEN,   // tensor-core modes, generic path: the fp32 layouts, and the generic (16-bit) layouts behind them
  FAST,  // tensor-core modes: the persistent decoder / the cluster-resident recurrence (fast_*.cu), which own their blocks' layouts
};
static void* behind(const void* base, size_t offset) { return base ? static_cast<char*>(const_cast<void*>(base)) + offset : nullptr; }

// The one place that decides the listener's path and its 16-bit operand format, and knows where its blocks sit: the fp32 layouts at
// the start of the pack and the workspace, the generic ones behind them; or the cluster-resident recurrence's own layouts, which then
// fill both buffers.  Null bases give the sizes alone.  `d` has passed listener_check.
struct ListenerLayout {
  Path path;
  bool f16;            // GEN, FAST: IEEE fp16 operands (LAS_MODE_F16), else bf16
  ListenerPackF32 pk;  // F32, GEN
  ListenerWsF32 ws;
  ListenerGen gp, gw;  // GEN
  size_t pack_bytes, ws_bytes;
};
static ListenerLayout listener_layout(const las_listener_dims* d, int mode, const void* packed, void* ws) {
  ListenerLayout L = {};
  L.path = !tc_mode(mode) ? Path::F32 : fast_listener_fits(d) ? Path::FAST : Path::GEN;
  L.f16 = mode == LAS_MODE_F16;
  if (L.path == Path::FAST) {
    L.pack_bytes = fast_listener_packed_bytes(d);
    L.ws_bytes = fast_listener_workspace_bytes(d);
    return L;
  }
  L.pk = listener_pack_layout_f32(d, const_cast<void*>(packed));
  L.ws = listener_ws_layout_f32(d, ws);
  L.pack_bytes = L.pk.bytes;
  L.ws_bytes = L.ws.bytes;
  if (L.path == Path::GEN) {
    L.gp = listener_pack_layout_gen(d, behind(packed, L.pk.bytes));
    L.gw = listener_ws_layout_gen(d, behind(ws, L.ws.bytes));
    L.pack_bytes += L.gp.bytes;
    L.ws_bytes += L.gw.bytes;
  }
  return L;
}

static int listener_forward_f32(const float* x, const int32_t* x_lengths, const las_listener_dims* d, const ListenerLayout& L, float* enc,
                                int32_t* enc_lengths, cudaStream_t st) {
  const ListenerPackF32& pk = L.pk;
  const ListenerWsF32& w = L.ws;
  const ListenerGen &gp = L.gp, &gw = L.gw;
  const bool gen = L.path == Path::GEN;
  const int B = d->B, H = d->H;
  const int GH = n_gates(d->cell) * H;
  const bool lstm = d->cell == LAS_CELL_LSTM;
  const float* cur = x;
  int Tin = d->T, Fin = d->F;
  for (int l = 0; l < d->L; ++l) {
    const int Tl = Tin / 2, K = 2 * Fin, M = B * Tl;
    const int32_t* len_l = nullptr;
    if (x_lengths) {
      LAS_TRY(launch_pyramid_lengths(l == 0 ? x_lengths : w.len + (size_t)(l - 1) * B, w.len + (size_t)l * B, B, Tl, st));
      len_l = w.len + (size_t)l * B;
    }
    // pyramid fold = reading [B, Tin, Fin] as [B*Tl, 2*Fin]: same memory, lda = 2*Fin (model/las_model.py:86-87)
    char nm[48];
    {
      snprintf(nm, sizeof(nm), "listener.L%d.input_gemm", l);
      ProfScope ps(nm, st);
      if (gen) {
        LAS_TRY(launch_f32_to_bf16(cur, gw.w[0], (size_t)M * K, L.f16, st));
        LAS_TRY(launch_gemm_bf16_tc(gw.w[0], K, gp.w[l], K, pk.bias[l], w.P, 2 * GH, M, 2 * GH, K, L.f16, st));
      } else {
        LAS_TRY(launch_sgemm_nt_bias(cur, K, pk.wcat[l], K, pk.bias[l], w.P, 2 * GH, M, 2 * GH, K, false, st));
      }
    }
    snprintf(nm, sizeof(nm), "listener.L%d.recurrence", l);
    ProfScope ps(nm, st);
    float* out = (l == d->L - 1) ? enc : w.act[l & 1];
    LAS_CUDA_OK(cudaMemsetAsync(w.c, 0, sizeof(float) * 2 * (size_t)B * H, st));
    const long long row_ld = (long long)Tl * 2 * H;
    for (int step = 0; step < Tl; ++step) {
      const int tf = step, tb = Tl - 1 - step;
      CellArgs a[2];
      memset(a, 0, sizeof(a));
      a[0].h_prev = step ? out + (size_t)(tf - 1) * 2 * H : nullptr;
      a[0].h_ld = row_ld;
      a[0].w_hh = pk.whh[l];
      a[0].pre_add = w.P + (size_t)tf * 2 * GH;
      a[0].pre_ld = (long long)Tl * 2 * GH;
      a[0].b_hh = lstm ? nullptr : pk.bhh[l];
      a[0].c = w.c;
      a[0].h_out = out + (size_t)tf * 2 * H;
      a[0].hout_ld = row_ld;
      a[0].lengths = len_l;
      a[0].t = tf;
      a[1].lengths = len_l;
      a[1].t = tb;
      a[1].h_prev = step ? out + (size_t)(tb + 1) * 2 * H + H : nullptr;
      a[1].h_ld = row_ld;
      a[1].w_hh = pk.whh[l] + (size_t)GH * H;
      a[1].pre_add = w.P + (size_t)tb * 2 * GH + GH;
      a[1].pre_ld = (long long)Tl * 2 * GH;
      a[1].b_hh = lstm ? nullptr : pk.bhh[l] + GH;
      a[1].c = w.c + (size_t)B * H;
      a[1].h_out = out + (size_t)tb * 2 * H + H;
      a[1].hout_ld = row_ld;
      LAS_TRY(launch_lstm_cell_f32(a, 2, B, H, st, d->cell));
    }
    cur = out;
    Tin = Tl;
    Fin = 2 * H;
  }
  if (x_lengths && enc_lengths)
    LAS_CUDA_OK(cudaMemcpyAsync(enc_lengths, w.len + (size_t)(d->L - 1) * B, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, st));
  return LAS_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Speller, fp32 mode.  Packed layout = contiguous fp32 copies in the reference's own shapes.
// ---------------------------------------------------------------------------------------------------------
struct SpellerPackF32 {
  float *w_ih[8], *w_hh[8], *b_ih[8], *b_hh[8];
  float *w_phi, *b_phi, *w_psi, *b_psi, *w_cd, *b_cd, *w_dr, *b_dr;
  size_t bytes;
};
static inline int n_heads(const las_speller_dims* d) { return d->heads > 1 ? d->heads : 1; }
static inline int att_dim(const las_speller_dims* d) { return d->no_mlp ? d->Hs : d->D; }  // width of one head's query / of a key
static int speller_check(const las_speller_dims* d) {
  LAS_REQUIRE(d != nullptr, "dims is NULL");
  LAS_REQUIRE(d->B > 0 && d->U > 0 && d->E > 0 && d->Hs > 0 && d->V > 0 && (d->D > 0 || d->no_mlp),
              "speller dims must be positive (B=%d U=%d E=%d Hs=%d V=%d D=%d)", d->B, d->U, d->E, d->Hs, d->V, d->D);
  LAS_REQUIRE(d->heads >= 0 && d->heads <= 16, "multi_head must be in [1,16] (heads=%d)", d->heads);
  LAS_REQUIRE(d->cell >= LAS_CELL_LSTM && d->cell <= LAS_CELL_RNN, "unknown recurrent cell %d", d->cell);
  LAS_REQUIRE(!(d->no_mlp && n_heads(d) > 1), "multi_head > 1 needs use_mlp_in_attention=True (the heads are slices of phi's output)");
  LAS_REQUIRE(d->sl >= 1 && d->sl <= 8, "speller layers must be in [1,8] (sl=%d)", d->sl);
  LAS_REQUIRE(d->Hs == d->E,
              "speller hidden_size (%d) must equal 2*listener_hidden_size (%d): rnn input is [one-hot || encoder feature] "
              "(model/las_model.py:165,198)", d->Hs, d->E);
  return LAS_OK;
}
static SpellerPackF32 speller_pack_layout_f32(const las_speller_dims* d, void* base) {
  SpellerPackF32 p;
  Carver cv(base);
  const size_t G = (size_t)n_gates(d->cell) * d->Hs;
  for (int l = 0; l < d->sl; ++l) {
    const size_t Kx = (l == 0) ? (size_t)d->V + d->E : (size_t)d->Hs;
    p.w_ih[l] = cv.take<float>(G * Kx);
    p.w_hh[l] = cv.take<float>(G * d->Hs);
    p.b_ih[l] = cv.take<float>(G);
    p.b_hh[l] = cv.take<float>(G);
  }
  const size_t Dm = d->no_mlp ? 0 : (size_t)d->D;  // no MLP: no phi / psi parameters exist
  p.w_phi = cv.take<float>(Dm * n_heads(d) * d->Hs);
  p.b_phi = cv.take<float>(Dm * n_heads(d));
  p.w_psi = cv.take<float>(Dm * d->E);
  p.b_psi = cv.take<float>(Dm);
  p.w_cd = cv.take<float>((size_t)d->V * (d->Hs + d->E));
  p.b_cd = cv.take<float>(d->V);
  p.w_dr = cv.take<float>(n_heads(d) > 1 ? (size_t)d->E * d->E * n_heads(d) : 0);
  p.b_dr = cv.take<float>(n_heads(d) > 1 ? (size_t)d->E : 0);
  p.bytes = cv.total();
  return p;
}

struct SpellerWsF32 {
  float* psi;
  float* xin;
  float* h[2];
  float* c;
  int32_t* eos_state;  // <eos> early exit bookkeeping of one launch group (66 int32)
  size_t bytes;
};
static SpellerWsF32 speller_ws_layout_f32(const las_speller_dims* d, void* base) {
  SpellerWsF32 w;
  Carver cv(base);
  w.psi = cv.take<float>((size_t)d->B * d->U * (d->no_mlp ? 0 : d->D));
  w.xin = cv.take<float>((size_t)d->B * (d->V + d->E));
  w.h[0] = cv.take<float>((size_t)d->sl * d->B * d->Hs);
  w.h[1] = cv.take<float>((size_t)d->sl * d->B * d->Hs);
  w.c = cv.take<float>((size_t)d->sl * d->B * d->Hs);
  w.eos_state = cv.take<int32_t>(66);
  w.bytes = cv.total();
  return w;
}

// ---------------------------------------------------------------------------------------------------------
// Speller, LAS_MODE_BF16 beyond what the persistent decoder keeps on chip (1024-wide cells such as the reference's shipped
// config/librispeech-config.yaml:13-34, GRU / RNN cells, multi_head > 1, use_mlp_in_attention=False): the generic tensor-core
// path.  Same step structure as the fp32 mode, but every cell's [x | h_prev] . [W_ih | W_hh]^T is ONE tcgen05 GEMM over bf16
// operands with fp32 accumulation (the weights stream from L2 each step), psi(enc) is a tcgen05 GEMM too, and the cell state,
// the attention and the character distribution stay fp32 -- north_star's "bf16-GEMM / fp32-state" mode, launch per step.
// ---------------------------------------------------------------------------------------------------------
struct GenGeom {
  int R, Kx[8], Kxp[8], Kp[8], Kp_max;
};
static GenGeom gen_geom(const las_speller_dims* d) {
  GenGeom g;
  g.R = (d->cell == LAS_CELL_RNN ? 1 : 4) * d->Hs;
  g.Kp_max = 0;
  for (int l = 0; l < d->sl; ++l) {
    g.Kx[l] = (l == 0) ? d->V + d->E : d->Hs;
    g.Kxp[l] = (g.Kx[l] + 7) & ~7;
    g.Kp[l] = (g.Kxp[l] + d->Hs + 63) & ~63;  // (whole 64-column K blocks: gen_step.cu fetches them by block index)
    if (g.Kp[l] > g.Kp_max) g.Kp_max = g.Kp[l];
  }
  return g;
}
struct SpellerPackGen {
  __nv_bfloat16* w[8];
  float* bias[8];
  __nv_bfloat16* w_psi;
  size_t bytes;
};
static SpellerPackGen speller_pack_layout_gen(const las_speller_dims* d, void* base) {
  SpellerPackGen p;
  const GenGeom g = gen_geom(d);
  Carver cv(base);
  for (int l = 0; l < d->sl; ++l) {
    p.w[l] = cv.take<__nv_bfloat16>((size_t)g.R * g.Kp[l]);
    p.bias[l] = cv.take<float>(g.R);
  }
  p.w_psi = cv.take<__nv_bfloat16>(d->no_mlp ? 0 : (size_t)d->D * d->E);
  p.bytes = cv.total();
  return p;
}
struct SpellerWsGen {
  __nv_bfloat16* a;    // [B, Kp_max] bf16 GEMM operand of the current layer
  float* pre;          // [B, R] gate pre-activations
  __nv_bfloat16* enc;  // [B*U, E] bf16 copy for the psi GEMM
  float* zero;         // [256] zeros: the swapped small-batch GEMM's (unused) per-column bias
  __nv_bfloat16* a2;   // [sl][2][B, Kp_max]: per layer, the operand rows of even / odd steps (fused step, gen_step.cu)
  size_t bytes;
};
static SpellerWsGen speller_ws_layout_gen(const las_speller_dims* d, void* base) {
  SpellerWsGen w;
  const GenGeom g = gen_geom(d);
  Carver cv(base);
  w.a = cv.take<__nv_bfloat16>((size_t)d->B * g.Kp_max);
  w.pre = cv.take<float>((size_t)d->B * g.R);
  w.enc = cv.take<__nv_bfloat16>(d->no_mlp ? 0 : (size_t)d->B * d->U * d->E);
  w.zero = cv.take<float>(256);
  w.a2 = cv.take<__nv_bfloat16>((size_t)d->sl * 2 * d->B * g.Kp_max);
  w.bytes = cv.total();
  return w;
}
// psi GEMM / cell GEMMs read bf16 rows through TMA: 16-byte aligned rows
static bool gen_ok(const las_speller_dims* d) { return d->no_mlp || d->E % 8 == 0; }

// The one place that decides the speller's path and its 16-bit operand format, and knows where its blocks sit: the fp32 layouts at
// the start of the pack and the workspace (in the tensor-core modes too: the persistent decoder reads biases and psi there), then in
// the tensor-core modes the generic layouts or the persistent decoder's blocks.  The beam pack holds the generic layout also where the
// persistent decoder covers the model.  Null bases give the sizes alone.  `d` has passed speller_check.
struct SpellerLayout {
  Path path;
  bool f16;           // GEN, FAST: IEEE fp16 operands (LAS_MODE_F16), else bf16
  SpellerPackF32 pk;
  SpellerWsF32 ws;
  SpellerPackGen gp;  // GEN
  SpellerWsGen gw;
  void* pk_fast;      // FAST
  void* ws_fast;
  size_t pack_bytes, ws_bytes;
};
static SpellerLayout speller_layout(const las_speller_dims* d, int mode, bool beam_pack, const void* packed, void* ws) {
  SpellerLayout L = {};
  L.path = !tc_mode(mode) ? Path::F32 : (!beam_pack && fast_speller_fits(d)) ? Path::FAST : Path::GEN;
  L.f16 = mode == LAS_MODE_F16;
  L.pk = speller_pack_layout_f32(d, const_cast<void*>(packed));
  L.ws = speller_ws_layout_f32(d, ws);
  L.pack_bytes = L.pk.bytes;
  L.ws_bytes = L.ws.bytes;
  if (L.path == Path::GEN) {
    L.gp = speller_pack_layout_gen(d, behind(packed, L.pk.bytes));
    L.gw = speller_ws_layout_gen(d, behind(ws, L.ws.bytes));
    L.pack_bytes += L.gp.bytes;
    L.ws_bytes += L.gw.bytes;
  } else if (L.path == Path::FAST) {
    L.pk_fast = behind(packed, L.pk.bytes);
    L.ws_fast = behind(ws, L.ws.bytes);
    L.pack_bytes += fast_speller_packed_bytes(d);
    L.ws_bytes += fast_speller_workspace_bytes(d);
  }
  return L;
}
static SpellerF32Inputs fast_f32_inputs(const SpellerLayout& L) { return {L.pk.b_phi, L.pk.b_psi, L.pk.b_cd, L.ws.psi}; }

// psi = act(enc . W_psi^T + b_psi) of B utterances into `psi` (generic path: a bf16 copy of enc in `enc16` and a tcgen05 GEMM); without
// the attention MLP the keys are the listener features themselves
static const float* speller_psi(const las_speller_dims* d, int B, const SpellerPackF32& pk, const SpellerPackGen* gp, const float* enc, float* psi,
                                __nv_bfloat16* enc16, int relu, bool f16, cudaStream_t st, int* status) {
  *status = LAS_OK;
  if (d->no_mlp) return enc;  // use_mlp_in_attention=False (model/las_model.py:283-285)
  const int U = d->U, E = d->E, D = d->D;
  ProfScope ps("speller.psi", st);
  if (gp) {
    if ((*status = launch_f32_to_bf16(enc, enc16, (size_t)B * U * E, f16, st)) != LAS_OK) return nullptr;
    *status = launch_gemm_bf16_tc(enc16, E, gp->w_psi, E, pk.b_psi, psi, D, B * U, D, E, f16, st, relu != 0);
  } else {
    *status = launch_sgemm_nt_bias(enc, E, pk.w_psi, E, pk.b_psi, psi, D, B * U, D, E, relu != 0, st);
  }
  return psi;
}

// Which kernels a launch-per-step decoder step runs on `rows` rows (greedy: B, beam: B*K), decided here alone; the one reader of debug keys 12 and 13
struct StepPlan {
  enum Cell { F32, SWAPPED, PLAIN, FUSED } cell;  // lstm_cell_f32 | gen_build_a + GEMM (operands swapped or not) + gen_cell | fused step
  bool cluster_att; int C;                        // attend_cluster_kernel with C CTAs per row, else attend_f32_kernel
};
static StepPlan step_plan(const las_speller_dims* d, int rows, const SpellerLayout& L, bool beam, const float* enc) {
  const DebugOptions& o = debug_options();
  // beam search keeps to the unfused step (DESIGN §4f); small batches swap the GEMM's operands (speller_step)
  const StepPlan::Cell cell = L.path != Path::GEN ? StepPlan::F32 : (!beam && o.gen_fused && rows <= 256) ? StepPlan::FUSED
                              : rows <= 64 ? StepPlan::SWAPPED : StepPlan::PLAIN;
  // The cluster kernel is plain fp32 arithmetic, so the fp32 mode uses it as well.  Multi-head attention keeps the one-CTA kernel, and
  // so do encoders the cluster kernel cannot read (16-byte vector loads of the encoder rows, four features per thread).
  const bool cluster_att = n_heads(d) == 1 && d->E % 4 == 0 && o.gen_fused && (reinterpret_cast<uintptr_t>(enc) & 15) == 0 && d->E <= 4 * AC_THREADS;
  // The step's kernels overlap pairwise (programmatic dependent launch) and each wants an SM to itself: by default the attention keeps
  // to half the chip so that the next step's first cell kernel (<= 64 CTAs) starts on the other half while it runs.
  const int half = sm_count() / 2;
  int C = o.gen_cluster;
  if (C != 1 && C != 2 && C != 4 && C != 8) C = rows * 8 <= half ? 8 : (rows * 4 <= half ? 4 : (rows * 2 <= half ? 2 : 1));
  return {cell, cluster_att, C};
}

// One decoder step of the launch-per-step loop on `rows` decoder rows, with the kernels of `plan` and the attention arguments `t`
struct StepPath {
  const las_speller_dims* d;
  int rows;
  StepPlan plan;
  SpellerPackF32 pk;
  const SpellerPackGen* gp;  // generic tensor-core path, else nullptr (fp32 mode)
  bool f16;                  // generic path: the 16-bit operand format (SpellerLayout::f16)
  GenGeom gg;
  __nv_bfloat16* a;          // generic path: [rows, Kp_max] GEMM operand
  float* pre;                // [rows, R] gate pre-activations
  const float* zero;         // [256] zeros
  float* xin;                // [rows, V+E] layer-0 input: fed-back word | context
  float* c;                  // [sl, rows, Hs]
  const GenStepMaps* maps;   // fused step
  __nv_bfloat16* (*abuf)[2];
};
static AttendArgs speller_attend_args(const StepPath& p, const float* enc, const float* psi, const int32_t* enc_lengths, const float* hn, int relu) {
  const las_speller_dims* d = p.d;
  AttendArgs t;
  memset(&t, 0, sizeof(t));
  t.state = hn + (size_t)(d->sl - 1) * p.rows * d->Hs;
  t.state_ld = d->Hs;
  t.enc = enc;
  t.psi = psi;
  t.w_phi = d->no_mlp ? nullptr : p.pk.w_phi; t.b_phi = p.pk.b_phi; t.w_cd = p.pk.w_cd; t.b_cd = p.pk.b_cd;
  t.enc_lengths = enc_lengths;
  t.B = p.rows; t.U = d->U; t.E = d->E; t.Hs = d->Hs; t.V = d->V; t.D = att_dim(d);
  t.relu = d->no_mlp ? 0 : relu;
  t.heads = n_heads(d); t.w_dr = p.pk.w_dr; t.b_dr = p.pk.b_dr;
  t.ctx_out = p.xin + d->V;
  t.ctx_ld = d->V + d->E;
  t.word_out = p.xin;
  t.word_ld = d->V + d->E;
  return t;
}
static int speller_step(const StepPath& p, int s, const float* hp, float* hn, const AttendArgs& t, cudaStream_t st) {
  const las_speller_dims* d = p.d;
  const int B = p.rows, Hs = d->Hs, sl = d->sl, xld = d->V + d->E;
  const GenGeom& gg = p.gg;
  for (int l = 0; l < sl; ++l) {
    if (p.plan.cell == StepPlan::FUSED) {
      const int q = s & 1;
      LAS_TRY(launch_gen_cell_step(p.maps[l], q, p.gp->bias[l], p.c + (size_t)l * B * Hs, hp + (size_t)l * B * Hs, Hs, hn + (size_t)l * B * Hs, Hs,
                                   p.abuf[l][q ^ 1] + gg.Kxp[l], gg.Kp[l], l + 1 < sl ? p.abuf[l + 1][q] : nullptr, l + 1 < sl ? gg.Kp[l + 1] : 0, B,
                                   Hs, d->cell, gg.Kxp[l], gg.Kp[l], true, p.f16, st, l));
      continue;
    }
    if (p.plan.cell != StepPlan::F32) {
      const float* xin_l = (l == 0) ? p.xin : hn + (size_t)(l - 1) * B * Hs;
      const float* hp_l = hp + (size_t)l * B * Hs;
      LAS_TRY(launch_gen_build_a(xin_l, (l == 0) ? xld : Hs, hp_l, Hs, p.a, B, Hs, gg.Kx[l], gg.Kxp[l], gg.Kp[l], p.f16, st));
      if (p.plan.cell == StepPlan::SWAPPED) {
        // Small batches: the GEMM's 128 x 256 tiles would leave it R/256 CTAs (16 at R = 4096), each streaming 1 MB of weights.  With
        // the operands swapped -- "M" = the R weight rows, "N" = the batch -- R/128 CTAs stream half as much each; the result arrives
        // transposed ([R, B]) and the cell kernel adds the bias.
        LAS_TRY(launch_gemm_bf16_tc(p.gp->w[l], gg.Kp[l], p.a, gg.Kp[l], p.zero, p.pre, B, gg.R, B, gg.Kp[l], p.f16, st));
        LAS_TRY(launch_gen_cell(p.pre, 1, B, p.gp->bias[l], hp_l, Hs, p.c + (size_t)l * B * Hs, hn + (size_t)l * B * Hs, Hs, B, Hs, d->cell, st));
      } else {
        LAS_TRY(launch_gemm_bf16_tc(p.a, gg.Kp[l], p.gp->w[l], gg.Kp[l], p.gp->bias[l], p.pre, gg.R, B, gg.R, gg.Kp[l], p.f16, st));
        LAS_TRY(launch_gen_cell(p.pre, gg.R, 1, nullptr, hp_l, Hs, p.c + (size_t)l * B * Hs, hn + (size_t)l * B * Hs, Hs, B, Hs, d->cell, st));
      }
      continue;
    }
    CellArgs a;
    memset(&a, 0, sizeof(a));
    a.x = (l == 0) ? p.xin : hn + (size_t)(l - 1) * B * Hs;
    a.x_ld = (l == 0) ? xld : Hs;
    a.Kx = (l == 0) ? xld : Hs;
    a.w_ih = p.pk.w_ih[l];
    a.h_prev = hp + (size_t)l * B * Hs;
    a.h_ld = Hs;
    a.w_hh = p.pk.w_hh[l];
    a.b_ih = p.pk.b_ih[l];
    a.b_hh = p.pk.b_hh[l];
    a.c = p.c + (size_t)l * B * Hs;
    a.h_out = hn + (size_t)l * B * Hs;
    a.hout_ld = Hs;
    LAS_TRY(launch_lstm_cell_f32(&a, 1, B, Hs, st, d->cell));
  }
  if (p.plan.cluster_att) return launch_attend_cluster(t, p.plan.C, p.gp != nullptr, st);
  return launch_attend_f32(t, st);
}

static int speller_decode_f32(const las_decode_io* io, const las_speller_dims* d, const SpellerLayout& L, int steps, int decode_mode, int relu,
                              cudaStream_t st) {
  const SpellerPackF32& pk = L.pk;
  const SpellerWsF32& w = L.ws;
  const SpellerPackGen& gp = L.gp;
  const SpellerWsGen& gw = L.gw;
  // the generic tensor-core path of LAS_MODE_BF16 (see above); everything but the GEMMs is shared
  const bool gen = L.path == Path::GEN;
  const GenGeom gg = gen_geom(d);
  if (gen) LAS_CUDA_OK(cudaMemsetAsync(gw.zero, 0, sizeof(float) * 256, st));
  const int B = d->B, Hs = d->Hs, V = d->V, E = d->E, U = d->U, sl = d->sl;
  const int xld = V + E;
  const size_t state_n = (size_t)sl * B * Hs;

  const int NH = n_heads(d);
  const float* psi = io->psi;
  if (d->no_mlp || !psi) {
    int status;
    psi = speller_psi(d, B, pk, gen ? &gp : nullptr, io->enc, w.psi, gw.enc, relu, L.f16, st, &status);
    LAS_TRY(status);
  }
  if (io->word && io->context) {
    LAS_TRY(launch_copy2d(w.xin, xld, io->word, V, B, V, st));
    LAS_TRY(launch_copy2d(w.xin + V, xld, io->context, E, B, E, st));
  } else {
    LAS_TRY(launch_speller_init(w.xin, xld, io->enc, B, U, E, V, st));
  }
  if (io->h_state && (io->c_state || d->cell != LAS_CELL_LSTM)) {
    LAS_CUDA_OK(cudaMemcpyAsync(w.h[0], io->h_state, sizeof(float) * state_n, cudaMemcpyDeviceToDevice, st));
    if (io->c_state) LAS_CUDA_OK(cudaMemcpyAsync(w.c, io->c_state, sizeof(float) * state_n, cudaMemcpyDeviceToDevice, st));
    else LAS_CUDA_OK(cudaMemsetAsync(w.c, 0, sizeof(float) * state_n, st));
  } else {
    LAS_CUDA_OK(cudaMemsetAsync(w.h[0], 0, sizeof(float) * state_n, st));
    LAS_CUDA_OK(cudaMemsetAsync(w.c, 0, sizeof(float) * state_n, st));
  }

  // Fused generic step (gen_step.cu): per layer the 16-bit operand rows [x | h_prev] of even / odd steps live in abuf[l][parity]; the
  // kernels that produce x and h write them there directly.  Step 0's rows are built from the initial state here.
  const StepPlan plan = step_plan(d, B, L, false, io->enc);
  GenStepMaps maps[8];
  __nv_bfloat16* abuf[8][2];
  if (plan.cell == StepPlan::FUSED) {
    LAS_CUDA_OK(cudaMemsetAsync(gw.a2, 0, sizeof(__nv_bfloat16) * (size_t)sl * 2 * B * gg.Kp_max, st));
    for (int l = 0; l < sl; ++l) {
      for (int q = 0; q < 2; ++q) abuf[l][q] = gw.a2 + (size_t)(l * 2 + q) * B * gg.Kp_max;
      LAS_TRY(gen_step_make_maps(&maps[l], gp.w[l], abuf[l][0], abuf[l][1], Hs, d->cell == LAS_CELL_RNN ? 1 : 4, B, gg.Kxp[l], gg.Kp[l]));
      LAS_TRY(launch_gen_build_a(l == 0 ? w.xin : w.h[0], l == 0 ? xld : Hs, w.h[0] + (size_t)l * B * Hs, Hs, abuf[l][0], B, Hs, gg.Kx[l],
                                 gg.Kxp[l], gg.Kp[l], L.f16, st));
    }
  }

  StepPath path;
  path.d = d; path.rows = B; path.plan = plan; path.pk = pk; path.gp = gen ? &gp : nullptr; path.f16 = L.f16; path.gg = gg;
  path.a = gw.a; path.pre = gw.pre; path.zero = gw.zero; path.xin = w.xin; path.c = w.c;
  path.maps = maps; path.abuf = abuf;
  ProfScope ps_steps("speller.steps", st);
  for (int s = 0; s < steps; ++s) {
    float* hp = w.h[s & 1];
    float* hn = w.h[(s & 1) ^ 1];
    AttendArgs t = speller_attend_args(path, io->enc, psi, io->enc_lengths, hn, relu);
    t.score_out = io->attn ? io->attn + (size_t)s * NH * B * U : nullptr;
    t.logp_out = io->logp + (size_t)s * B * V;
    t.token_out = io->tokens ? io->tokens + (size_t)s * B : nullptr;
    if (io->gt_dense) {
      t.gt_dense_step = io->gt_dense + (size_t)s * V;
      t.gt_ld = (long long)io->gt_steps * V;
    } else if (io->gt_index) {
      t.gt_index_step = io->gt_index + s;
      t.gt_index_ld = io->gt_steps;
    }
    t.decode_mode = decode_mode;
    t.sample_seed = io->sample_seed;
    t.step = s;
    if (io->nll_terms) {
      t.nll_term_out = io->nll_terms + (size_t)s * B;
      t.nll_label_step = (io->nll_labels && s < io->nll_steps) ? io->nll_labels + s : nullptr;
      t.nll_label_ld = io->nll_steps;
    }
    if (plan.cell == StepPlan::FUSED) {
      t.op_out = abuf[0][(s & 1) ^ 1];
      t.op_ld = gg.Kp[0];
      t.op_f16 = L.f16;
    }
    LAS_TRY(speller_step(path, s, hp, hn, t, st));
  }
  if (io->h_state && (io->c_state || d->cell != LAS_CELL_LSTM)) {
    LAS_CUDA_OK(cudaMemcpyAsync(io->h_state, w.h[steps & 1], sizeof(float) * state_n, cudaMemcpyDeviceToDevice, st));
    if (io->c_state) LAS_CUDA_OK(cudaMemcpyAsync(io->c_state, w.c, sizeof(float) * state_n, cudaMemcpyDeviceToDevice, st));
  }
  if (io->word && io->context) {
    LAS_TRY(launch_copy2d(io->word, V, w.xin, xld, B, V, st));
    LAS_TRY(launch_copy2d(io->context, E, w.xin + V, xld, B, E, st));
  }
  if (io->early_exit) {
    // The fp32 mode is launch-per-step and gains nothing from stopping early; it reproduces the early-exit OUTPUT contract of
    // las_decode_io (groups of <= 64 utterances, checked every segment, the undecoded tail filled) so that both modes agree.
    const int seg = io->segment_steps > 0 ? (io->segment_steps + 1) & ~1 : 32;
    if (io->steps_done) LAS_CUDA_OK(cudaMemsetAsync(io->steps_done, 0, sizeof(int32_t), st));
    for (int b0 = 0; b0 < B; b0 += 64) {
      const int Bc = B - b0 < 64 ? B - b0 : 64;
      LAS_CUDA_OK(cudaMemsetAsync(w.eos_state, 0, sizeof(int32_t) * 66, st));
      for (int sb = 0; sb < steps; sb += seg)
        LAS_TRY(launch_eos_check(io->tokens, B, b0, Bc, sb, sb + seg < steps ? sb + seg : steps, io->eos_token, w.eos_state, st));
      LAS_TRY(launch_eos_fill(w.eos_state, steps, B, b0, Bc, V, U, NH, io->eos_token, io->logp, io->attn, io->tokens, io->nll_terms,
                              io->steps_done, st));
    }
  }
  return LAS_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Beam search (include/las_b200.h las_beam_io) on the launch-per-step decoder: B*K decoder rows, row b*K + k = hypothesis k of
// utterance b.  The whole recurrent state is xin / h / c in fp32, so beam_step_kernel reorders hypotheses with a row gather.
// ---------------------------------------------------------------------------------------------------------
static int beam_args_check(const las_speller_dims* d, int steps, int beam) {
  LAS_TRY(speller_check(d));
  LAS_REQUIRE(beam >= 1 && beam <= 32, "beam width must be in [1, 32] (beam=%d)", beam);
  LAS_REQUIRE(steps >= 1, "beam search needs steps >= 1 (steps=%d)", steps);
  return LAS_OK;
}
struct BeamWs {
  float* psi;        // [B*U, D] (per utterance)
  float* xin;        // [BK, V+E]
  float* h[2];       // [sl, BK, Hs]
  float* c;          // [sl, BK, Hs]
  float* logp;       // [BK, V] one step's log-probabilities
  float* score;      // [BK]
  int32_t* fin;      // [BK]
  int32_t* parent;   // [S, B, K] back-pointers
  int32_t* token;    // [S, B, K]
  float* token_logp; // [S, B, K]
  // generic tensor-core path
  __nv_bfloat16* a;  // [BK, Kp_max]
  float* pre;        // [BK, R]
  __nv_bfloat16* enc16;  // [B*U, E]
  float* zero;       // [256]
  size_t bytes;
};
static BeamWs beam_ws_layout(const las_speller_dims* d, int steps, int beam, bool gen, void* base) {
  BeamWs w;
  Carver cv(base);
  const size_t B = d->B, BK = B * beam;
  w.psi = cv.take<float>(B * d->U * (d->no_mlp ? 0 : d->D));
  w.xin = cv.take<float>(BK * (d->V + d->E));
  w.h[0] = cv.take<float>((size_t)d->sl * BK * d->Hs);
  w.h[1] = cv.take<float>((size_t)d->sl * BK * d->Hs);
  w.c = cv.take<float>((size_t)d->sl * BK * d->Hs);
  w.logp = cv.take<float>(BK * d->V);
  w.score = cv.take<float>(BK);
  w.fin = cv.take<int32_t>(BK);
  w.parent = cv.take<int32_t>((size_t)steps * BK);
  w.token = cv.take<int32_t>((size_t)steps * BK);
  w.token_logp = cv.take<float>((size_t)steps * BK);
  const GenGeom g = gen_geom(d);
  w.a = cv.take<__nv_bfloat16>(gen ? BK * g.Kp_max : 0);
  w.pre = cv.take<float>(gen ? BK * g.R : 0);
  w.enc16 = cv.take<__nv_bfloat16>(gen && !d->no_mlp ? B * d->U * d->E : 0);
  w.zero = cv.take<float>(gen ? 256 : 0);
  w.bytes = cv.total();
  return w;
}

// `L`: the beam pack's layout
static int speller_beam_f32(const las_beam_io* io, const las_speller_dims* d, const SpellerLayout& L, int steps, int relu, void* ws,
                            cudaStream_t st) {
  const int B = d->B, K = io->beam, BK = B * K, V = d->V, E = d->E, Hs = d->Hs;
  const bool gen = L.path == Path::GEN;
  const SpellerPackF32& pk = L.pk;
  const SpellerPackGen& gp = L.gp;
  const BeamWs w = beam_ws_layout(d, steps, K, gen, ws);
  if (gen) LAS_CUDA_OK(cudaMemsetAsync(w.zero, 0, sizeof(float) * 256, st));

  int status;
  const float* psi = speller_psi(d, B, pk, gen ? &gp : nullptr, io->enc, w.psi, w.enc16, relu, L.f16, st, &status);  // once per utterance
  LAS_TRY(status);
  LAS_TRY(launch_beam_init(w.xin, V + E, io->enc, w.score, w.fin, B, K, d->U, E, V, st));
  const size_t state_n = (size_t)d->sl * BK * Hs;
  LAS_CUDA_OK(cudaMemsetAsync(w.h[0], 0, sizeof(float) * state_n, st));
  LAS_CUDA_OK(cudaMemsetAsync(w.c, 0, sizeof(float) * state_n, st));

  StepPath path = {};
  path.d = d; path.rows = BK; path.plan = step_plan(d, BK, L, true, io->enc); path.pk = pk; path.gp = gen ? &gp : nullptr;
  path.f16 = L.f16; path.gg = gen_geom(d);
  path.a = w.a; path.pre = w.pre; path.zero = w.zero; path.xin = w.xin; path.c = w.c;
  BeamStepArgs ba;
  memset(&ba, 0, sizeof(ba));
  ba.logp = w.logp; ba.score = w.score; ba.fin = w.fin;
  ba.c = d->cell == LAS_CELL_LSTM ? w.c : nullptr;
  ba.xin = w.xin; ba.xld = V + E;
  ba.B = B; ba.K = K; ba.V = V; ba.E = E; ba.Hs = Hs; ba.sl = d->sl; ba.eos = io->eos_token;
  // attention scratch (las_beam_io.attn_work): every row's attention of every step, then the source rows of the n-best paths
  const int NH = n_heads(d), U = d->U;
  float* attn_work = io->attn ? io->attn_work : nullptr;
  int32_t* src_rows = io->attn ? reinterpret_cast<int32_t*>(io->attn_work + (size_t)steps * NH * BK * U) : nullptr;
  // Early exit.  Once every row has ended (a -inf slot counts as ended), each row's only candidate is itself: eos at log-prob 0, score
  // unchanged.  Every merge fills the slots by rank, so the rows are already in (score desc, slot asc) order, which is the merge key
  // of those candidates: every later step keeps every row in its slot and records parent = slot, eos, 0.  Stopping there and padding
  // the tail with eos / 0 (finalize) and zero attention (the trace: its source rows are -1 past every length) therefore gives exactly
  // the outputs of the full run.  The host has to learn the flag to stop issuing steps: one 4-byte copy and a stream synchronisation
  // per check.
  const int seg = io->segment_steps > 0 ? io->segment_steps : 32;
  int steps_run = steps;
  if (io->early_exit) LAS_CUDA_OK(cudaMemsetAsync(io->steps_done, 0, sizeof(int32_t), st));
  ProfScope ps_steps("speller.beam_steps", st);
  for (int s = 0; s < steps; ++s) {
    float* hp = w.h[s & 1];
    float* hn = w.h[(s & 1) ^ 1];
    AttendArgs t = speller_attend_args(path, io->enc, psi, io->enc_lengths, hn, relu);
    t.rows_per_utt = K;
    t.word_out = nullptr;  // beam_step_kernel writes the fed-back words
    t.logp_out = w.logp;
    t.score_out = attn_work ? attn_work + (size_t)s * NH * BK * U : nullptr;  // [heads, B*K, U]: indexed by decoder row
    LAS_TRY(speller_step(path, s, hp, hn, t, st));
    ba.parent = w.parent + (size_t)s * BK;
    ba.token = w.token + (size_t)s * BK;
    ba.token_logp = w.token_logp + (size_t)s * BK;
    ba.h = hn;
    LAS_TRY(launch_beam_step(ba, st));
    if (io->early_exit && (s + 1) % seg == 0 && s + 1 < steps) {
      LAS_TRY(launch_beam_all_ended(w.fin, BK, s + 1, io->steps_done, st));
      int32_t ended = 0;
      LAS_CUDA_OK(cudaMemcpyAsync(&ended, io->steps_done, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      LAS_CUDA_OK(cudaStreamSynchronize(st));
      if (ended) {
        steps_run = s + 1;
        break;
      }
    }
  }
  if (io->early_exit && steps_run == steps) LAS_CUDA_OK(cudaMemcpyAsync(io->steps_done, &steps, sizeof(int32_t), cudaMemcpyHostToDevice, st));
  BeamFinalArgs fa;
  memset(&fa, 0, sizeof(fa));
  fa.score = w.score; fa.parent = w.parent; fa.token = w.token; fa.token_logp = w.token_logp;
  fa.tokens_out = io->tokens; fa.token_logp_out = io->token_logp; fa.lengths_out = io->lengths; fa.scores_out = io->scores;
  fa.src_rows = src_rows;
  fa.B = B; fa.K = K; fa.N = io->nbest; fa.S_run = steps_run; fa.S_out = steps; fa.eos = io->eos_token; fa.alpha = io->length_penalty;
  LAS_TRY(launch_beam_finalize(fa, st));
  if (io->attn) LAS_TRY(launch_beam_attention_trace(attn_work, src_rows, io->attn, B, K, io->nbest, steps, NH, U, st));
  return LAS_OK;
}

// The las_decode_io checks of las_speller_decode, which las_pipeline_step's concurrent branch makes as well.  `d` has passed
// speller_check.
static int decode_args_check(const las_decode_io* io, const las_speller_dims* d, int steps, int decode_mode, int mode, size_t ws_bytes) {
  LAS_REQUIRE(io->enc && io->logp, "io->enc and io->logp are required");
  LAS_REQUIRE(steps >= 0, "steps must be >= 0");
  LAS_REQUIRE(mode == LAS_MODE_FP32 || tc_mode(mode), "unknown mode %d", mode);
  LAS_REQUIRE(decode_mode == LAS_DECODE_RAW || decode_mode == LAS_DECODE_GREEDY || decode_mode == LAS_DECODE_SAMPLE,
              "decode_mode %d is not supported (0 = raw, 1 = greedy, 2 = sample)", decode_mode);
  LAS_REQUIRE(!(io->gt_dense || io->gt_index) || io->gt_steps >= steps, "ground truth has %d steps, %d requested", io->gt_steps, steps);
  LAS_REQUIRE(d->cell != LAS_CELL_LSTM || (io->h_state == nullptr) == (io->c_state == nullptr), "h_state and c_state must be given together");
  LAS_REQUIRE((io->word == nullptr) == (io->context == nullptr), "word and context must be given together");
  LAS_REQUIRE(!io->early_exit || io->tokens, "<eos> early exit needs io->tokens");
  LAS_TRY(device_ok());
  const size_t need = speller_layout(d, mode, false, nullptr, nullptr).ws_bytes;
  if (ws_bytes < need) return fail(LAS_ENOMEM, "workspace too small: %zu < %zu", ws_bytes, need);
  return LAS_OK;
}

// Can las_pipeline_step run the listener next to the persistent decoder (fast_pipeline.cu)?  Both models valid, both on their FAST paths.
static bool pipeline_fast(const las_listener_dims* ld, const las_speller_dims* sd, int mode) {
  return ld && sd && listener_check(ld) == LAS_OK && speller_check(sd) == LAS_OK && listener_layout(ld, mode, nullptr, nullptr).path == Path::FAST &&
         speller_layout(sd, mode, false, nullptr, nullptr).path == Path::FAST;
}

}  // namespace las

using namespace las;

extern "C" {

int las_abi_version(void) { return LAS_B200_ABI_VERSION; }
const char* las_last_error(void) { return err_buf(); }
int las_device_check(void) { return device_ok(); }
int las_mode_available(int mode) { return mode == LAS_MODE_FP32 || tc_mode(mode); }
int las_prof_enable(int on) {
  for (int i = 0; i < g_prof_n; ++i) {
    cudaEventDestroy(g_prof[i].e0);
    cudaEventDestroy(g_prof[i].e1);
  }
  g_prof_n = 0;
  g_prof_on = on != 0;
  g_prof_starts = on == 2;
  return LAS_OK;
}
int las_prof_report(char* buf, size_t buf_bytes) {
  LAS_REQUIRE(buf && buf_bytes > 0, "null buffer");
  size_t off = 0;
  buf[0] = 0;
  for (int i = 0; i < g_prof_n; ++i) {
    float ms = 0.f;
    LAS_CUDA_OK(cudaEventSynchronize(g_prof[i].e1));
    LAS_CUDA_OK(cudaEventElapsedTime(&ms, g_prof[i].e0, g_prof[i].e1));
    int n;
    if (g_prof_starts) {  // las_prof_enable(2): name@start-offset (ms since the first recorded group) instead of the bare name
      float t0 = 0.f;
      cudaEventElapsedTime(&t0, g_prof[0].e0, g_prof[i].e0);
      n = snprintf(buf + off, buf_bytes - off, "%s@%.3f %.6f %lld\n", g_prof[i].name, t0, ms, (long long)(g_prof[i].launches1 - g_prof[i].launches0));
    } else {
      n = snprintf(buf + off, buf_bytes - off, "%s %.6f %lld\n", g_prof[i].name, ms, (long long)(g_prof[i].launches1 - g_prof[i].launches0));
    }
    if (n < 0 || (size_t)n >= buf_bytes - off) return fail(LAS_ENOMEM, "report buffer too small");
    off += n;
  }
  return LAS_OK;
}
int64_t las_launch_count(int reset) {
  const int64_t v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

// ---- listener ------------------------------------------------------------------------------------------
size_t las_listener_packed_bytes(const las_listener_dims* d, int mode) {
  if (listener_check(d) != LAS_OK) return 0;
  return listener_layout(d, mode, nullptr, nullptr).pack_bytes;
}

int las_listener_pack(const las_lstm_weights* w, const las_listener_dims* d, int mode, void* packed, size_t packed_bytes,
                      void* stream) {
  LAS_TRY(listener_check(d));
  LAS_REQUIRE(w && packed, "null weights / packed buffer");
  LAS_REQUIRE(mode == LAS_MODE_FP32 || tc_mode(mode), "unknown mode %d", mode);
  LAS_TRY(device_ok());
  const ListenerLayout L = listener_layout(d, mode, packed, nullptr);
  if (packed_bytes < L.pack_bytes) return fail(LAS_ENOMEM, "packed buffer too small: %zu < %zu", packed_bytes, L.pack_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAS_REQUIRE(L.path != Path::GEN || listener_gen_ok(d),
              "LAS_MODE_BF16 needs 16-byte aligned bf16 rows for TMA: 2F (%d) and 4H (%d) must be multiples of 8; use LAS_MODE_FP32", 2 * d->F, 4 * d->H);
  if (L.path == Path::FAST) return fast_listener_pack(w, d, packed, L.f16, st);
  const ListenerPackF32& pk = L.pk;
  const size_t H = d->H, GH = (size_t)n_gates(d->cell) * H;
  for (int l = 0; l < d->L; ++l) {
    const size_t K = (l == 0) ? 2 * (size_t)d->F : 4 * H;
    for (int dir = 0; dir < 2; ++dir) {
      const las_lstm_weights& s = w[2 * l + dir];
      LAS_REQUIRE(s.w_ih && s.w_hh && s.b_ih && s.b_hh, "null weight pointer in layer %d dir %d", l, dir);
      LAS_CUDA_OK(cudaMemcpyAsync(pk.wcat[l] + dir * GH * K, s.w_ih, sizeof(float) * GH * K, cudaMemcpyDeviceToDevice, st));
      LAS_CUDA_OK(cudaMemcpyAsync(pk.whh[l] + dir * GH * H, s.w_hh, sizeof(float) * GH * H, cudaMemcpyDeviceToDevice, st));
      LAS_CUDA_OK(cudaMemcpyAsync(pk.bhh[l] + dir * GH, s.b_hh, sizeof(float) * GH, cudaMemcpyDeviceToDevice, st));
      if (d->cell == LAS_CELL_LSTM) {  // both biases fold into the input projection
        bias_sum_kernel<<<(unsigned)((GH + 255) / 256), 256, 0, st>>>(pk.bias[l] + dir * GH, s.b_ih, s.b_hh, (int)GH);
        LAS_LAUNCH_OK("bias_sum_kernel");
      } else {  // GRU / RNN: the projection carries b_ih only, the cell kernel adds b_hh on the recurrent side
        LAS_CUDA_OK(cudaMemcpyAsync(pk.bias[l] + dir * GH, s.b_ih, sizeof(float) * GH, cudaMemcpyDeviceToDevice, st));
      }
    }
  }
  if (L.path == Path::GEN) {  // bf16 copies of [W_ih fwd ; W_ih reverse]
    for (int l = 0; l < d->L; ++l) {
      const size_t K = (l == 0) ? 2 * (size_t)d->F : 4 * H;
      LAS_TRY(launch_f32_to_bf16(pk.wcat[l], L.gp.w[l], 2 * GH * K, L.f16, st));
    }
  }
  return LAS_OK;
}

size_t las_listener_workspace_bytes(const las_listener_dims* d, int mode) {
  if (listener_check(d) != LAS_OK) return 0;
  return listener_layout(d, mode, nullptr, nullptr).ws_bytes;
}

int las_listener_forward(const float* x, const void* packed, const las_listener_dims* d, int mode, float* enc,
                         void* workspace, size_t workspace_bytes, void* stream) {
  return las_listener_forward_masked(x, nullptr, packed, d, mode, enc, nullptr, workspace, workspace_bytes, stream);
}

int las_listener_forward_masked(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d,
                                int mode, float* enc, int32_t* enc_lengths, void* workspace, size_t workspace_bytes,
                                void* stream) {
  LAS_TRY(listener_check(d));
  LAS_REQUIRE(x && packed && enc && workspace, "null pointer argument");
  LAS_REQUIRE(mode == LAS_MODE_FP32 || tc_mode(mode), "unknown mode %d", mode);
  LAS_TRY(device_ok());
  const ListenerLayout L = listener_layout(d, mode, packed, workspace);
  if (workspace_bytes < L.ws_bytes) return fail(LAS_ENOMEM, "workspace too small: %zu < %zu", workspace_bytes, L.ws_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (L.path == Path::FAST) return fast_listener_forward(x, x_lengths, packed, d, enc, enc_lengths, workspace, L.f16, st);
  LAS_REQUIRE(L.path != Path::GEN || listener_gen_ok(d), "LAS_MODE_BF16 needs 2F (%d) and 4H (%d) to be multiples of 8; use LAS_MODE_FP32",
              2 * d->F, 4 * d->H);
  return listener_forward_f32(x, x_lengths, d, L, enc, enc_lengths, st);
}

// ---- speller -------------------------------------------------------------------------------------------
size_t las_speller_packed_bytes(const las_speller_dims* d, int mode) {
  if (speller_check(d) != LAS_OK) return 0;
  return speller_layout(d, mode, false, nullptr, nullptr).pack_bytes;
}

static int speller_pack(const las_speller_weights* w, const las_speller_dims* d, int mode, void* packed, size_t packed_bytes, void* stream,
                        bool beam_pack) {
  LAS_TRY(speller_check(d));
  LAS_REQUIRE(w && packed && w->rnn_host, "null weights / packed buffer");
  LAS_REQUIRE(mode == LAS_MODE_FP32 || tc_mode(mode), "unknown mode %d", mode);
  LAS_REQUIRE(w->w_cd && w->b_cd, "null output weight pointer");
  LAS_REQUIRE(d->no_mlp || (w->w_phi && w->b_phi && w->w_psi && w->b_psi), "null attention weight pointer");
  LAS_REQUIRE(n_heads(d) == 1 || (w->w_dr && w->b_dr), "multi_head > 1 needs attention.dim_reduce weights");
  const SpellerLayout L = speller_layout(d, mode, beam_pack, packed, nullptr);
  LAS_REQUIRE(L.path != Path::GEN || gen_ok(d), "LAS_MODE_BF16 needs E %% 8 == 0 for the psi GEMM's TMA rows (E=%d); use LAS_MODE_FP32", d->E);
  LAS_TRY(device_ok());
  if (packed_bytes < L.pack_bytes) return fail(LAS_ENOMEM, "packed buffer too small: %zu < %zu", packed_bytes, L.pack_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SpellerPackF32& pk = L.pk;
  const size_t G = (size_t)n_gates(d->cell) * d->Hs;
#define CP(dst, src, n) LAS_CUDA_OK(cudaMemcpyAsync(dst, src, sizeof(float) * (n), cudaMemcpyDeviceToDevice, st))
  for (int l = 0; l < d->sl; ++l) {
    const las_lstm_weights& s = w->rnn_host[l];
    LAS_REQUIRE(s.w_ih && s.w_hh && s.b_ih && s.b_hh, "null weight pointer in speller layer %d", l);
    const size_t Kx = (l == 0) ? (size_t)d->V + d->E : (size_t)d->Hs;
    CP(pk.w_ih[l], s.w_ih, G * Kx);
    CP(pk.w_hh[l], s.w_hh, G * d->Hs);
    CP(pk.b_ih[l], s.b_ih, G);
    CP(pk.b_hh[l], s.b_hh, G);
  }
  if (!d->no_mlp) {
    CP(pk.w_phi, w->w_phi, (size_t)d->D * n_heads(d) * d->Hs);
    CP(pk.b_phi, w->b_phi, (size_t)d->D * n_heads(d));
    CP(pk.w_psi, w->w_psi, (size_t)d->D * d->E);
    CP(pk.b_psi, w->b_psi, d->D);
  }
  CP(pk.w_cd, w->w_cd, (size_t)d->V * (d->Hs + d->E));
  CP(pk.b_cd, w->b_cd, d->V);
  if (n_heads(d) > 1) {
    CP(pk.w_dr, w->w_dr, (size_t)d->E * d->E * n_heads(d));
    CP(pk.b_dr, w->b_dr, d->E);
  }
#undef CP
  if (L.path == Path::FAST) return fast_speller_pack(w, d, L.pk_fast, L.f16, st);
  if (L.path == Path::GEN) {  // generic tensor-core path: [W_ih | W_hh] per layer as one bf16 matrix, psi weights in bf16
    const SpellerPackGen& gp = L.gp;
    const GenGeom g = gen_geom(d);
    for (int l = 0; l < d->sl; ++l) {
      const las_lstm_weights& s = w->rnn_host[l];
      LAS_TRY(launch_gen_pack_w(s.w_ih, s.w_hh, s.b_ih, s.b_hh, gp.w[l], gp.bias[l], d->cell, d->Hs, g.Kx[l], g.Kxp[l], g.Kp[l], L.f16, st));
    }
    if (!d->no_mlp) LAS_TRY(launch_f32_to_bf16(w->w_psi, gp.w_psi, (size_t)d->D * d->E, L.f16, st));
  }
  return LAS_OK;
}

int las_speller_pack(const las_speller_weights* w, const las_speller_dims* d, int mode, void* packed, size_t packed_bytes,
                     void* stream) {
  return speller_pack(w, d, mode, packed, packed_bytes, stream, false);
}

int las_psi_precompute(const float* enc, const float* w_psi, const float* b_psi, int B, int U, int E, int D, int relu,
                       float* psi, void* stream) {
  LAS_REQUIRE(enc && w_psi && b_psi && psi, "null pointer argument");
  LAS_REQUIRE(B > 0 && U > 0 && E > 0 && D > 0, "bad dims (B=%d U=%d E=%d D=%d)", B, U, E, D);
  LAS_TRY(device_ok());
  return launch_sgemm_nt_bias(enc, E, w_psi, E, b_psi, psi, D, B * U, D, E, relu != 0, static_cast<cudaStream_t>(stream));
}

int las_attention_forward(const float* state, const float* enc, const float* psi, const float* w_phi, const float* b_phi,
                          int B, int U, int E, int Hs, int D, int relu, int heads, const float* w_dr, const float* b_dr,
                          const int32_t* enc_lengths, float* score, float* context, void* stream) {
  LAS_REQUIRE(state && enc && psi && context, "null pointer argument");
  LAS_REQUIRE(B > 0 && U > 0 && E > 0 && Hs > 0 && D > 0, "bad dims (B=%d U=%d E=%d Hs=%d D=%d)", B, U, E, Hs, D);
  LAS_REQUIRE(w_phi ? (b_phi != nullptr) : (D == Hs), "without phi the query is the decoder state itself: D (%d) must equal Hs (%d)", D, Hs);
  if (heads < 1) heads = 1;
  LAS_REQUIRE(heads == 1 || (w_phi && w_dr && b_dr), "multi_head > 1 needs phi and dim_reduce weights");
  LAS_TRY(device_ok());
  AttendArgs t;
  memset(&t, 0, sizeof(t));
  t.state = state; t.state_ld = Hs;
  t.enc = enc; t.psi = psi;
  t.w_phi = w_phi; t.b_phi = b_phi;
  t.enc_lengths = enc_lengths;
  t.B = B; t.U = U; t.E = E; t.Hs = Hs; t.V = 0; t.D = D;
  t.relu = relu;
  t.heads = heads; t.w_dr = w_dr; t.b_dr = b_dr;
  t.score_out = score;
  t.ctx_out = context; t.ctx_ld = E;
  return launch_attend_f32(t, static_cast<cudaStream_t>(stream));
}

size_t las_speller_workspace_bytes(const las_speller_dims* d, int steps, int mode) {
  if (speller_check(d) != LAS_OK || steps < 0) return 0;
  return speller_layout(d, mode, false, nullptr, nullptr).ws_bytes;
}

int las_speller_decode(const las_decode_io* io, const void* packed, const las_speller_dims* d, int steps, int decode_mode,
                       int mode, int relu, void* workspace, size_t workspace_bytes, void* stream) {
  LAS_TRY(speller_check(d));
  LAS_REQUIRE(io && packed && workspace, "null pointer argument");
  LAS_TRY(decode_args_check(io, d, steps, decode_mode, mode, workspace_bytes));
  if (steps == 0) return LAS_OK;
  const SpellerLayout L = speller_layout(d, mode, false, packed, workspace);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (L.path == Path::FAST) return fast_speller_decode(io, fast_f32_inputs(L), L.pk_fast, d, steps, decode_mode, relu, L.ws_fast, L.f16, st);
  LAS_REQUIRE(L.path != Path::GEN || gen_ok(d), "LAS_MODE_BF16 needs E %% 8 == 0 (E=%d); use LAS_MODE_FP32", d->E);
  return speller_decode_f32(io, d, L, steps, decode_mode, relu, st);
}

// ---- beam search -----------------------------------------------------------------------------------------
size_t las_speller_beam_packed_bytes(const las_speller_dims* d, int mode) {
  if (speller_check(d) != LAS_OK) return 0;
  if (mode != LAS_MODE_FP32 && !tc_mode(mode)) return 0;
  return speller_layout(d, mode, true, nullptr, nullptr).pack_bytes;
}

int las_speller_beam_pack(const las_speller_weights* w, const las_speller_dims* d, int mode, void* packed, size_t bytes, void* stream) {
  return speller_pack(w, d, mode, packed, bytes, stream, true);
}

size_t las_speller_beam_workspace_bytes(const las_speller_dims* d, int steps, int beam, int mode) {
  if (beam_args_check(d, steps, beam) != LAS_OK) return 0;
  if (mode != LAS_MODE_FP32 && !tc_mode(mode)) return 0;
  return beam_ws_layout(d, steps, beam, speller_layout(d, mode, true, nullptr, nullptr).path == Path::GEN, nullptr).bytes;
}

int las_speller_beam_search(const las_beam_io* io, const void* packed, const las_speller_dims* d, int steps, int mode, int relu,
                            void* workspace, size_t workspace_bytes, void* stream) {
  LAS_REQUIRE(io && packed && workspace, "null pointer argument");
  LAS_TRY(beam_args_check(d, steps, io->beam));
  LAS_REQUIRE(io->enc && io->tokens && io->lengths && io->scores, "io->enc, io->tokens, io->lengths and io->scores are required");
  LAS_REQUIRE(io->nbest >= 1 && io->nbest <= io->beam, "nbest must be in [1, beam] (nbest=%d beam=%d)", io->nbest, io->beam);
  LAS_REQUIRE(io->eos_token >= 0 && io->eos_token < d->V, "eos_token %d is not in [0, V=%d)", io->eos_token, d->V);
  LAS_REQUIRE(isfinite(io->length_penalty) && io->length_penalty >= 0.f, "length_penalty must be finite and >= 0 (%g)", (double)io->length_penalty);
  LAS_REQUIRE(mode == LAS_MODE_FP32 || tc_mode(mode), "unknown mode %d", mode);
  LAS_REQUIRE(!tc_mode(mode) || gen_ok(d), "LAS_MODE_BF16 beam search needs E %% 8 == 0 (E=%d); use LAS_MODE_FP32", d->E);
  LAS_REQUIRE(!io->attn || io->attn_work, "io->attn needs io->attn_work");
  LAS_REQUIRE(!io->early_exit || io->steps_done, "io->early_exit needs io->steps_done");
  LAS_REQUIRE(io->segment_steps >= 0, "segment_steps must be >= 0 (%d)", io->segment_steps);
  LAS_TRY(device_ok());
  if (io->early_exit) {
    // early exit waits on the stream for its flag, which a stream being captured into a graph cannot do
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    LAS_CUDA_OK(cudaStreamIsCapturing(static_cast<cudaStream_t>(stream), &cs));
    LAS_REQUIRE(cs == cudaStreamCaptureStatusNone, "io->early_exit synchronises with the host and cannot run on a capturing stream");
  }
  const size_t need = las_speller_beam_workspace_bytes(d, steps, io->beam, mode);
  if (workspace_bytes < need) return fail(LAS_ENOMEM, "workspace too small: %zu < %zu", workspace_bytes, need);
  return speller_beam_f32(io, d, speller_layout(d, mode, true, packed, nullptr), steps, relu, workspace, static_cast<cudaStream_t>(stream));
}

int las_pipeline_step(const las_pipeline_args* a, int mode, void* stream) {
  LAS_REQUIRE(a, "null pointer argument");
  const bool dec = a->dec_io != nullptr, lis = a->x != nullptr;
  LAS_REQUIRE(dec || lis, "nothing to do: neither a batch to decode nor a batch to encode");
  if (!dec)
    return las_listener_forward_masked(a->x, a->x_lengths, a->listener_packed, a->listener_dims, mode, a->enc, a->enc_lengths, a->listener_ws,
                                       a->listener_ws_bytes, stream);
  if (!lis)
    return las_speller_decode(a->dec_io, a->speller_packed, a->speller_dims, a->steps, a->decode_mode, mode, a->relu, a->speller_ws,
                              a->speller_ws_bytes, stream);
  const las_speller_dims* sd = a->speller_dims;
  const las_listener_dims* ld = a->listener_dims;
  if (!pipeline_fast(ld, sd, mode) || a->steps <= 0) {  // fp32 mode / variants: the same results, one after the other
    LAS_TRY(las_speller_decode(a->dec_io, a->speller_packed, sd, a->steps, a->decode_mode, mode, a->relu, a->speller_ws, a->speller_ws_bytes, stream));
    return las_listener_forward_masked(a->x, a->x_lengths, a->listener_packed, ld, mode, a->enc, a->enc_lengths, a->listener_ws,
                                       a->listener_ws_bytes, stream);
  }
  // argument checks of the two entry points this call stands for (both dims have passed their checks)
  const las_decode_io* io = a->dec_io;
  LAS_REQUIRE(a->speller_packed && a->speller_ws && a->listener_packed && a->listener_ws && a->enc, "null pointer argument");
  LAS_TRY(decode_args_check(io, sd, a->steps, a->decode_mode, mode, a->speller_ws_bytes));
  const ListenerLayout LL = listener_layout(ld, mode, a->listener_packed, a->listener_ws);
  if (a->listener_ws_bytes < LL.ws_bytes) return fail(LAS_ENOMEM, "listener workspace too small: %zu < %zu", a->listener_ws_bytes, LL.ws_bytes);
  const SpellerLayout SL = speller_layout(sd, mode, false, a->speller_packed, a->speller_ws);
  return fast_pipeline_step(io, fast_f32_inputs(SL), SL.pk_fast, sd, a->steps, a->decode_mode, a->relu, SL.ws_fast, a->x, a->x_lengths,
                            a->listener_packed, ld, a->enc, a->enc_lengths, a->listener_ws, SL.f16, static_cast<cudaStream_t>(stream));
}

int las_pipeline_overlaps(const las_listener_dims* ld, const las_speller_dims* sd, int steps, int mode) {
  return pipeline_fast(ld, sd, mode) && fast_pipeline_plan(ld, sd, steps).bc > 0 ? 1 : 0;
}

int las_nll_sums(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len, float* out2,
                 void* stream) {
  LAS_REQUIRE(logp && labels && out2, "null pointer argument");
  LAS_REQUIRE(S > 0 && S_lab > 0 && B > 0 && V > 0, "bad dims");
  LAS_TRY(device_ok());
  return launch_nll_sums(logp, labels, S, S_lab, B, V, max_label_len, out2, static_cast<cudaStream_t>(stream));
}

int las_label_smoothing_terms(const float* logp, const int32_t* labels, int S, int S_lab, int B, int V, int max_label_len,
                              float label_smoothing, float* per_utt, void* stream) {
  LAS_REQUIRE(logp && labels && per_utt, "null pointer argument");
  LAS_REQUIRE(S > 0 && S_lab > 0 && B > 0 && V > 0, "bad dims");
  LAS_TRY(device_ok());
  return launch_label_smoothing(logp, labels, S, S_lab, B, V, max_label_len, label_smoothing, per_utt, static_cast<cudaStream_t>(stream));
}

int las_debug_gemm_bf16(const void* a, const void* w, const float* bias, float* c, int M, int N, int K, void* stream) {
  LAS_REQUIRE(a && w && bias && c, "null pointer argument");
  LAS_TRY(device_ok());
  return launch_gemm_bf16_tc(static_cast<const __nv_bfloat16*>(a), K, static_cast<const __nv_bfloat16*>(w), K, bias, c, N, M, N, K, false,
                             static_cast<cudaStream_t>(stream));
}
int las_debug_set_option(int key, int value) {
  // The one implementation of the key list in include/las_b200.h: keys [key, key + n) set field[0, n) to a value `ok` accepts.
  struct Key { int key, n; int* field; bool (*ok)(int); };
  auto on_off = [](int v) { return v == 0 || v == 1; };
  auto chunk = [](int v) { return v == 0 || v == 16 || v == 32 || v == 64; };
  auto cluster = [](int v) { return v == 0 || v == 1 || v == 2 || v == 4 || v == 8; };
  auto steps = [](int v) { return v >= 0; };
  auto units = [](int v) { return v == 0 || v == 16 || v == 32; };
  DebugOptions& o = g_debug;
  const Key keys[] = {
      {2, 1, &o.ctx_tmem, on_off},
      {6, 1, &o.rec_overlap, on_off},
      {8, 1, &o.gemm_direct_store, on_off},
      {9, 1, &o.rec_force_bc, chunk},
      {11, 1, &o.att_split, on_off},
      {12, 1, &o.gen_fused, on_off},
      {13, 1, &o.gen_cluster, cluster},
      {19, 1, &o.dec_groups, on_off},
      {20, 8, o.pipe_split, steps},
      {30, 1, &o.dec_units, units},
      {31, 1, &o.pipe_beside, on_off},
  };
  const Key* k = nullptr;
  for (const Key& c : keys)
    if (key >= c.key && key < c.key + c.n) k = &c;
  LAS_REQUIRE(k && k->ok(value), "las_debug_set_option: key %d is not an option, or %d is not one of its values", key, value);
  k->field[key - k->key] = value;
  return LAS_OK;
}
int las_debug_set_trace(void* dev_buf) {
  g_debug.trace = static_cast<long long*>(dev_buf);
  return LAS_OK;
}
int las_debug_umma_probe(const void* a, const void* b, float* d, int N, int K, int a_sw128, int b_sw128, int variant, void* stream) {
  LAS_REQUIRE(a && b && d, "null pointer argument");
  LAS_TRY(device_ok());
  return launch_umma_probe(a, b, d, N, K, a_sw128, b_sw128, variant, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
