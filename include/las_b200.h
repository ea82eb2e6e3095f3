/* las_b200.h -- C ABI of the B200-native LAS forward hot path.
 *
 * Drop-in boundary for jiwidi/las-pytorch's `model/las_model.py`.  The reference has no FFI of its own (it is
 * pure Python over torch); the one call site into the path is `las_model(batch_data, batch_label,
 * teacher_force_rate, is_training)` at solver/solver.py:65-67.  Each entry point below names the reference
 * code it replaces; `las_pytorch_b200/las_model.py` binds them with ctypes behind the reference's own
 * Listener / Speller / LAS / Attention classes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer on the current CUDA device unless the
 *     parameter name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - tensors are dense row-major fp32 with the reference's shapes unless stated otherwise;
 *   - every function returns LAS_OK (0) or a negative LAS_E* code; `las_last_error()` returns a thread-local
 *     message.  The library never aborts and never falls back to the CPU: on a device that is not sm_100 the
 *     compute entry points return LAS_EDEVICE;
 *   - entry points are re-entrant and one thread per GPU replica (nn.DataParallel, train.py:76-78) is safe.  The
 *     library's mutable global state is per-device constant lookups (SM count) and the test hooks at the end of this
 *     header: the las_debug_set_option switches and the las_debug_set_trace buffer are process-wide and unsynchronised;
 *     set them while no other thread calls into the library.
 */
#ifndef LAS_B200_H_
#define LAS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LAS_B200_ABI_VERSION 7

enum {
  LAS_OK = 0,
  LAS_EINVAL = -1,   /* bad shape / null pointer / unsupported configuration */
  LAS_ECUDA = -2,    /* a CUDA runtime call or launch failed (message has the CUDA error string) */
  LAS_EDEVICE = -3,  /* current device is not compute capability 10.x */
  LAS_ENOMEM = -4    /* caller-provided buffer too small */
};

/* Arithmetic mode (north_star: "fp32 mode" 1e-4 / "bf16-GEMM, fp32-state mode" 2e-2). */
enum {
  LAS_MODE_FP32 = 0, /* fp32 operands, fp32 FMA accumulate everywhere */
  LAS_MODE_BF16 = 1, /* bf16 GEMM operands on tcgen05 tensor cores, fp32 accumulate, fp32 c/h state, fp32 softmax */
  LAS_MODE_F16 = 2   /* the same kernels with IEEE fp16 GEMM operands (10 mantissa bits instead of 7: ~8x smaller operand rounding at the
                        same speed; the model's operands -- weights, activations in [-1,1], filterbank features -- are far inside fp16's
                        range, values below 6e-5 lose relative precision).  Everything said about LAS_MODE_BF16 below applies. */
};

/* Recurrent cell (`rnn_unit`, model/las_model.py:69,156: getattr(nn, rnn_unit.upper())).  Weight rows are torch's:
 * LSTM [4H, K] gates i,f,g,o; GRU [3H, K] gates r,z,n; RNN [H, K] (tanh).  GRU / RNN: LAS_MODE_FP32 only. */
enum {
  LAS_CELL_LSTM = 0,
  LAS_CELL_GRU = 1,
  LAS_CELL_RNN = 2
};

/* decode feedback, model/las_model.py:216-234 */
enum {
  LAS_DECODE_RAW = 0,    /* decode_mode 0: feed the log-prob vector back */
  LAS_DECODE_GREEDY = 1, /* decode_mode 1: feed one-hot(argmax) back (ties -> lowest index) */
  LAS_DECODE_SAMPLE = 2  /* decode_mode 2 (:229-234): feed one-hot(sample) back.  The reference draws from Categorical(raw_pred),
                            i.e. it hands the LOG-probabilities to `probs`, which torch renormalises: p_i = logp_i / sum_j logp_j
                            (SURVEY.md A.5.6) -- reproduced.  Its draws come from torch's global generator; here they come from
                            a counter-based generator keyed on (io->sample_seed, step, utterance), so a run is reproducible from
                            its seed but not draw-for-draw equal to the reference's.  `tokens` then holds the sampled tokens. */
};

int las_abi_version(void);
const char* las_last_error(void);
/* 0 if the current device can run the kernels (sm_100), LAS_EDEVICE otherwise. */
int las_device_check(void);
/* 1 if `mode` (LAS_MODE_*) is compiled into this library, else 0. */
int las_mode_available(int mode);
/* number of kernels this library has launched on the calling thread since the last reset (bench.py gpu_launches) */
int64_t las_launch_count(int reset);
/* Optional device-side phase timing for bench.py's roofline: when enabled (per calling thread) the library
 * brackets each named launch group with cudaEvents on the caller's stream.  las_prof_report synchronises those
 * events and writes one "name milliseconds launches" line per recorded group into buf. */
int las_prof_enable(int on);
int las_prof_report(char* buf, size_t buf_bytes);

/* --------------------------------------------------------------------------------------------------------
 * Listener: pyramidal BLSTM encoder.  Replaces Listener.forward / pBLSTMLayer.forward,
 * model/las_model.py:81-91,129-134 (torch nn.LSTM call at :90).
 * ------------------------------------------------------------------------------------------------------ */
typedef struct las_listener_dims {
  int32_t B; /* utterances */
  int32_t T; /* input frames, T % 2^L == 0 (model/las_model.py:86-87 raises otherwise; we return LAS_EINVAL) */
  int32_t F; /* input feature dim (40) */
  int32_t H; /* hidden size per direction */
  int32_t L; /* pyramid layers; output has U = T / 2^L steps of E = 2H features */
  int32_t cell; /* LAS_CELL_* */
} las_listener_dims;

/* One direction of one layer, in the reference's state_dict layout (SURVEY.md A.2); G = 4 (LSTM: i,f,g,o), 3 (GRU: r,z,n)
 * or 1 (RNN) gate blocks of H rows. */
typedef struct las_lstm_weights {
  const float* w_ih; /* [G*H, K_in]  (K_in = 2F for layer 0, 4H for layers >= 1) */
  const float* w_hh; /* [G*H, H] */
  const float* b_ih; /* [G*H] */
  const float* b_hh; /* [G*H] */
} las_lstm_weights;

/* Packed (kernel-layout) weights.  `w_host` is a HOST array of 2L entries ordered
 * layer0.fwd, layer0.reverse, layer1.fwd, ... whose members are device pointers. */
size_t las_listener_packed_bytes(const las_listener_dims* d, int mode);
int las_listener_pack(const las_lstm_weights* w_host, const las_listener_dims* d, int mode, void* packed,
                      size_t packed_bytes, void* stream);
size_t las_listener_workspace_bytes(const las_listener_dims* d, int mode);
/* x [B,T,F] fp32 -> enc [B, T/2^L, 2H] fp32 (forward half first).  The pyramid fold (:86-87) is an index
 * map, never a copy. */
int las_listener_forward(const float* x, const void* packed, const las_listener_dims* d, int mode, float* enc,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Length-mask extension (north_star: "padding is handled by length masks"; SURVEY.md section 8 row f2: the reference's
 * collate_fn computes inputs_length, utils/data.py:146, and train.py:117 drops it).  x_lengths [B] int32 = valid frames per
 * utterance (nullable: NULL reproduces the reference, which runs the BLSTMs over the zero padding).  Layer l keeps
 * len_l = ceil(len_{l-1} / 2) steps: each direction runs over the valid prefix only, exactly as torch's
 * pack_padded_sequence -> nn.LSTM -> pad_packed_sequence does, and outputs past len_l are zero.  enc_lengths [B] int32
 * (nullable) receives len_{L-1}, the attention mask for las_speller_decode. */
int las_listener_forward_masked(const float* x, const int32_t* x_lengths, const void* packed, const las_listener_dims* d,
                                int mode, float* enc, int32_t* enc_lengths, void* workspace, size_t workspace_bytes,
                                void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Speller: attention decoder step loop.  Replaces Speller.forward / forward_step and Attention.forward,
 * model/las_model.py:178-238, 275-297, and the one-hot / TimeDistributed helpers utils/functions.py:54-77.
 * ------------------------------------------------------------------------------------------------------ */
typedef struct las_speller_dims {
  int32_t B;  /* utterances */
  int32_t U;  /* encoder steps */
  int32_t E;  /* encoder feature dim = 2 * listener hidden */
  int32_t Hs; /* speller hidden size; the reference requires Hs == E (SURVEY.md A.4) */
  int32_t sl; /* stacked LSTM layers */
  int32_t V;  /* vocabulary (label_dim) */
  int32_t D;  /* attention MLP dim per head (phi out features = D * heads, psi out features = D) */
  int32_t heads;  /* multi_head (model/las_model.py:268-269, 298-314); 0 is read as 1.  heads > 1: LAS_MODE_FP32 only */
  int32_t no_mlp; /* 1: use_mlp_in_attention=False (:283-285): query = decoder state, keys = enc, D ignored.  LAS_MODE_FP32 only */
  int32_t cell;   /* LAS_CELL_* of rnn_layer; GRU / RNN carry no cell state (c_state is ignored) */
} las_speller_dims;

typedef struct las_speller_weights {
  const las_lstm_weights* rnn_host; /* HOST array [sl]; layer 0 w_ih is [4Hs, V+E] (one-hot columns first) */
  const float* w_phi; /* [D, E]  attention.phi  (model/las_model.py:266) */
  const float* b_phi; /* [D] */
  const float* w_psi; /* [D, E]  attention.psi  (:267) */
  const float* b_psi; /* [D] */
  const float* w_cd;  /* [V, Hs+E] character_distribution (:174) */
  const float* b_cd;  /* [V] */
  const float* w_dr;  /* [E, E*heads] attention.dim_reduce (:269), heads > 1 only (else NULL) */
  const float* b_dr;  /* [E] */
} las_speller_weights;

size_t las_speller_packed_bytes(const las_speller_dims* d, int mode);
int las_speller_pack(const las_speller_weights* w, const las_speller_dims* d, int mode, void* packed,
                     size_t packed_bytes, void* stream);

/* psi = act(enc . W_psi^T + b_psi), [B,U,E] -> [B,U,D] fp32.  Replaces the per-step
 * TimeDistributed(psi, listener_feature) at model/las_model.py:279: it is step-invariant, so it is computed
 * once per utterance batch.  Takes the reference-layout weights directly (attention.psi.weight [D,E], .bias [D]).
 * `relu` = 0 for mlp_activate_in_attention == "None". */
int las_psi_precompute(const float* enc, const float* w_psi, const float* b_psi, int B, int U, int E, int D, int relu,
                       float* psi, void* stream);

/* One attention evaluation (Attention.forward, :275-314, 'dot'):
 * state [B,Hs], enc [B,U,E], psi [B,U,D] -> score [heads,B,U], context [B,E].  w_phi [D*heads,Hs] / b_phi [D*heads]
 * are attention.phi; w_phi == NULL means use_mlp_in_attention=False (q = state, needs D == Hs and heads == 1; pass
 * psi = enc).  heads > 1 (:298-314): every head attends with its own D-wide slice of q over the same keys, the per-head
 * contexts are concatenated and reduced by w_dr [E, E*heads] / b_dr [E] (attention.dim_reduce).
 * enc_lengths (nullable, int32 [B]) is the length-mask extension; NULL reproduces the reference (softmax
 * over all U). */
int las_attention_forward(const float* state, const float* enc, const float* psi, const float* w_phi,
                          const float* b_phi, int B, int U, int E, int Hs, int D, int relu, int heads,
                          const float* w_dr, const float* b_dr, const int32_t* enc_lengths, float* score,
                          float* context, void* stream);

typedef struct las_decode_io {
  /* inputs */
  const float* enc;           /* [B,U,E] listener features */
  const float* psi;           /* [B,U,D] from las_psi_precompute, or NULL to have it computed into the workspace */
  const float* gt_dense;      /* nullable [B,S,V] fp32: teacher forcing, next input = gt[:,step,:] (:216-217) */
  const int32_t* gt_index;    /* nullable [B,S] int32: same, as label indices (one-hot implied) */
  int32_t gt_steps;           /* S dimension of gt_dense / gt_index (>= steps) */
  const int32_t* enc_lengths; /* nullable [B]: attention length mask extension */
  uint64_t sample_seed;       /* LAS_DECODE_SAMPLE: seed of the counter-based generator */
  /* recurrent state, in/out, nullable: NULL = start from zeros / <sos> / enc[:,0,:] (:193-200) */
  float* h_state;             /* [sl,B,Hs] */
  float* c_state;             /* [sl,B,Hs] */
  float* word;                /* [B,V] current input word vector */
  float* context;             /* [B,E] current context */
  /* outputs */
  float* logp;                /* [S,B,V] log-probabilities per step (raw_pred_seq, :213) */
  float* attn;                /* nullable [S,heads,B,U] attention scores per step (attention_record, :214) */
  int32_t* tokens;            /* nullable [S,B] argmax of logp per step (LAS_DECODE_SAMPLE: the sampled tokens) */
  /* Fused loss terms ("next" row f1: NLLLoss(ignore_index=0), solver/solver.py:62,70-77).  nll_labels (nullable, int32
   * [B, nll_steps], independent of teacher forcing) -> nll_terms [S,B] = -logp[s,b,label] where label != 0 and s < nll_steps, else
   * 0.  loss = sum(nll_terms) / count(labels != 0): the caller never has to read the [S,B,V] log-probabilities back. */
  const int32_t* nll_labels;
  int32_t nll_steps;
  float* nll_terms;
  /* Segmented decode.  segment_steps > 0 (rounded up to even): the step loop runs as ceil(steps / segment_steps) persistent launches
   * instead of one, the recurrent state carried between them on the device -- outputs are bit-identical to a single launch
   * (LAS_MODE_BF16; LAS_MODE_FP32 is launch-per-step anyway and ignores it).
   * early_exit != 0 ("next" row f4, <eos> early-exit batching; an extension -- the reference always runs max_label_len steps,
   * model/las_model.py:205-209): after each segment (default 32 steps) the library checks on the device whether every utterance of the
   * launch group (<= 64 consecutive utterances) has emitted `eos_token` (1 in the reference's vocabulary, utils/functions.py:124-125);
   * if so the group's remaining segments return immediately, and its outputs for the steps it did not decode are filled with
   * tokens = eos_token, logp = attn = nll_terms = 0.  Needs `tokens`.  steps_done (nullable, device int32[1]) receives the number of
   * steps decoded (max over the groups).  No host synchronisation is involved. */
  int32_t segment_steps;
  int32_t early_exit;
  int32_t eos_token;
  int32_t* steps_done;
} las_decode_io;

size_t las_speller_workspace_bytes(const las_speller_dims* d, int steps, int mode);
/* Runs `steps` decoder steps (Speller.forward loop, :209-236).  relu: attention activation flag. */
int las_speller_decode(const las_decode_io* io, const void* packed, const las_speller_dims* d, int steps,
                       int decode_mode, int mode, int relu, void* workspace, size_t workspace_bytes, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Beam search (extension: the reference decodes greedily).  Every utterance keeps `beam` = K hypotheses as K decoder rows of the
 * step-per-launch decoder (the fp32 mode's loop and the unfused generic tensor-core step); the K rows share the utterance's encoder
 * features.  Semantics, with S = steps:
 *   - start: K rows in the initial state (<sos>, context = enc[b,0], h = c = 0); row 0 scores 0, the others -inf;
 *   - each step every row runs the decoder step.  A live row k offers (k, v, score[k] + logp[k,v]) for every v (one fp32 add), a
 *     finished row exactly (k, eos_token, score[k]) with token log-prob 0, a -inf row nothing.  The K best candidates by
 *     (score desc, parent asc, token asc) become the new rows (parent's h, c and context; fed-back word one_hot(token)); a row is
 *     finished once its token is eos_token.  A slot left without a finite candidate scores -inf.  All S steps run (see early exit);
 *   - the K final rows are ranked by score / length^length_penalty (fp32 powf; ties to the lower slot), length = tokens up to and
 *     including the first eos_token, or S.  The first `nbest` = N are returned: tokens [B,N,S] (eos_token after the end),
 *     token_logp [B,N,S] (0 after the end), lengths [B,N], scores [B,N] = the raw sums of token_logp.  A -inf slot has length 0;
 *   - attention (attn != NULL): attn[b,n,t] ([heads,U]) is the attention weight vector the decoder computed at step t for the row whose
 *     candidate became token t of hypothesis n, i.e. the PARENT row at step t, before the step's reorder (token_logp follows the same
 *     rule).  0 for t >= lengths[b,n] and for a -inf slot, as greedy early exit leaves undecoded steps; masked encoder steps hold what
 *     greedy decoding's attention record holds;
 *   - early exit (early_exit != 0): every `segment_steps` steps (0 = 32; any count >= 1) the library checks on the device whether all
 *     B*K rows have ended (a -inf slot counts as ended) and, if so, issues no further steps.  The outputs are bit-identical to
 *     early_exit = 0: once every row has ended, every later step keeps each row in place with eos at log-prob 0.  *steps_done receives
 *     the number of steps run.  The loop is driven from the host, so this is the one exception to "nothing synchronises": at each
 *     check the library copies the device flag back and waits on `stream`.  A call with early_exit on a stream that is being captured
 *     returns LAS_EINVAL before anything is enqueued.
 * Limits: 1 <= K <= 32, 1 <= N <= K, 0 <= eos_token < V, length_penalty finite and >= 0, steps >= 1, segment_steps >= 0.
 * ------------------------------------------------------------------------------------------------------ */
typedef struct las_beam_io {
  const float* enc;            /* [B,U,E] listener features */
  const int32_t* enc_lengths;  /* nullable [B] (per utterance, not per hypothesis): attention length mask */
  int32_t beam, nbest, eos_token;
  float length_penalty;
  int32_t* tokens;             /* [B,N,S] */
  float* token_logp;           /* nullable [B,N,S] */
  int32_t* lengths;            /* [B,N] */
  float* scores;               /* [B,N] */
  float* attn;                 /* nullable [B,N,S,heads,U] per-hypothesis attention (heads = max(d->heads, 1)) */
  float* attn_work;            /* caller-owned scratch, required with attn: 4 * S * (heads*B*K*U + B*N) bytes, 4-byte aligned --
                                  [S,heads,B*K,U] fp32 attention of every row and step, then [B,N,S] int32 source rows */
  int32_t early_exit;          /* 0: run all S steps; else stop once every hypothesis has ended (see above) */
  int32_t segment_steps;       /* steps between the early-exit checks (0 = 32) */
  int32_t* steps_done;         /* device int32[1], required with early_exit: steps run */
} las_beam_io;
/* The beam pack: in LAS_MODE_BF16 / LAS_MODE_F16 always the fp32 block followed by the generic tensor-core layout (also for shapes the
 * persistent decoder covers); in LAS_MODE_FP32 the ordinary pack.  The size queries return 0 for arguments the calls reject. */
size_t las_speller_beam_packed_bytes(const las_speller_dims* d, int mode);
int las_speller_beam_pack(const las_speller_weights* w, const las_speller_dims* d, int mode, void* packed, size_t bytes, void* stream);
size_t las_speller_beam_workspace_bytes(const las_speller_dims* d, int steps, int beam, int mode);
int las_speller_beam_search(const las_beam_io* io, const void* packed, const las_speller_dims* d, int steps, int mode, int relu,
                            void* workspace, size_t workspace_bytes, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Cross-batch serving pipeline.  One call stands for `las_speller_decode` of batch i AND `las_listener_forward[_masked]` of batch
 * i+1 (the two calls LAS.forward makes, model/las_model.py:31-39, for two consecutive batches) and produces exactly their
 * results.  In LAS_MODE_BF16, when the listener's recurrence fits on the SMs the persistent decoder leaves free, the two run
 * CONCURRENTLY: where those SMs also leave room for the input-projection GEMMs, the whole listener of the next batch runs beside ONE
 * decoder launch; otherwise the decoder's step loop is cut into L segments, each layer's recurrence runs next to one segment and its
 * GEMM alone on the chip between two segments (csrc/fast_pipeline.cu; debug key 31 forces the latter).  Otherwise (fp32 mode, variants,
 * no free SMs, early_exit) the two are simply enqueued one after the other.  dec_io == NULL: encode only; x == NULL: decode only.
 * `las_pipeline_overlaps` tells whether the concurrent schedule applies to a pair of shapes.
 * ------------------------------------------------------------------------------------------------------ */
typedef struct las_pipeline_args {
  /* batch i: what las_speller_decode takes */
  const las_decode_io* dec_io;
  const void* speller_packed;
  const las_speller_dims* speller_dims;
  int32_t steps, decode_mode, relu;
  void* speller_ws;
  size_t speller_ws_bytes;
  /* batch i+1: what las_listener_forward_masked takes */
  const float* x;
  const int32_t* x_lengths;  /* nullable */
  const void* listener_packed;
  const las_listener_dims* listener_dims;
  float* enc;
  int32_t* enc_lengths;      /* nullable */
  void* listener_ws;
  size_t listener_ws_bytes;
} las_pipeline_args;
int las_pipeline_step(const las_pipeline_args* a, int mode, void* stream);
int las_pipeline_overlaps(const las_listener_dims* ld, const las_speller_dims* sd, int steps, int mode);

/* --------------------------------------------------------------------------------------------------------
 * Solver epilogue ("next" row f1, solver/solver.py:62-92): NLL(ignore_index=0) sums on device.
 * out[0] = sum over non-ignored targets of -logp[s,b,label], out[1] = number of non-ignored targets.
 * ------------------------------------------------------------------------------------------------------ */
int las_nll_sums(const float* logp /*[S,B,V]*/, const int32_t* labels /*[B,S_lab]*/, int S, int S_lab, int B, int V,
                 int max_label_len, float* out2, void* stream);

/* label_smoothing_loss, solver/solver.py:33-45 (the training-branch loss, :79-84), reduced on the device per utterance:
 * per_utt[b] = sum_{s < min(S, S_lab, max_label_len), labels[b,s] >= 0} [ (1-ls) logp[s,b,labels[b,s]] + (ls/V) sum_v logp[s,b,v] ]
 *              / #{s: labels[b,s] >= 0};   the reference's scalar is  -mean_b per_utt[b].
 * labels int32 [B,S_lab]: the index of the 1 in the reference's one-hot target row, or -1 for an all-zero (padding) row. */
int las_label_smoothing_terms(const float* logp /*[S,B,V]*/, const int32_t* labels /*[B,S_lab]*/, int S, int S_lab, int B, int V,
                              int max_label_len, float label_smoothing, float* per_utt /*[B]*/, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Test hooks (used by tests/ only): exercise single kernels through the same ABI.
 * ------------------------------------------------------------------------------------------------------ */
/* C[M,N] fp32 = A[M,K] . W[N,K]^T + bias[N]; A, W bf16 row-major device buffers (the tcgen05 input-projection GEMM). */
int las_debug_gemm_bf16(const void* a_bf16, const void* w_bf16, const float* bias, float* c, int M, int N, int K, void* stream);
/* One CTA: D[128,N] fp32 = A[128,K] . B[N,K]^T through shared-memory operands laid out by the library's UMMA
 * layout helpers (a_sw128 / b_sw128: 0 = interleaved core matrices, 1 = 128-byte swizzle). */
int las_debug_umma_probe(const void* a_bf16, const void* b_bf16, float* d, int N, int K, int a_sw128, int b_sw128, int variant,
                         void* stream);

/* Device buffer that the layer-0 recurrence, the generic decoder step and the persistent decoder fill with clock64 / globaltimer
 * stamps (NULL disables).  Its size in int64: 512 + 5*32*8 + 8 * (SM count) wherever a persistent decoder can run, 64*8 otherwise
 * (layout: TRACE_* in las_pytorch_b200/csrc/las_common.cuh). */
int las_debug_set_trace(void* dev_buf);
/* Process-wide switches for tests and measurements.  Returns LAS_EINVAL (las_last_error names the key) for a key not listed
 * here or a value outside the key's set.  The table in las_debug_set_option (las_pytorch_b200/csrc/las_api.cu) is the one implementation of this list.
 *   key 2:  decoder context through tensor memory (1, default: all feature tiles when they fit, otherwise as many as fit + the rest
 *           on the CUDA cores) or on the CUDA cores only (0);
 *   key 6:  listener input-projection GEMM concurrent with the recurrence (1, default) or in front of it (0);
 *   key 8:  tcgen05 GEMM epilogue with row-per-thread global stores (1) instead of shared-memory staging + TMA stores (0, default);
 *   key 9:  batch chunk per recurrence cluster (16 / 32 / 64; 0 = automatic);
 *   key 11: long encoders attended by a cluster of two CTAs per utterance where one CTA's tensor memory cannot hold enc[b]^T (1,
 *           default) or never (0);
 *   key 12: generic tensor-core decoder step fused (1, default: one launch per stacked-cell layer + a cluster of CTAs per utterance
 *           for the attention) or as separate GEMM / cell / operand kernels with one attention CTA per utterance (0);
 *   key 13: CTAs per utterance of that attention cluster (1 / 2 / 4 / 8; 0 = by batch size);
 *   key 19: two utterance groups pipelined through the persistent decoder's LSTM CTAs (1, default) or the whole batch in lockstep (0);
 *   keys 20 + l (l < 8): decoder steps of the serving pipeline's segment l (>= 0; 0 = proportional to the layer's time steps);
 *   key 30: hidden units per LSTM CTA of the persistent decoder (0, default: 32 for the decoder launch the serving pipeline runs beside
 *           the next batch's listener, 16 otherwise; 16; 32 -- a launch of more than 32
 *           utterances in lockstep, key 19 = 0, then returns LAS_EINVAL);
 *   key 31: serving pipeline schedule (1, default: the listener beside one decoder launch where the chip has room for it, segmented
 *           otherwise; 0: always segmented). */
int las_debug_set_option(int key, int value);

#ifdef __cplusplus
}
#endif
#endif /* LAS_B200_H_ */
