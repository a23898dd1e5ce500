/*
 * b200rnn.h — C-ABI of the B200-native GRU / (Bi)LSTM sequence-encoder library.
 *
 * This is the drop-in boundary for the ONE hot path of
 * speechandlanguageprocessing/ICASSP2022-Depression: the multi-layer torch.nn.GRU /
 * bidirectional torch.nn.LSTM forward + backward that the reference constructs at
 *   Classification/audio_gru_whole.py:59-60      (nn.GRU 256->256, 2 layers, batch_first)
 *   Classification/text_bilstm_whole.py:54-56    (nn.LSTM 1024->H, 2 layers, bidirectional)
 *   Classification/fuse_net_whole.py:266-268, 281-286
 *   Regression/audio_bilstm_perm.py:72-77, Regression/text_bilstm_perm.py:67-69,
 *   Regression/fuse_net.py:245-247, 260-265
 * and calls at audio_gru_whole.py:105, text_bilstm_whole.py:105, fuse_net_whole.py:347,361.
 * The arithmetic the reference reaches lives in PyTorch (torch/nn/modules/rnn.py:1221-1224 GRU
 * equations, :842-847 LSTM equations, :171-216 parameter order); every entry point below says
 * which piece of that interface it replaces.
 *
 * Rules of the ABI:
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller;
 *   - purely stream-ordered: all work is enqueued on `stream`, no host synchronisation, no hidden
 *     allocation on the hot path, capturable in a CUDA graph;
 *   - int return: 0 = ok, <0 = error (message via b200rnn_last_error(), thread-local);
 *   - fp32 everywhere ("dtype": "f32").
 */
#ifndef B200RNN_H_
#define B200RNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RNN_ABI_VERSION 2

#if defined(__GNUC__)
#define B200RNN_API __attribute__((visibility("default")))
#else
#define B200RNN_API
#endif

enum { B200RNN_GRU = 0, B200RNN_LSTM = 1 };

/* error codes */
enum {
  B200RNN_OK = 0,
  B200RNN_ERR_INVALID = -1,     /* bad descriptor / null pointer / misaligned buffer        */
  B200RNN_ERR_UNSUPPORTED = -2, /* shape outside what the sm_100a kernels are built for     */
  B200RNN_ERR_CUDA = -3         /* a CUDA runtime call failed (message has cudaGetErrorString) */
};

/* flags */
#define B200RNN_FLAG_ACCUMULATE_GRADS 1u  /* backward: dparams += grad (else dparams = grad)          */
#define B200RNN_FLAG_SAVE_FOR_BACKWARD 2u /* forward: keep gates / cell state / layer outputs in `reserve` */
#define B200RNN_FLAG_FUSED_LN 4u          /* the LayerNorm prologue is part of the differentiated graph: the forward keeps
                                             LN(x) in `reserve`, b200rnn_backward_fused runs the LayerNorm backward.
                                             Must be set identically for workspace_bytes / forward_fused / backward_fused */

/*
 * Problem descriptor. Mirrors the constructor arguments of torch.nn.GRU / torch.nn.LSTM
 * (rnn.py:1212 / :833) plus the call-time batch shape.
 */
typedef struct b200rnn_desc {
  int32_t mode;        /* B200RNN_GRU (gate order r,z,n) or B200RNN_LSTM (gate order i,f,g,o) */
  int32_t batch;       /* B */
  int32_t seq_len;     /* T */
  int32_t input_size;  /* I  (layer-0 feature width)                                        */
  int32_t hidden_size; /* H  (supported: 64, 128, 256, 512)                                 */
  int32_t num_layers;  /* L                                                                 */
  int32_t num_dirs;    /* D  (1, or 2 = bidirectional)                                      */
  int32_t training;    /* 1: module is in train() mode => inter-layer dropout is applied      */
  float dropout_p;     /* inter-layer dropout probability (rnn.py:857-860 / 1233-1236)       */
  uint32_t flags;      /* B200RNN_FLAG_*                                                    */
} b200rnn_desc;

/* ABI version of the loaded library (== B200RNN_ABI_VERSION). */
B200RNN_API int b200rnn_version(void);

/* Last error message of the calling thread ("" if none). Never NULL. */
B200RNN_API const char* b200rnn_last_error(void);

/* Kernels this library has launched in this process so far (captured launches count once per capture). */
B200RNN_API unsigned long long b200rnn_launch_count(void);

/* Number of SMs of the current device as seen by the library (148 on B200); <0 on error. */
B200RNN_API int b200rnn_sm_count(void);

/*
 * Bytes of the two caller-owned work buffers.
 *   reserve : forward(training=1) writes it, backward reads it (cuDNN-style reserve space)
 *   scratch : transient; max of what forward and backward need
 * Both must be 256-byte aligned (torch.empty on a CUDA device is).
 */
B200RNN_API int b200rnn_workspace_bytes(const b200rnn_desc* desc, size_t* reserve_bytes, size_t* scratch_bytes);

/*
 * Forward pass: replaces `_VF.gru` / `_VF.lstm` behind nn.GRU.forward / nn.LSTM.forward
 * (rnn.py:1449 / :1169) with hx = None (h0 = c0 = 0, rnn.py:1432-1440).
 *
 *   x         [T,B,I] addressed as x[t*x_stride_t + b*x_stride_b + i]  (feature stride 1), so both the
 *             batch_first layout of audio_gru_whole.py:60 and the permuted NON-contiguous view of
 *             text_bilstm_whole.py:103 are consumed in place
 *   params    4*L*D device pointers in nn order: for layer l, direction d:
 *             weight_ih[G*H, I_l], weight_hh[G*H, H], bias_ih[G*H], bias_hh[G*H]   (rnn.py:171-216)
 *   y         [T,B,D*H] addressed as y[t*y_stride_t + b*y_stride_b + c]
 *   h_n       [L*D, B, H] contiguous (layer-major, direction-minor: l0 fwd, l0 rev, l1 fwd, ...)
 *   c_n       same shape, LSTM only (NULL for GRU)
 *   reserve   written when flags has B200RNN_FLAG_SAVE_FOR_BACKWARD (may be NULL otherwise)
 *   scratch   always required (transient: split operands of the tensor-core input projection, and the
 *             gates / layer outputs when nothing is saved, e.g. the no_grad forward of fuse_net_whole.py:337)
 *   dropout_seed / dropout_offset / rng_state : Philox4x32-10 key / counter base of the inter-layer
 *             dropout mask. If rng_state (DEVICE pointer to {seed, offset}) is non-NULL the pair is read
 *             from it on the device and the offset is advanced there, so a captured CUDA graph draws a
 *             fresh mask at every replay; otherwise the by-value pair is used. The pair actually used is
 *             recorded in `reserve` for b200rnn_backward.
 */
B200RNN_API int b200rnn_forward(const b200rnn_desc* desc, const float* x, int64_t x_stride_t,
                                int64_t x_stride_b, const float* const* params, float* y, int64_t y_stride_t,
                                int64_t y_stride_b, float* h_n, float* c_n, void* reserve, void* scratch,
                                uint64_t dropout_seed, uint64_t dropout_offset, uint64_t* rng_state,
                                void* stream /* cudaStream_t */);

/*
 * Forward with the model-shell fusions around the encoder (SURVEY.md 8f rank 1), used by the audio branch
 * `x = self.ln(x); x, _ = self.lstm_net_audio(x); x = x.sum(dim=1)` of fuse_net_whole.py:360-362:
 *   ln_gamma/ln_beta/ln_eps : LayerNorm over the feature dimension applied to x on the fly (folded into the operand
 *                             preparation of the layer-0 input projection); NULL = no LayerNorm
 *   y_pool                  : optional [B, D*H] = sum over time of the top layer's output; with y == NULL the
 *                             [T,B,D*H] output is never written (only allowed without B200RNN_FLAG_SAVE_FOR_BACKWARD)
 *   lengths                 : optional DEVICE array [B] of valid step counts (torch PackedSequence semantics on the
 *                             padded [T,B,*] layout, DAICFeatureExtarction/feature_extraction.py:45-64 yields such
 *                             ragged sequences): past its length a sequence keeps its state (h_n / c_n are the state
 *                             at its last valid step) and its output rows are 0; the reverse direction starts at
 *                             lengths[b]-1. NULL = every sequence has T steps. Must be passed again to backward.
 *   wcache                  : optional weight cache written by b200rnn_prepare_weights for the SAME desc / params: the
 *                             TF32 hi/lo split of every weight_ih, so that frozen encoders (fuse_net_whole.py:590-593:
 *                             only fc_final.0.weight trains) do not re-split their weights at every step. NULL = split on
 *                             the fly. The caller owns it and must refresh it whenever a weight_ih changes.
 * Everything else as b200rnn_forward (which is this call with the six extra arguments zero).
 */
B200RNN_API int b200rnn_forward_fused(const b200rnn_desc* desc, const float* x, int64_t x_stride_t,
                                      int64_t x_stride_b, const float* const* params, float* y, int64_t y_stride_t,
                                      int64_t y_stride_b, float* h_n, float* c_n, void* reserve, void* scratch,
                                      uint64_t dropout_seed, uint64_t dropout_offset, uint64_t* rng_state,
                                      const float* ln_gamma, const float* ln_beta, float ln_eps, float* y_pool,
                                      const int32_t* lengths, const void* wcache, void* stream /* cudaStream_t */);

/* Weight cache of b200rnn_forward_fused: size for this descriptor (batch / seq_len are ignored), and the pass that
 * fills it (one small launch per weight_ih; 256-byte aligned caller-owned buffer). */
B200RNN_API int b200rnn_wcache_bytes(const b200rnn_desc* desc, size_t* bytes);
B200RNN_API int b200rnn_prepare_weights(const b200rnn_desc* desc, const float* const* params, void* wcache,
                                        void* stream /* cudaStream_t */);

/*
 * Backward pass (BPTT): what autograd runs for loss.backward() through nn.GRU / nn.LSTM
 * (audio_gru_whole.py:190, text_bilstm_whole.py:182). `desc` must equal the forward's.
 *
 *   y, dy     forward output and its gradient, strided like y above (dy has its own strides)
 *   dh_n,dc_n gradients w.r.t. h_n / c_n, [L*D,B,H] contiguous, or NULL (= zero)
 *   dx        [T,B,I] strided like x, or NULL to skip (the reference asks for it:
 *             audio_gru_whole.py:179 sets requires_grad=True on the input)
 *   dparams   4*L*D device pointers shaped like params (e.g. views into ONE flat gradient bucket that
 *             a single ncclAllReduce consumes); entries may be NULL to skip; written or accumulated per
 *             B200RNN_FLAG_ACCUMULATE_GRADS
 *   lengths   the array given to b200rnn_forward_fused, or NULL
 */
B200RNN_API int b200rnn_backward(const b200rnn_desc* desc, const float* x, int64_t x_stride_t,
                                 int64_t x_stride_b, const float* const* params, const float* y,
                                 int64_t y_stride_t, int64_t y_stride_b, const float* dy, int64_t dy_stride_t,
                                 int64_t dy_stride_b, const float* dh_n, const float* dc_n, const void* reserve,
                                 void* scratch, float* dx, int64_t dx_stride_t, int64_t dx_stride_b,
                                 float* const* dparams, const int32_t* lengths, void* stream /* cudaStream_t */);

/*
 * Backward with the model-shell fusions of the TRAINING path (SURVEY.md 8f rank 1; audio_gru_whole.py:103-108 with
 * loss.backward() at :190): b200rnn_backward plus
 *   dy_pool / dy_pool_scale : when dy == NULL the top layer's output gradient is dy_pool[b, c] * dy_pool_scale for
 *                             EVERY time step - the gradient of `x.mean(dim=1)` / `x.sum(dim=1)` over the encoder output
 *                             (audio_gru_whole.py:106, audio_bilstm_perm.py:125) broadcast inside the BPTT kernel, so the
 *                             [T,B,D*H] gradient tensor is never written nor read
 *   ln_gamma / ln_eps       : with B200RNN_FLAG_FUSED_LN: the layer-0 input gradient is d/dLN(x); it is pushed through
 *                             the LayerNorm backward (statistics recomputed from x) into dx, and
 *   dln_gamma / dln_beta    : (+)= the LayerNorm parameter gradients (NULL to skip), per B200RNN_FLAG_ACCUMULATE_GRADS
 */
B200RNN_API int b200rnn_backward_fused(const b200rnn_desc* desc, const float* x, int64_t x_stride_t,
                                       int64_t x_stride_b, const float* const* params, const float* y,
                                       int64_t y_stride_t, int64_t y_stride_b, const float* dy, int64_t dy_stride_t,
                                       int64_t dy_stride_b, const float* dy_pool, float dy_pool_scale,
                                       const float* dh_n, const float* dc_n, const void* reserve, void* scratch,
                                       float* dx, int64_t dx_stride_t, int64_t dx_stride_b, float* const* dparams,
                                       const int32_t* lengths, const float* ln_gamma, float ln_eps, float* dln_gamma,
                                       float* dln_beta, void* stream /* cudaStream_t */);

/*
 * Dense helper used by the path (time-parallel input projection, wgrad, dgrad):
 *   C[m,n] (+)= sum_k A(m,k) * B(k,n) + bias[n]
 * exposed so the parity tests can pin the GEMM on its own.
 *   a_kcontig : 1 -> A is [M,K] row-major with leading dimension lda; 0 -> A is [K,M] row-major (lda)
 *   b_kcontig : 1 -> B is [N,K] row-major (ldb) ("NT");               0 -> B is [K,N] row-major (ldb)
 */
B200RNN_API int b200rnn_gemm_f32(int M, int N, int K, const float* A, int64_t lda, int a_kcontig, const float* B,
                     int64_t ldb, int b_kcontig, float* C, int64_t ldc, const float* bias, int accumulate,
                     void* scratch, size_t scratch_bytes, void* stream);

/*
 * Model-shell kernels of the fuse step (SURVEY.md 8f ranks 1 and 3). Each replaces a chain of tiny framework
 * launches on either side of the encoders; all stream-ordered, caller-owned fp32 buffers.
 *
 *  b200rnn_attention_pool : attention_net_with_w (text_bilstm_whole.py:74-99, fuse_net_whole.py:310-334)
 *       seq [T,B,2H] at t*s_t + b*s_b + c, h_n [n_states,B,H], w_a [H,H], b_a [H]  ->  ctx [B,H]
 *  b200rnn_mlp_dropout    : Dropout -> Linear(n,n) -> ReLU -> Dropout (fc_out / fc_audio, fuse_net_whole.py:270-275, 288-293)
 *       dropout masks: Philox streams stream_id and stream_id+1 keyed by rng_hdr = {seed, offset}
 *  b200rnn_rng_next       : rng_hdr <- *rng_state ; rng_state.offset += consume   (device side, graph replayable)
 *  b200rnn_fuse_loss_grad : probs = Softmax(cat(tf,af) W^T); loss = CE(tf W[:, :Ht]^T, y) + CE(af W[:, Ht:]^T, y);
 *       dW (+)= d loss / dW   for W = fc_final.0.weight [2, Ht+Ha]  (fuse_net_whole.py:368-395, 445-454)
 *  b200rnn_adam           : one torch.optim.Adam step (no weight decay, no amsgrad) over n contiguous parameters;
 *       m, v, step (a device float counting completed steps) are the optimiser state  (fuse_net_whole.py:416, 456)
 */
B200RNN_API int b200rnn_attention_pool(const float* seq, int64_t s_t, int64_t s_b, const float* h_n, int n_states,
                                       int B, int T, int H, const float* w_a, const float* b_a, float* ctx,
                                       void* stream);
/* Backward of b200rnn_attention_pool (the text models train through it: text_bilstm_whole.py:74-99, 182): one launch
 * recomputes the forward per batch row and writes dseq [T,B,2H] (both halves), dh_n [n_states,B,H], and the two [B,H]
 * row buffers dqpre / hsum from which the caller forms d attention_layer.0.weight = dqpre^T hsum (one small GEMM) and
 * d attention_layer.0.bias = column sums of dqpre. */
B200RNN_API int b200rnn_attention_pool_bwd(const float* seq, int64_t s_t, int64_t s_b, const float* h_n, int n_states,
                                           int B, int T, int H, const float* w_a, const float* b_a, const float* dctx,
                                           float* dseq, int64_t d_t, int64_t d_b, float* dh_n, float* dqpre,
                                           float* hsum, void* stream);
B200RNN_API int b200rnn_mlp_dropout(const float* x, int B, int n, const float* W, const float* bias, float* out,
                                    int training, float p, const uint64_t* rng_hdr, uint32_t stream_id, void* stream);
B200RNN_API int b200rnn_rng_next(uint64_t* rng_hdr, uint64_t* rng_state, uint64_t consume, void* stream);
B200RNN_API int b200rnn_fuse_loss_grad(const float* text_feature, int Ht, const float* audio_feature, int Ha,
                                       const int64_t* labels, int B, const float* W, float* dW, int accumulate,
                                       float* loss, float* probs, void* stream);
/* CrossEntropyLoss on Softmax OUTPUTS, as the classification scripts compute it (audio_gru_whole.py:73,188,308;
 * text_bilstm_whole.py:68,180,304): probs = softmax(logits) [B,C]; loss = mean_b -log softmax(probs_b)[y_b]; and
 * dlogits = d loss / d logits through both softmaxes, all in one pass (C <= 32). row_loss [B] is scratch. */
B200RNN_API int b200rnn_softmax_ce(const float* logits, const int64_t* labels, int B, int C, float* probs, float* dlogits,
                                   float* row_loss, float* loss, void* stream);
B200RNN_API int b200rnn_adam(float* p, const float* g, float* m, float* v, float* step, size_t n, float lr,
                             float beta1, float beta2, float eps, void* stream);
/* AdamW over one flat parameter group (audio_gru_whole.py:247-255, 307: optim.AdamW with a decay and a no-decay group):
 * p = p*(1 - lr*weight_decay) - lr/(1-b1^t) * m / (sqrt(v/(1-b2^t)) + eps), with g scaled by grad_scale (the 1/world of
 * the data-parallel mean) on the fly. Groups sharing `step` pass advance_step = 1 only for the last group. */
B200RNN_API int b200rnn_adamw(float* p, const float* g, float* m, float* v, float* step, size_t n, float lr,
                              float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                              int advance_step, void* stream);

/*
 * The whole tail of the fuse step in ONE launch (csrc/fuse_head.cu): attention pooling, the two
 * Dropout-Linear-ReLU-Dropout heads, the model output (Softmax(fc_final(cat)) of fuse_net_whole.py:368-374, or
 * ReLU(fc_final(sigmoid(modal_attn x) * x)) of Regression/fuse_net.py:345-351), MyLoss (two-head cross entropy,
 * fuse_net_whole.py:380-395, or two-head SmoothL1, fuse_net.py:357-366), d loss / d fc_final.0.weight, the
 * data-parallel sum of that gradient over the ranks (one-shot NVLink exchange through peer-mapped buffers, see
 * b200rnn_comm_*), and the torch.optim.Adam step (fuse_net_whole.py:416, 456). Replaces b200rnn_attention_pool +
 * b200rnn_rng_next + 2 x b200rnn_mlp_dropout + b200rnn_fuse_loss_grad + ncclAllReduce + b200rnn_adam.
 *
 * All pointers are device pointers. Stages are switched by which pointers are set:
 *   seq != NULL            : attention pooling from the BiLSTM output (else ctx_in [B,Ht] is the attention context)
 *   tf_in != NULL          : text stage done by an earlier launch (its text_feature output); skips attention + fc_out
 *   pooled == NULL         : text stage only (requires W == NULL): lets the text half run on the text branch's stream
 *                            while the audio encoder is still busy, the final launch then takes tf_in
 *   W   != NULL            : output + loss + gradient (+ exchange when world > 1) (+ Adam when do_adam); W == NULL
 *                            stops after text_feature / audio_feature
 * Dropout: Philox streams 0,1 (text head in/out) and 2,3 (audio head in/out) keyed by rng_state = {seed, offset}
 * (read on the device; with the loss stage the offset is advanced by rng_consume at the end, so a captured CUDA graph
 * draws fresh masks per replay) - the same streams b200rnn_mlp_dropout uses.
 */
#define B200RNN_COMM_MAX_WORLD 8
#define B200RNN_IPC_HANDLE_BYTES 64
typedef struct b200rnn_fuse_head_args {
  uint32_t struct_bytes;  /* sizeof(b200rnn_fuse_head_args): binding / library mismatch is rejected            */
  int32_t B, T, Ht, Ha;   /* batch rows, text time steps, text / audio feature widths (multiples of 4)          */
  int32_t n_states;       /* rows of h_n summed by the attention query (L*D = 4)                                */
  int32_t training;       /* 1: Dropout active (model.train())                                                  */
  float p;                /* Dropout probability of the heads                                                   */
  int32_t regression;     /* 0: 2-class classification flavour; 1: regression flavour (1 output, float labels)  */
  int32_t accumulate;     /* dw += gradient instead of dw = gradient                                            */
  int32_t do_adam;        /* apply the Adam update to W in the same launch                                      */
  int32_t world, rank;    /* data-parallel ranks (1 = no exchange) and this rank                                */
  int32_t defer_exchange; /* world > 1: 1 = send this step's gradient to the peers and return; the wait for theirs, the
                             rank-ordered sum and Adam are done by b200rnn_fuse_head_finish (normally enqueued at the
                             START of the next step beside the encoders), so a rank never idles for a slower one */
  float lr, beta1, beta2, eps, grad_scale; /* Adam hyper-parameters; grad_scale = 1/world                        */
  uint64_t rng_consume;   /* Philox offset advance per call: ceil(B*max(Ht,Ha)/4)                               */
  int64_t seq_st, seq_sb; /* element strides of seq: seq[t*seq_st + b*seq_sb + c], c in [0, 2*Ht)              */
  const float* seq;       /* BiLSTM output [T,B,2*Ht] (fwd | rev halves) or NULL                                */
  const float* h_n;       /* [n_states,B,Ht]                                                                    */
  const float* w_att;     /* attention_layer.0.weight [Ht,Ht]                                                   */
  const float* b_att;     /* attention_layer.0.bias [Ht]                                                        */
  const float* ctx_in;    /* [B,Ht] attention context when seq == NULL                                          */
  float* ctx_out;         /* optional [B,Ht]: the attention context before Dropout                              */
  const float* tf_in;     /* [B,Ht] text_feature computed by an earlier launch of this entry point (text stage on its
                             own stream, see below): the text stage is skipped entirely                         */
  const float* w_t;       /* fc_out.1.weight [Ht,Ht]                                                            */
  const float* b_t;       /* fc_out.1.bias [Ht]                                                                 */
  const float* pooled;    /* [B,Ha] time-summed GRU output                                                      */
  const float* w_a;       /* fc_audio.1.weight [Ha,Ha]                                                          */
  const float* b_a;       /* fc_audio.1.bias [Ha]                                                               */
  uint64_t* rng_state;    /* {seed, offset}; required when training && p > 0                                    */
  float* text_feature;    /* optional out [B,Ht]                                                                */
  float* audio_feature;   /* optional out [B,Ha]                                                                */
  float* W;               /* fc_final.0.weight [C, Ht+Ha], C = 2 (classification) or 1 (regression); NULL = stop */
  const float* w_modal;   /* regression: modal_attn.weight [F,F] (NULL: output = ReLU(fc_final(x)))              */
  const void* labels;     /* int64 class indices [B] (classification) or float targets [B] (regression)         */
  float* out;             /* optional: probs [B,2] or prediction [B]                                            */
  float* loss;            /* scalar                                                                             */
  float* dw_part;         /* scratch, b200rnn_fuse_head_scratch_floats() floats                                  */
  float* dw;              /* [C*(Ht+Ha) + 1]: the reduced gradient (and this rank's loss in the last element)    */
  uint32_t* ticket;       /* one zero-initialised uint32 (CTA completion counter; the kernel re-arms it)        */
  float* adam_m;          /* Adam state, each [C*(Ht+Ha)]                                                       */
  float* adam_v;
  float* adam_step;       /* device float counting completed steps                                              */
  uint32_t* comm_step;    /* world > 1: device uint32 step counter of the exchange (zero-initialised)           */
  uint32_t* comm_done;    /* defer_exchange: device uint32 count of steps whose update has been applied (zero-init.) */
  void* comm_buf[B200RNN_COMM_MAX_WORLD]; /* world > 1: every rank's exchange buffer as mapped in THIS process    */
} b200rnn_fuse_head_args;

B200RNN_API size_t b200rnn_fuse_head_scratch_floats(int B, int Ht, int Ha, int regression);
B200RNN_API int b200rnn_fuse_head(const b200rnn_fuse_head_args* args, void* stream);
/* Second half of a deferred exchange (defer_exchange = 1): if a step's gradient has been sent but not applied yet, wait
 * for every peer's slot of that step, add the slots in rank order and apply Adam to W; otherwise do nothing. Uses the
 * W / adam_* / lr.. / grad_scale / world / rank / comm_* fields of the same argument block. One tiny launch. */
B200RNN_API int b200rnn_fuse_head_finish(const b200rnn_fuse_head_args* args, void* stream);

/*
 * Exchange buffers of the one-shot gradient exchange (setup path; the only allocation the library ever makes, done
 * once per process, never on the hot path). Each rank creates its buffer, ships the 64-byte CUDA IPC handle to its
 * peers (any side channel, e.g. torch.distributed.all_gather), and opens theirs:
 *   b200rnn_comm_bytes()               size of a buffer (flags + 2 parities x MAX_WORLD slots of 4 KB)
 *   b200rnn_comm_create(&buf, handle)  cudaMalloc + zero + cudaIpcGetMemHandle on the current device
 *   b200rnn_comm_open(handle, &peer)   cudaIpcOpenMemHandle (peer access over NVLink is enabled lazily)
 *   b200rnn_comm_close / _destroy      unmap a peer buffer / free the own one
 */
B200RNN_API size_t b200rnn_comm_bytes(void);
B200RNN_API int b200rnn_comm_create(void** local_buf, unsigned char* ipc_handle_out);
B200RNN_API int b200rnn_comm_open(const unsigned char* ipc_handle, void** peer_buf);
B200RNN_API int b200rnn_comm_close(void* peer_buf);
B200RNN_API int b200rnn_comm_destroy(void* local_buf);

/*
 * Optional device-side timing of the library's own launches (CUDA event pairs on the launching stream),
 * used by bench.py for the roofline figure. kind: 0 = forward recurrence, 1 = backward recurrence,
 * 2 = GEMM, 3 = other. Do not enable while capturing a CUDA graph.
 *   b200rnn_profile(enable)       : switch on/off and forget what was recorded so far
 *   b200rnn_profile_read(kind,..) : wait for the recorded launches of `kind`; sum of their durations + count
 */
B200RNN_API int b200rnn_profile(int enable);
B200RNN_API int b200rnn_profile_read(int kind, float* total_ms, int* launches);

#ifdef __cplusplus
}
#endif
#endif /* B200RNN_H_ */
