// api.cu — the C ABI (include/b200rnn.h) and the host-side sequencing of one multi-layer GRU / (Bi)LSTM
// forward or backward pass. Everything is enqueued on the caller's stream; no allocation, no sync.
//
// Per layer, forward:   [K1 GEMM per direction]  ->  [one persistent recurrence launch, all directions]
//                       -> [K7 dropout, train mode, not after the last layer]
// Per layer, backward:  [W_hh transpose per direction] -> [one persistent BPTT launch, all directions]
//                       -> [bias reduce, wgrad GEMMs (split-K, deterministic), dgrad GEMM]
#include <atomic>
#include <mutex>
#include <stdarg.h>
#include <string.h>

#include "gemm_f32.cuh"
#include "misc_kernels.cuh"
#include "rnn_kernels.cuh"

namespace b200rnn {

static thread_local char g_err[512] = {0};
static std::atomic<unsigned long long> g_launches{0};
long long* g_trace = nullptr;  // debug hook: device buffer [T][8] for rec_fwd phase timestamps

void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Dims {
  int mode, B, T, I, H, L, D, G;
  size_t TB, GH, DH;
  bool training;
  float p;
};

int check_desc(const b200rnn_desc* d, Dims* o) {
  if (!d) {
    set_error("null descriptor");
    return B200RNN_ERR_INVALID;
  }
  if (d->mode != B200RNN_GRU && d->mode != B200RNN_LSTM) {
    set_error("mode must be B200RNN_GRU or B200RNN_LSTM (got %d)", d->mode);
    return B200RNN_ERR_INVALID;
  }
  if (d->batch < 0 || d->seq_len < 0 || d->input_size <= 0 || d->num_layers <= 0 ||
      (d->num_dirs != 1 && d->num_dirs != 2)) {
    set_error("bad shape: B=%d T=%d I=%d L=%d D=%d", d->batch, d->seq_len, d->input_size, d->num_layers,
              d->num_dirs);
    return B200RNN_ERR_INVALID;
  }
  if (d->hidden_size != 64 && d->hidden_size != 128 && d->hidden_size != 256 && d->hidden_size != 512) {
    set_error("hidden_size %d unsupported: the sm_100a persistent kernels are built for 64, 128, 256 and 512",
              d->hidden_size);
    return B200RNN_ERR_UNSUPPORTED;
  }
  if (!(d->dropout_p >= 0.f && d->dropout_p <= 1.f)) {
    set_error("dropout_p must be in [0,1] (got %f)", (double)d->dropout_p);
    return B200RNN_ERR_INVALID;
  }
  o->mode = d->mode;
  o->B = d->batch;
  o->T = d->seq_len;
  o->I = d->input_size;
  o->H = d->hidden_size;
  o->L = d->num_layers;
  o->D = d->num_dirs;
  o->G = d->mode == B200RNN_GRU ? 3 : 4;
  o->TB = (size_t)d->seq_len * d->batch;
  o->GH = (size_t)o->G * o->H;
  o->DH = (size_t)o->D * o->H;
  o->training = d->training != 0;
  o->p = d->dropout_p;
  return B200RNN_OK;
}

constexpr size_t ALIGN_F = 64;  // floats (256 B)

// ---- reserve layout (floats) ------------------------------------------------------------------
struct ReserveLayout {
  size_t gates[8][2], extra[8][2];  // up to 8 layers
  size_t ylayer[8], ydrop[8];
  size_t xln;  // LayerNorm(x) of the folded prologue, kept for the layer-0 wgrad (B200RNN_FLAG_FUSED_LN)
  size_t total;
};

int make_reserve(const Dims& d, ReserveLayout* r, bool fused_ln = false) {
  if (d.L > 8) {
    set_error("num_layers %d > 8 unsupported", d.L);
    return B200RNN_ERR_UNSUPPORTED;
  }
  size_t off = ALIGN_F;  // [0, ALIGN_F): header {dropout seed, dropout offset} written by the forward
  for (int l = 0; l < d.L; ++l)
    for (int k = 0; k < d.D; ++k) {
      r->gates[l][k] = off;
      off += align_up(d.TB * d.GH, ALIGN_F);
      r->extra[l][k] = off;
      off += align_up(d.TB * d.H, ALIGN_F);
    }
  for (int l = 0; l + 1 < d.L; ++l) {
    r->ylayer[l] = off;
    off += align_up(d.TB * d.DH, ALIGN_F);
    r->ydrop[l] = off;
    if (d.p > 0.f) off += align_up(d.TB * d.DH, ALIGN_F);
  }
  r->xln = off;
  if (fused_ln) off += align_up(d.TB * (size_t)d.I, ALIGN_F);
  r->total = off;
  return B200RNN_OK;
}

// ---- scratch layout (floats) ------------------------------------------------------------------
struct ScratchLayout {
  // forward
  size_t f_gates[2], f_y[2], f_tc;
  size_t f_tc_bytes;
  size_t f_total;
  // backward
  size_t b_dgates[2], b_dghn[2], b_wt[2], b_bpart[2], b_dy, b_gemm;
  size_t b_gemm_bytes;
  // tcgen05 backward GEMMs: dense TF32 hi/lo splits of the operands (hi at the offset, lo right behind it)
  size_t b_tc_dg, b_tc_hn, b_tc_x, b_tc_y, b_tc_w, b_tc_part;
  size_t b_tc_part_bytes;
  size_t b_dxln, b_lnpart;  // fused LayerNorm backward: dense d/dLN(x) [TB][I], per-CTA column partials
  size_t b_total;
};

void make_scratch(const Dims& d, ScratchLayout* s) {
  size_t off = ALIGN_F;  // header (dropout seed/offset when nothing is saved for backward)
  for (int k = 0; k < d.D; ++k) {
    s->f_gates[k] = off;
    off += align_up(d.TB * d.GH, ALIGN_F);
  }
  for (int k = 0; k < 2; ++k) {
    s->f_y[k] = off;
    off += align_up(d.TB * d.DH, ALIGN_F);
  }
  // split operands (hi/lo) of the tcgen05 3xTF32 input projection
  {
    const int Kmax = d.I > (int)d.DH ? d.I : (int)d.DH;
    s->f_tc = off;
    s->f_tc_bytes = gemm_tc_scratch_bytes((int)d.TB, (int)d.GH, Kmax);
    off += align_up(s->f_tc_bytes / sizeof(float) + 1, ALIGN_F);
  }
  s->f_total = off;

  off = 0;
  for (int k = 0; k < d.D; ++k) {
    s->b_dgates[k] = off;
    off += align_up(d.TB * d.GH, ALIGN_F);
    s->b_dghn[k] = off;
    off += align_up(d.TB * d.H, ALIGN_F);
    s->b_wt[k] = off;
    off += align_up(d.GH * d.H, ALIGN_F);
    s->b_bpart[k] = off;
    off += align_up((size_t)rec_bwd_max_slices(d.B) * (d.G + 1) * d.H, ALIGN_F);
  }
  s->b_dy = off;
  off += align_up(d.TB * d.DH, ALIGN_F);
  size_t gb = 0;
  const int K = (int)d.TB;
  size_t g0 = gemm_scratch_bytes((int)d.GH, d.I, K);
  size_t g1 = gemm_scratch_bytes((int)d.GH, (int)d.DH, K);
  size_t g2 = gemm_scratch_bytes((int)d.GH, d.H, K);
  gb = g0 > g1 ? g0 : g1;
  gb = gb > g2 ? gb : g2;
  s->b_gemm = off;
  s->b_gemm_bytes = gb;
  off += align_up(gb / sizeof(float) + 1, ALIGN_F);
  {
    const size_t Imax = d.I > (int)d.DH ? (size_t)d.I : d.DH;
    s->b_tc_dg = off;  off += align_up(2 * d.TB * d.GH, ALIGN_F);
    s->b_tc_hn = off;  off += align_up(2 * d.TB * d.H, ALIGN_F);
    s->b_tc_x = off;   off += align_up(2 * d.TB * Imax, ALIGN_F);
    s->b_tc_y = off;   off += align_up(2 * d.TB * d.H, ALIGN_F);
    s->b_tc_w = off;   off += align_up(2 * d.GH * Imax, ALIGN_F);
    s->b_tc_part = off;
    s->b_tc_part_bytes = (size_t)160 * 128 * 128 * sizeof(float);  // <= (#SMs / tiles) * M * N
    off += align_up(s->b_tc_part_bytes / sizeof(float), ALIGN_F);
  }
  s->b_dxln = off;
  off += align_up(d.TB * (size_t)d.I, ALIGN_F);
  s->b_lnpart = off;
  off += align_up(layernorm_bwd_scratch_floats(d.I), ALIGN_F);
  s->b_total = off;
}

// ---- weight cache layout (floats): per (layer, direction) the TF32 hi then lo split of weight_ih [G*H, I_l] -------
struct WCacheLayout {
  size_t hi[8][2], lo[8][2];
  size_t total;
};

void make_wcache(const Dims& d, WCacheLayout* w) {
  size_t off = 0;
  for (int l = 0; l < d.L && l < 8; ++l) {
    const size_t Il = l == 0 ? (size_t)d.I : d.DH;
    for (int k = 0; k < d.D; ++k) {
      w->hi[l][k] = off;
      off += align_up(d.GH * Il, ALIGN_F);
      w->lo[l][k] = off;
      off += align_up(d.GH * Il, ALIGN_F);
    }
  }
  w->total = off;
}

inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

}  // namespace
}  // namespace b200rnn

using namespace b200rnn;

extern "C" {

B200RNN_API int b200rnn_version(void) { return B200RNN_ABI_VERSION; }

B200RNN_API const char* b200rnn_last_error(void) { return g_err; }

B200RNN_API unsigned long long b200rnn_launch_count(void) { return g_launches.load(); }

/* debug only (not declared in the public header): device buffer of [T][8] int64 phase timestamps */
B200RNN_API void b200rnn_debug_set_trace(long long* dev_buf) { g_trace = dev_buf; }

B200RNN_API int b200rnn_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    set_error("cannot query the CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    return B200RNN_ERR_CUDA;
  }
  return n;
}

B200RNN_API int b200rnn_workspace_bytes(const b200rnn_desc* desc, size_t* reserve_bytes, size_t* scratch_bytes) {
  Dims d;
  int rc = check_desc(desc, &d);
  if (rc) return rc;
  ReserveLayout r;
  rc = make_reserve(d, &r, (desc->flags & B200RNN_FLAG_FUSED_LN) != 0);
  if (rc) return rc;
  ScratchLayout s;
  make_scratch(d, &s);
  if (reserve_bytes) *reserve_bytes = (r.total + ALIGN_F) * sizeof(float);
  if (scratch_bytes) *scratch_bytes = ((s.f_total > s.b_total ? s.f_total : s.b_total) + ALIGN_F) * sizeof(float);
  return B200RNN_OK;
}

B200RNN_API int b200rnn_forward_fused(const b200rnn_desc* desc, const float* x, int64_t xs_t, int64_t xs_b,
                                      const float* const* params, float* y, int64_t ys_t, int64_t ys_b, float* h_n,
                                      float* c_n, void* reserve, void* scratch, uint64_t seed, uint64_t offset,
                                      uint64_t* rng_state, const float* ln_gamma, const float* ln_beta, float ln_eps,
                                      float* y_pool, const int32_t* lengths, const void* wcache, void* stream_) {
  Dims d;
  int rc = check_desc(desc, &d);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (d.B == 0 || d.T == 0) return B200RNN_OK;
  if (wcache && !aligned_to(wcache, 256)) {
    set_error("forward: the weight cache must be 256-byte aligned");
    return B200RNN_ERR_INVALID;
  }
  WCacheLayout wl;
  make_wcache(d, &wl);
  const float* WC = static_cast<const float*>(wcache);
  const bool save = (desc->flags & B200RNN_FLAG_SAVE_FOR_BACKWARD) != 0;
  if (!x || !params || (!y && !y_pool) || !h_n || (d.mode == B200RNN_LSTM && !c_n)) {
    set_error("forward: null pointer argument");
    return B200RNN_ERR_INVALID;
  }
  if (!y && save) {
    set_error("forward: the full output is needed by backward (h_{t-1} of every step): pass y as well as y_pool");
    return B200RNN_ERR_INVALID;
  }
  const bool fused_ln = (desc->flags & B200RNN_FLAG_FUSED_LN) != 0;
  if (fused_ln && !ln_gamma) {
    set_error("forward: B200RNN_FLAG_FUSED_LN without ln_gamma / ln_beta");
    return B200RNN_ERR_INVALID;
  }
  if ((ln_gamma == nullptr) != (ln_beta == nullptr)) {
    set_error("forward: LayerNorm prologue needs both gamma and beta");
    return B200RNN_ERR_INVALID;
  }
  if (save && !reserve) {
    set_error("forward: B200RNN_FLAG_SAVE_FOR_BACKWARD needs a reserve buffer");
    return B200RNN_ERR_INVALID;
  }
  if (!scratch) {
    set_error("forward: a scratch buffer is required");
    return B200RNN_ERR_INVALID;
  }
  if ((reserve && !aligned_to(reserve, 256)) || (scratch && !aligned_to(scratch, 256))) {
    set_error("forward: reserve/scratch must be 256-byte aligned");
    return B200RNN_ERR_INVALID;
  }
  ReserveLayout rl;
  rc = make_reserve(d, &rl, fused_ln);
  if (rc) return rc;
  ScratchLayout sl;
  make_scratch(d, &sl);
  float* R = static_cast<float*>(reserve);
  float* S = static_cast<float*>(scratch);
  const bool drop = d.training && d.p > 0.f && d.L > 1;
  uint64_t* hdr = reinterpret_cast<uint64_t*>(save ? R : S);
  if (drop || save) {
    rc = launch_rng_setup(hdr, seed, offset, rng_state, drop ? (uint64_t)((d.TB * d.DH + 3) / 4) : 0, st);
    if (rc) return rc;
  }

  const bool tc = tc_available();
  bool a_ready = false;  // the next layer's A operand (hi/lo) was already produced by this layer's dropout pass
  for (int l = 0; l < d.L; ++l) {
    const int Il = l == 0 ? d.I : (int)d.DH;
    // ---- layer input ---------------------------------------------------------------------------
    const float* in;
    RowMap in_rows;
    if (l == 0) {
      in = x;
      in_rows = tb_rows(xs_t, xs_b, d.B);
    } else {
      if (save)
        in = R + (drop ? rl.ydrop[l - 1] : rl.ylayer[l - 1]);
      else
        in = S + sl.f_y[(l - 1) & 1];
      in_rows = simple_rows((long long)d.DH);
    }
    // ---- A operand of the tensor-core input projection, prepared once per layer (shared by the directions)
    const bool tc_layer = tc && (Il % 32 == 0) && (d.GH % 128 == 0);
    void* tc_ws = S + sl.f_tc;
    if (tc_layer) {
      float* a_hi = tc_a_hi(tc_ws);
      float* a_lo = tc_a_lo(tc_ws, (int)d.TB, Il);
      if (l == 0 && ln_gamma)
        rc = tc_layernorm_split(in, in_rows, (int)d.TB, Il, ln_gamma, ln_beta, ln_eps, a_hi, a_lo, st,
                                (save && fused_ln) ? R + rl.xln : nullptr);
      else if (!a_ready)
        rc = tc_split(in, in_rows, (int)d.TB, Il, a_hi, a_lo, st);
      if (rc) return rc;
    } else if (l == 0 && ln_gamma) {
      set_error("forward: the fused LayerNorm prologue needs the tensor-core input projection (input_size %% 32 == 0)");
      return B200RNN_ERR_UNSUPPORTED;
    }
    a_ready = false;
    RecFwdParams rp;
    memset(&rp, 0, sizeof(rp));
    rp.mode = d.mode; rp.B = d.B; rp.T = d.T; rp.H = d.H; rp.D = d.D;
    rp.training = save ? 1 : 0;
    for (int k = 0; k < d.D; ++k) {
      const float* const* pp = params + (size_t)(l * d.D + k) * 4;
      const float *w_ih = pp[0], *w_hh = pp[1], *b_ih = pp[2], *b_hh = pp[3];
      if (!w_ih || !w_hh || !b_ih || !b_hh) {
        set_error("forward: null parameter pointer (layer %d dir %d)", l, k);
        return B200RNN_ERR_INVALID;
      }
      if (!aligned_to(w_hh, 16)) {
        set_error("forward: weight_hh must be 16-byte aligned for the TMA bulk copy (layer %d dir %d)", l, k);
        return B200RNN_ERR_INVALID;
      }
      float* gates = save ? R + rl.gates[l][k] : S + sl.f_gates[k];
      // K1: x-projection of every time step at once, biases folded (GRU: b_hh only for r,z)
      GemmParams g;
      memset(&g, 0, sizeof(g));
      g.A = in; g.a_rows = in_rows; g.a_kcontig = 1;
      g.B = w_ih; g.b_rows = simple_rows(Il); g.b_kcontig = 1;
      g.C = gates; g.c_rows = simple_rows((long long)d.GH);
      g.M = (int)d.TB; g.N = (int)d.GH; g.K = Il;
      g.bias1 = b_ih; g.bias2 = b_hh;
      g.bias2_n = d.mode == B200RNN_GRU ? 2 * d.H : 4 * d.H;
      if (tc_layer) {
        g.tc_ws = tc_ws;
        g.tc_ws_bytes = sl.f_tc_bytes;
        g.tc_a_presplit = 1;
        if (WC) {  // weight_ih was split once by b200rnn_prepare_weights (frozen encoders)
          g.tc_b_hi = WC + wl.hi[l][k];
          g.tc_b_lo = WC + wl.lo[l][k];
        }
      }
      rc = launch_gemm(g, nullptr, 0, st);
      if (rc) return rc;
      rp.w_hh[k] = w_hh;
      rp.b_hh[k] = b_hh;
      rp.gates[k] = gates;
      rp.extra[k] = save ? R + rl.extra[l][k] : nullptr;
    }
    float* ylay = nullptr;
    if (l == d.L - 1) {
      rp.y = y; rp.y_st = ys_t; rp.y_sb = ys_b;
      rp.y_pool = y_pool;
    } else {
      ylay = save ? R + rl.ylayer[l] : S + sl.f_y[l & 1];
      rp.y = ylay;
      rp.y_st = (long long)d.B * d.DH; rp.y_sb = (long long)d.DH;
    }
    rp.h_n = h_n + (size_t)l * d.D * d.B * d.H;
    rp.c_n = c_n ? c_n + (size_t)l * d.D * d.B * d.H : nullptr;
    rp.trace = g_trace;
    rp.lengths = lengths;
    rc = launch_rec_fwd(rp, st);
    if (rc) return rc;
    if (drop && l + 1 < d.L) {  // K7; keeps the raw output when it is needed by backward, else in place
      float* dropped = save ? R + rl.ydrop[l] : ylay;
      if (tc) {  // also emit the hi/lo split the next layer's tensor-core GEMM consumes (one pass instead of two)
        rc = launch_dropout_split(ylay, dropped, tc_a_hi(tc_ws), tc_a_lo(tc_ws, (int)d.TB, (int)d.DH), d.TB * d.DH, d.p, hdr,
                                  (uint32_t)l, st);
        a_ready = true;
      } else {
        rc = launch_dropout(ylay, dropped, d.TB * d.DH, d.p, hdr, (uint32_t)l, st);
      }
      if (rc) return rc;
    }
  }
  return B200RNN_OK;
}

B200RNN_API int b200rnn_forward(const b200rnn_desc* desc, const float* x, int64_t xs_t, int64_t xs_b,
                                const float* const* params, float* y, int64_t ys_t, int64_t ys_b, float* h_n,
                                float* c_n, void* reserve, void* scratch, uint64_t seed, uint64_t offset,
                                uint64_t* rng_state, void* stream_) {
  return b200rnn_forward_fused(desc, x, xs_t, xs_b, params, y, ys_t, ys_b, h_n, c_n, reserve, scratch, seed, offset,
                               rng_state, nullptr, nullptr, 0.f, nullptr, nullptr, nullptr, stream_);
}

B200RNN_API int b200rnn_wcache_bytes(const b200rnn_desc* desc, size_t* bytes) {
  Dims d;
  int rc = check_desc(desc, &d);
  if (rc) return rc;
  if (d.L > 8) {
    set_error("num_layers %d > 8 unsupported", d.L);
    return B200RNN_ERR_UNSUPPORTED;
  }
  WCacheLayout wl;
  make_wcache(d, &wl);
  if (bytes) *bytes = (wl.total + ALIGN_F) * sizeof(float);
  return B200RNN_OK;
}

B200RNN_API int b200rnn_prepare_weights(const b200rnn_desc* desc, const float* const* params, void* wcache,
                                        void* stream_) {
  Dims d;
  int rc = check_desc(desc, &d);
  if (rc) return rc;
  if (!params || !wcache || !aligned_to(wcache, 256) || d.L > 8) {
    set_error("prepare_weights: null / misaligned argument");
    return B200RNN_ERR_INVALID;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  WCacheLayout wl;
  make_wcache(d, &wl);
  float* WC = static_cast<float*>(wcache);
  for (int l = 0; l < d.L; ++l) {
    const int Il = l == 0 ? d.I : (int)d.DH;
    for (int k = 0; k < d.D; ++k) {
      const float* w_ih = params[(size_t)(l * d.D + k) * 4];
      if (!w_ih) {
        set_error("prepare_weights: null weight_ih (layer %d dir %d)", l, k);
        return B200RNN_ERR_INVALID;
      }
      if (Il % 4 != 0) continue;  // such a layer takes the FFMA projection, which reads the fp32 weights directly
      rc = tc_split(w_ih, simple_rows(Il), (int)d.GH, Il, WC + wl.hi[l][k], WC + wl.lo[l][k], st);
      if (rc) return rc;
    }
  }
  return B200RNN_OK;
}

B200RNN_API int b200rnn_backward_fused(const b200rnn_desc* desc, const float* x, int64_t xs_t, int64_t xs_b,
                                       const float* const* params, const float* y, int64_t ys_t, int64_t ys_b,
                                       const float* dy, int64_t dys_t, int64_t dys_b, const float* dy_pool,
                                       float dy_pool_scale, const float* dh_n, const float* dc_n, const void* reserve,
                                       void* scratch, float* dx, int64_t dxs_t, int64_t dxs_b, float* const* dparams,
                                       const int32_t* lengths, const float* ln_gamma, float ln_eps, float* dln_gamma,
                                       float* dln_beta, void* stream_) {
  Dims d;
  int rc = check_desc(desc, &d);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (d.B == 0 || d.T == 0) return B200RNN_OK;
  if (!x || !params || !y || (!dy && !dy_pool) || !reserve || !scratch || !dparams) {
    set_error("backward: null pointer argument");
    return B200RNN_ERR_INVALID;
  }
  const bool fused_ln = (desc->flags & B200RNN_FLAG_FUSED_LN) != 0;
  if (fused_ln != (ln_gamma != nullptr)) {
    set_error("backward: B200RNN_FLAG_FUSED_LN and ln_gamma must be given together (as in the forward)");
    return B200RNN_ERR_INVALID;
  }
  if (fused_ln && (!(d.I == 128 || d.I == 256 || d.I == 512 || d.I == 1024) || !tc_available())) {
    set_error("backward: the fused LayerNorm needs input_size 128, 256, 512 or 1024");
    return B200RNN_ERR_UNSUPPORTED;
  }
  if (!aligned_to(reserve, 256) || !aligned_to(scratch, 256)) {
    set_error("backward: reserve/scratch must be 256-byte aligned");
    return B200RNN_ERR_INVALID;
  }
  ReserveLayout rl;
  rc = make_reserve(d, &rl, fused_ln);
  if (rc) return rc;
  ScratchLayout sl;
  make_scratch(d, &sl);
  const float* R = static_cast<const float*>(reserve);
  float* S = static_cast<float*>(scratch);
  const bool drop = d.training && d.p > 0.f && d.L > 1;
  const uint64_t* hdr = reinterpret_cast<const uint64_t*>(R);  // dropout seed/offset used by the forward
  const int accumulate = (desc->flags & B200RNN_FLAG_ACCUMULATE_GRADS) ? 1 : 0;
  void* gemm_ws = sl.b_gemm_bytes ? (void*)(S + sl.b_gemm) : nullptr;

  for (int l = d.L - 1; l >= 0; --l) {
    const int Il = l == 0 ? d.I : (int)d.DH;
    RecBwdParams bp;
    memset(&bp, 0, sizeof(bp));
    bp.mode = d.mode; bp.B = d.B; bp.T = d.T; bp.H = d.H; bp.D = d.D;
    if (l == d.L - 1) {
      bp.y = y; bp.y_st = ys_t; bp.y_sb = ys_b;
      bp.dy = dy; bp.dy_st = dys_t; bp.dy_sb = dys_b;
      bp.dy_pool = dy_pool; bp.dy_scale = dy_pool_scale;
    } else {
      bp.y = R + rl.ylayer[l]; bp.y_st = (long long)d.B * d.DH; bp.y_sb = (long long)d.DH;
      bp.dy = S + sl.b_dy; bp.dy_st = (long long)d.B * d.DH; bp.dy_sb = (long long)d.DH;
    }
    bp.dh_n = dh_n ? dh_n + (size_t)l * d.D * d.B * d.H : nullptr;
    bp.dc_n = dc_n ? dc_n + (size_t)l * d.D * d.B * d.H : nullptr;
    for (int k = 0; k < d.D; ++k) {
      const float* const* pp = params + (size_t)(l * d.D + k) * 4;
      if (!pp[0] || !pp[1]) {
        set_error("backward: null parameter pointer (layer %d dir %d)", l, k);
        return B200RNN_ERR_INVALID;
      }
      bp.w_hh[k] = pp[1];
      bp.w_prep[k] = S + sl.b_wt[k];
      bp.gates[k] = R + rl.gates[l][k];
      bp.extra[k] = R + rl.extra[l][k];
      bp.dgates[k] = S + sl.b_dgates[k];
      bp.dghn[k] = S + sl.b_dghn[k];
      bp.dbias_part[k] = S + sl.b_bpart[k];
    }
    bp.lengths = lengths;
    rc = launch_rec_bwd(bp, st);
    if (rc) return rc;

    // layer input as seen by the forward GEMM
    const float* in;
    RowMap in_rows;
    if (l == 0 && fused_ln) {  // what the forward GEMM multiplied: LayerNorm(x), saved densely by the prologue
      in = R + rl.xln;
      in_rows = simple_rows((long long)d.I);
    } else if (l == 0) {
      in = x;
      in_rows = tb_rows(xs_t, xs_b, d.B);
    } else {
      in = R + (drop ? rl.ydrop[l - 1] : rl.ylayer[l - 1]);
      in_rows = simple_rows((long long)d.DH);
    }
    // with the fused LayerNorm the layer-0 dgrad is d/dLN(x): it goes to scratch and through the LN backward below
    const bool ln_l0 = (l == 0) && fused_ln;
    const bool want_dx = (l > 0) || (dx != nullptr) || (ln_l0 && (dln_gamma || dln_beta));
    // ---- tcgen05 3xTF32 path for the wgrad / dgrad GEMMs (falls back to the FFMA kernel per GEMM) -------------
    const bool tc_l = tc_available() && (Il % 128 == 0);
    // Operands whose contraction index (t,b) is their ROW index - X_l, dG, h_prev, dn*r - go to the tensor cores as
    // MN-major tiles (gemm_tc.cu): they only need the dense TF32 hi/lo split, no transposing pass (round 1 transposed
    // every one of them: 10 passes, 8 % of the c2 train step).
    float* xS = S + sl.b_tc_x;  // [TB][Il] hi, then lo
    if (tc_l) {  // X_l, shared by both directions
      rc = tc_split(in, in_rows, (int)d.TB, Il, xS, xS + d.TB * (size_t)Il, st);
      if (rc) return rc;
    }
    for (int k = 0; k < d.D; ++k) {
      const float* const* pp = params + (size_t)(l * d.D + k) * 4;
      float* const* gp = dparams + (size_t)(l * d.D + k) * 4;
      float *dw_ih = gp[0], *dw_hh = gp[1], *db_ih = gp[2], *db_hh = gp[3];
      const float* dG = S + sl.b_dgates[k];
      const float* dHN = S + sl.b_dghn[k];
      if (db_ih || db_hh) {
        rc = launch_bias_reduce(S + sl.b_bpart[k], bp.nslices_out, d.mode, d.H, db_ih, db_hh, accumulate, st);
        if (rc) return rc;
      }
      bool done_dwih = (dw_ih == nullptr), done_dwhh = (dw_hh == nullptr), done_dx = !want_dx;
      if (tc_l) {
        float* dGs = S + sl.b_tc_dg;   // [TB][GH] hi, then lo: MN-major A of the wgrads AND K-major A of the dgrad
        float* hnS = S + sl.b_tc_hn;   // [TB][H]   (GRU: dn * r)
        const TcOperand opX{xS, xS + d.TB * (size_t)Il, (long long)Il, true};
        // the tcgen05 epilogue stores float4: a gradient target that is not 16-byte aligned (a view into a caller's
        // flat bucket behind an odd-sized tensor) takes the FFMA GEMM below instead of failing. The dW_hh GEMMs are
        // H wide (N = H) and the tensor-core tile is 128 wide: H = 64 takes the FFMA GEMM for them. The other two have
        // N = Il (a multiple of 128 here) and contract over T*B or G*H, which the tiles' zero fill covers at any size.
        const bool tc_wih = dw_ih && aligned_to(dw_ih, 16);
        const bool tc_whh = dw_hh && aligned_to(dw_hh, 16) && d.T > 1 && d.H % 128 == 0;
        float* Cx = nullptr;
        RowMap cx_rows = simple_rows(1);
        bool tc_dx = false;
        if (want_dx) {
          if (ln_l0) {
            Cx = S + sl.b_dxln; cx_rows = simple_rows((long long)d.I);
          } else if (l == 0) {
            Cx = dx; cx_rows = tb_rows(dxs_t, dxs_b, d.B);
          } else {
            Cx = S + sl.b_dy; cx_rows = simple_rows((long long)d.DH);
          }
          tc_dx = (reinterpret_cast<uintptr_t>(Cx) % 16 == 0) && cx_rows.s_outer % 4 == 0 && cx_rows.s_inner % 4 == 0;
        }
        if (tc_wih || tc_whh || tc_dx) {
          rc = tc_split(dG, simple_rows((long long)d.GH), (int)d.TB, (int)d.GH, dGs, dGs + d.TB * d.GH, st);
          if (rc) return rc;
        }
        if (tc_wih) {  // dW_ih[GH, Il] = sum_tb dG[tb, :]^T X_l[tb, :]
          const TcOperand opA{dGs, dGs + d.TB * d.GH, (long long)d.GH, true};
          rc = tc_gemm_presplit(opA, opX, (int)d.GH, Il, (int)d.TB, dw_ih, simple_rows(Il), nullptr, nullptr, 0,
                                accumulate, S + sl.b_tc_part, sl.b_tc_part_bytes, st);
          if (rc) return rc;
          done_dwih = true;
        }
        if (tc_whh) {
          // dW_hh = sum_t dGh[t]^T h_{prev(t)}: rows are (t,b) flattened time-major, so the one-step shift is a ROW
          // offset of B (forward: dG[t] with y[t-1]; reverse: dG[t] with y[t+1]); rows beyond Kp read as zero (TMA)
          float* yS = S + sl.b_tc_y;  // [TB][H]
          rc = tc_split(bp.y + (long long)k * d.H, tb_rows(bp.y_st, bp.y_sb, d.B), (int)d.TB, d.H, yS,
                        yS + d.TB * (size_t)d.H, st);
          if (rc) return rc;
          const int Kp = (d.T - 1) * d.B;
          const size_t rowA = (k == 0) ? (size_t)d.B : 0, rowY = (k == 0) ? 0 : (size_t)d.B;
          const TcOperand opY{yS + rowY * d.H, yS + d.TB * (size_t)d.H + rowY * d.H, (long long)d.H, true};
          if (d.mode == B200RNN_LSTM) {
            const TcOperand opA{dGs + rowA * d.GH, dGs + d.TB * d.GH + rowA * d.GH, (long long)d.GH, true};
            rc = tc_gemm_presplit(opA, opY, (int)d.GH, d.H, Kp, dw_hh, simple_rows(d.H), nullptr, nullptr, 0,
                                  accumulate, S + sl.b_tc_part, sl.b_tc_part_bytes, st);
            if (rc) return rc;
          } else {
            rc = tc_split(dHN, simple_rows((long long)d.H), (int)d.TB, d.H, hnS, hnS + d.TB * (size_t)d.H, st);
            if (rc) return rc;
            // columns [0, 2H) of dG: r and z gates
            const TcOperand opRZ{dGs + rowA * d.GH, dGs + d.TB * d.GH + rowA * d.GH, (long long)d.GH, true};
            rc = tc_gemm_presplit(opRZ, opY, 2 * d.H, d.H, Kp, dw_hh, simple_rows(d.H), nullptr, nullptr, 0,
                                  accumulate, S + sl.b_tc_part, sl.b_tc_part_bytes, st);
            if (rc) return rc;
            const TcOperand opN{hnS + rowA * d.H, hnS + d.TB * (size_t)d.H + rowA * d.H, (long long)d.H, true};  // n rows: dn * r
            rc = tc_gemm_presplit(opN, opY, d.H, d.H, Kp, dw_hh + (size_t)2 * d.H * d.H, simple_rows(d.H), nullptr,
                                  nullptr, 0, accumulate, S + sl.b_tc_part, sl.b_tc_part_bytes, st);
            if (rc) return rc;
          }
          done_dwhh = true;
        }
        if (tc_dx) {  // dX_l (+)= dG[TB, GH] * W_ih[GH, Il]: A K-major (the same split of dG), B = W_ih as it lies (MN-major)
          float* wS = S + sl.b_tc_w;   // [GH][Il] hi, then lo
          rc = tc_split(pp[0], simple_rows(Il), (int)d.GH, Il, wS, wS + d.GH * (size_t)Il, st);
          if (rc) return rc;
          const TcOperand opA{dGs, dGs + d.TB * d.GH, (long long)d.GH, false};
          const TcOperand opB{wS, wS + d.GH * (size_t)Il, (long long)Il, true};
          rc = tc_gemm_presplit(opA, opB, (int)d.TB, Il, (int)d.GH, Cx, cx_rows, nullptr, nullptr, 0, (k > 0) ? 1 : 0,
                                nullptr, 0, st);
          if (rc) return rc;
          done_dx = true;
        }
      }
      if (!done_dwih) {  // dW_ih = dGi^T * X_l
        GemmParams g;
        memset(&g, 0, sizeof(g));
        g.A = dG; g.a_rows = simple_rows((long long)d.GH); g.a_kcontig = 0;
        g.B = in; g.b_rows = in_rows; g.b_kcontig = 0;
        g.C = dw_ih; g.c_rows = simple_rows(Il);
        g.M = (int)d.GH; g.N = Il; g.K = (int)d.TB;
        g.accumulate = accumulate;
        rc = launch_gemm(g, gemm_ws, sl.b_gemm_bytes, st);
        if (rc) return rc;
      }
      if (!done_dwhh) {  // dW_hh = sum_t dGh[t]^T * h_{prev(t)}   (h_prev of the first scanned step is 0)
        const int Kp = (d.T - 1) * d.B;
        // forward direction: pairs (dG[t], y[t-1]) for t = 1..T-1 ; reverse: (dG[t], y[t+1]) for t = 0..T-2
        const size_t g_t0 = (k == 0) ? (size_t)d.B : 0;  // first dG row
        const long long y_t0 = (k == 0) ? 0 : bp.y_st;   // first y row offset (elements)
        const float* hp = bp.y + y_t0 + (long long)k * d.H;
        RowMap hp_rows = tb_rows(bp.y_st, bp.y_sb, d.B);
        GemmParams g;
        memset(&g, 0, sizeof(g));
        g.B = hp; g.b_rows = hp_rows; g.b_kcontig = 0;
        g.N = d.H; g.K = Kp;
        g.accumulate = accumulate;
        g.a_kcontig = 0;
        if (d.mode == B200RNN_LSTM) {
          g.A = dG + g_t0 * d.GH; g.a_rows = simple_rows((long long)d.GH);
          g.C = dw_hh; g.c_rows = simple_rows(d.H);
          g.M = (int)d.GH;
          rc = launch_gemm(g, gemm_ws, sl.b_gemm_bytes, st);
          if (rc) return rc;
        } else {
          // r,z rows share dGi; the n rows use dn*r
          g.A = dG + g_t0 * d.GH; g.a_rows = simple_rows((long long)d.GH);
          g.C = dw_hh; g.c_rows = simple_rows(d.H);
          g.M = 2 * d.H;
          rc = launch_gemm(g, gemm_ws, sl.b_gemm_bytes, st);
          if (rc) return rc;
          g.A = dHN + g_t0 * d.H; g.a_rows = simple_rows((long long)d.H);
          g.C = dw_hh + (size_t)2 * d.H * d.H;
          g.M = d.H;
          rc = launch_gemm(g, gemm_ws, sl.b_gemm_bytes, st);
          if (rc) return rc;
        }
      }
      if (!done_dx) {  // dX_l (+)= dGi * W_ih
        GemmParams g;
        memset(&g, 0, sizeof(g));
        g.A = dG; g.a_rows = simple_rows((long long)d.GH); g.a_kcontig = 1;
        g.B = pp[0]; g.b_rows = simple_rows(Il); g.b_kcontig = 0;
        if (ln_l0) {
          g.C = S + sl.b_dxln; g.c_rows = simple_rows((long long)d.I);
        } else if (l == 0) {
          g.C = dx; g.c_rows = tb_rows(dxs_t, dxs_b, d.B);
        } else {
          g.C = S + sl.b_dy; g.c_rows = simple_rows((long long)d.DH);
        }
        g.M = (int)d.TB; g.N = Il; g.K = (int)d.GH;
        g.accumulate = (k > 0) ? 1 : 0;
        rc = launch_gemm(g, nullptr, 0, st);
        if (rc) return rc;
      }
    }
    if (l > 0 && drop) {  // gradient through the inter-layer dropout of layer l-1's output (same mask)
      rc = launch_dropout(S + sl.b_dy, S + sl.b_dy, d.TB * d.DH, d.p, hdr, (uint32_t)(l - 1), st);
      if (rc) return rc;
    }
    if (ln_l0 && want_dx) {  // LayerNorm backward: dx (caller's layout), dgamma, dbeta
      rc = launch_layernorm_bwd(x, tb_rows(xs_t, xs_b, d.B), S + sl.b_dxln, (int)d.TB, d.I, ln_gamma, ln_eps, dx,
                                tb_rows(dxs_t, dxs_b, d.B), dln_gamma, dln_beta, accumulate, S + sl.b_lnpart, st);
      if (rc) return rc;
    }
  }
  return B200RNN_OK;
}

B200RNN_API int b200rnn_backward(const b200rnn_desc* desc, const float* x, int64_t xs_t, int64_t xs_b,
                                 const float* const* params, const float* y, int64_t ys_t, int64_t ys_b,
                                 const float* dy, int64_t dys_t, int64_t dys_b, const float* dh_n,
                                 const float* dc_n, const void* reserve, void* scratch, float* dx, int64_t dxs_t,
                                 int64_t dxs_b, float* const* dparams, const int32_t* lengths, void* stream_) {
  if (!dy) {
    set_error("backward: null pointer argument");
    return B200RNN_ERR_INVALID;
  }
  return b200rnn_backward_fused(desc, x, xs_t, xs_b, params, y, ys_t, ys_b, dy, dys_t, dys_b, nullptr, 0.f, dh_n, dc_n,
                                reserve, scratch, dx, dxs_t, dxs_b, dparams, lengths, nullptr, 0.f, nullptr, nullptr,
                                stream_);
}

B200RNN_API int b200rnn_gemm_f32(int M, int N, int K, const float* A, int64_t lda, int a_kcontig, const float* B,
                     int64_t ldb, int b_kcontig, float* C, int64_t ldc, const float* bias, int accumulate,
                     void* scratch, size_t scratch_bytes, void* stream_) {
  if (M < 0 || N < 0 || K < 0) {
    set_error("gemm: negative dimension");
    return B200RNN_ERR_INVALID;
  }
  GemmParams g;
  memset(&g, 0, sizeof(g));
  g.A = A; g.a_rows = simple_rows(lda); g.a_kcontig = a_kcontig;
  g.B = B; g.b_rows = simple_rows(ldb); g.b_kcontig = b_kcontig;
  g.C = C; g.c_rows = simple_rows(ldc);
  g.M = M; g.N = N; g.K = K;
  g.bias1 = bias;
  g.accumulate = accumulate;
  g.tc_ws = scratch;  // used by the tcgen05 3xTF32 path when the problem is eligible and the buffer is large enough
  g.tc_ws_bytes = scratch_bytes;
  return launch_gemm(g, scratch, scratch_bytes, static_cast<cudaStream_t>(stream_));
}

}  // extern "C"
