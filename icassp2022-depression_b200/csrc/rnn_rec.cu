// rnn_rec.cu — persistent recurrence kernels for sm_100a (K2/K3 forward, K4/K5 backward).
//
// Replaces the T-serial inner loop the reference reaches through torch.nn.GRU / torch.nn.LSTM
// (GRU cell equations torch/nn/modules/rnn.py:1221-1224, LSTM cell :842-847; call sites
// audio_gru_whole.py:105, text_bilstm_whole.py:105, fuse_net_whole.py:347,361).
//
// Design (one launch = every time step of every direction of one layer):
//   * grid = D * nslices thread-block clusters of C CTAs. A cluster owns BS batch rows; CTA `rank` of the
//     cluster owns HS = H/C hidden units and keeps the matching rows of W_hh (forward) or columns of W_hh
//     (backward) on chip for the whole sequence: G-RG gate blocks in shared memory, staged once with TMA bulk
//     copies (cp.async.bulk ... mbarrier::complete_tx), and RG gate blocks in registers.
//   * per step every warp contracts its rows against the BS state vectors (rnn_core.cuh: K across lanes,
//     transposing shuffle butterfly); the lane that ends up owning (unit, batch) applies the gate
//     non-linearities and the state update in registers.
//   * the new state slice is all-gathered into the C peer CTAs with st.async (16-byte DSMEM stores that complete
//     transaction bytes on an mbarrier in the destination CTA): data and "ready" signal travel together, the
//     consumer waits on a local mbarrier, double buffered. No cluster barrier, fence or L1 flush in the loop.
//   * batch slices are independent clusters: no grid-wide synchronisation anywhere.
//
// fp32 FFMA by choice: the per-step contraction is [BS x H] x [H x G*HS] with BS = 4..8 rows per CTA —
// far too skinny for tcgen05 tiles, and parity is judged at 1e-5 against an fp32 reference.
#include <mutex>
#include <stdlib.h>

#include "profile.cuh"
#include "ptx.cuh"
#include "rnn_core.cuh"
#include "rnn_kernels.cuh"

namespace b200rnn {

namespace {

constexpr int MAX_SMEM = 232448;  // 227 KB opt-in limit per CTA on sm_100
// The CTA's own state slice is delivered locally (st.shared + mbarrier.arrive per warp). -DB200RNN_SELF_VIA_CLUSTER
// builds the round-1 behaviour (own slice through st.async like the peers'): compute-sanitizer's racecheck does not
// model the ordering that inline-PTX mbarrier.arrive / try_wait give to ordinary shared-memory stores and flags every
// local store / LDS pair of the default build, so the race-free evidence of the REST of the kernel is taken on that
// build (profiles/README.md); the ordering argument for the local path is in allgather_units' comment.
#ifdef B200RNN_SELF_VIA_CLUSTER
constexpr bool kLocalSelf = false;
#else
constexpr bool kLocalSelf = true;
#endif
constexpr unsigned FULLMASK = 0xffffffffu;

template <int MODE, int H, int C, int BS, int KL, int UPL, int RG>
struct RecCfg {
  static constexpr int G = (MODE == B200RNN_GRU) ? 3 : 4;
  static constexpr int GH = G * H;
  static constexpr int HS = H / C;
  static constexpr int UPW = (32 / KL) * UPL;
  static constexpr int NW = HS / UPW;
  static constexpr int NT = NW * 32;
  static constexpr int NSM = G - RG;  // gate blocks held in shared memory
  static constexpr int CW = 4 * KL;   // floats of the contraction dimension per chunk
  static constexpr int NCH = H / CW;  // chunks per state vector (per gate block in the backward)
  static constexpr bool ROT = (CW <= HS);           // chunk order rotates so the CTA's own slice comes first
  static constexpr int CPS = ROT ? HS / CW : 1;     // chunks per source slice (ROT)
  static constexpr int SPC = ROT ? 1 : CW / HS;     // source slices per chunk (!ROT)
  static constexpr int NBAR = 1 + 2 * C;            // [0] weights, [1 + buf*C + src] state slices
  static constexpr size_t BAR_BYTES = (NBAR * 8 <= 256) ? 256 : 512;  // 512 only for the 16-CTA clusters (H = 512)
  static constexpr size_t W_BYTES = (size_t)NSM * HS * H * sizeof(float);
  static constexpr size_t FWD_SMEM = W_BYTES + (size_t)2 * BS * H * sizeof(float) + BAR_BYTES;
  static constexpr size_t BWD_SMEM = W_BYTES + (size_t)2 * BS * GH * sizeof(float) + BAR_BYTES;
  static_assert(NBAR * 8 <= (int)BAR_BYTES, "barrier block too small");
  static_assert(ROT ? (HS % CW == 0) : (CW % HS == 0), "chunks must tile the per-CTA slices");
  static_assert(RG >= 0 && RG <= 2, "at most two register-resident gate blocks");
  static_assert(HS * C == H && NW * UPW == HS && NW >= 1, "bad split");
  static_assert(UPW % 4 == 0, "the exchange packs 4 units per 16-byte store");
  static_assert(NT <= 1024, "too many threads");
};

// All-gather `val` (owned by lane (unit, batch) of every warp) into vec[b][col0 + unit] of all C CTAs:
// 4 shuffles gather 4 consecutive units, one 16-byte store per (destination, chunk).
// Remote destinations get st.async (data + complete_tx on the destination's per-source mbarrier). With LOCAL_SELF the
// CTA's own copy does not take the trip through the cluster network (measured: >= 600 cycles from the store to the
// barrier flip even for the own CTA, tools/trace_rec.py): it is written with ordinary st.shared and published with one
// mbarrier.arrive per warp on the own-source barrier (initialised with the warp count instead of a byte count).
// Ordering of the local path: RAW - readers pass mbarrier.try_wait (acquire) on that barrier, which completes only
// after every warp's arrive (release) that follows its st.shared + __syncwarp. WAR - a warp writes buffer b at the end
// of step s; the last readers of b ran in step s-1's contraction, and no warp can leave chunk 0 of step s before all
// NW warps have arrived for step s-1, i.e. finished that contraction.
// PAIRED: the destination uses the batch-paired layout of rnn_core.cuh (paired_index): one 16-byte store carries units
// j and j+4 for the two batch rows of a pair (j % 8 < 4; both land in adjacent k-lanes of the same chunk row).
template <int C, int KL, int UPL, int BS, bool LOCAL_SELF = false, bool PAIRED = false>
__device__ __forceinline__ void allgather_units(float val, float* vec_local, int vstride, int col0,
                                                uint64_t* bar_local, int lane, uint32_t rank = 0) {
  using LM = LaneMap<KL, UPL, BS>;
  constexpr int UPW = LM::UPW;
  constexpr int NCH = UPW * BS / 4;  // 16-byte chunks per destination
  constexpr int NST = C * NCH;
  static_assert(!PAIRED || (UPW % 8 == 0 && BS % 2 == 0), "paired layout: 8 units per store group, even batch slice");
  const uint32_t bar_addr = ptx::smem_u32(bar_local);
#pragma unroll
  for (int it = 0; it < (NST + 31) / 32; ++it) {
    const int idx = it * 32 + lane;
    const bool act = idx < NST;
    const int id2 = act ? idx : 0;
    const int r = id2 / NCH, ch = id2 % NCH;
    float4 v;
    float* dst_ptr;
    if constexpr (PAIRED) {
      const int pr = ch % (BS / 2), ue = ch / (BS / 2);   // batch pair, unit slot (group of 8 units, e = unit % 4)
      const int u = (ue / 4) * 8 + (ue % 4);
      v.x = __shfl_sync(FULLMASK, val, LM::lane_of(u, 2 * pr));
      v.y = __shfl_sync(FULLMASK, val, LM::lane_of(u, 2 * pr + 1));
      v.z = __shfl_sync(FULLMASK, val, LM::lane_of(u + 4, 2 * pr));
      v.w = __shfl_sync(FULLMASK, val, LM::lane_of(u + 4, 2 * pr + 1));
      dst_ptr = &vec_local[paired_index<KL, BS>(col0 + u, 2 * pr)];
    } else {
      const int b = ch / (UPW / 4), quad = ch % (UPW / 4);
      v.x = __shfl_sync(FULLMASK, val, LM::lane_of(quad * 4 + 0, b));
      v.y = __shfl_sync(FULLMASK, val, LM::lane_of(quad * 4 + 1, b));
      v.z = __shfl_sync(FULLMASK, val, LM::lane_of(quad * 4 + 2, b));
      v.w = __shfl_sync(FULLMASK, val, LM::lane_of(quad * 4 + 3, b));
      dst_ptr = &vec_local[b * vstride + col0 + quad * 4];
    }
    if (act) {
      if (LOCAL_SELF && (uint32_t)r == rank) {
        *reinterpret_cast<float4*>(dst_ptr) = v;
      } else {
        const uint32_t dst = ptx::smem_u32(dst_ptr);
        ptx::st_async_v4(ptx::mapa(dst, (uint32_t)r), v, ptx::mapa(bar_addr, (uint32_t)r));
      }
    }
  }
  if (LOCAL_SELF) {
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(bar_local);
  }
}

// =================================================================================================
// forward
// =================================================================================================
// VL = true: per-sequence lengths (PackedSequence semantics): past its length a sequence keeps its state and emits 0
// PB = true: batch-paired FFMA2 contraction and state layout (rnn_core.cuh, dots_chunk2b); used where it measured
// faster (GRU H=256 4-row clusters, LSTM H=256), see launch_rec_fwd
template <int MODE, int H, int C, int BS, int KL, int UPL, int RG, bool VL = false, bool PB = false>
__global__ void __launch_bounds__(RecCfg<MODE, H, C, BS, KL, UPL, RG>::NT, 1)
    rec_fwd_kernel(const RecFwdParams p, const int nslices) {
  using Cfg = RecCfg<MODE, H, C, BS, KL, UPL, RG>;
  using LM = LaneMap<KL, UPL, BS>;
  constexpr int G = Cfg::G, HS = Cfg::HS, NT = Cfg::NT, UPW = Cfg::UPW, NSM = Cfg::NSM, GH = Cfg::GH;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* W_s = reinterpret_cast<float*>(smem_raw);                 // [NSM*HS][H]
  float* h_s = W_s + (size_t)NSM * HS * H;                         // [2][BS][H]
  uint64_t* bars = reinterpret_cast<uint64_t*>(h_s + 2 * BS * H);  // [0] weights, [1 + buf*C + src] state slices
  constexpr int NCH = Cfg::NCH, CPS = Cfg::CPS;

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint32_t rank = ptx::cluster_ctarank();
  const int cid = blockIdx.x / C;
  const int dir = cid / nslices;
  const int slice = cid - dir * nslices;
  const int b0 = slice * BS;
  const int j0 = (int)rank * HS;
  const int B = p.B, T = p.T;
  const float* w_hh = p.w_hh[dir];

  if (tid == 0) {
    // [0]: weights (tx bytes). [1 + buf*C + src]: slice of source CTA `src` - remote sources complete tx bytes
    // (one arrive.expect_tx by thread 0 per phase), the CTA's OWN slice is published by one plain arrive per warp
    for (int i = 0; i < Cfg::NBAR; ++i)
      ptx::mbar_init(&bars[i], (kLocalSelf && i >= 1 && (uint32_t)((i - 1) % C) == rank) ? (uint32_t)Cfg::NW : 1u);
    ptx::fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0) {
    // this CTA's rows of the first NSM gate blocks of W_hh: NSM contiguous [HS,H] blocks, one TMA bulk copy each
    ptx::mbar_arrive_expect_tx(&bars[0], (uint32_t)Cfg::W_BYTES);
#pragma unroll
    for (int g = 0; g < NSM; ++g)
      ptx::tma_bulk_g2s(W_s + (size_t)g * HS * H, w_hh + ((size_t)g * H + j0) * H,
                        (uint32_t)(HS * H * sizeof(float)), &bars[0]);
  }
  for (int i = tid; i < 2 * BS * H; i += NT) h_s[i] = 0.f;  // h_0 = 0 (rnn.py:1432-1440)
  const int rot = Cfg::ROT ? (int)rank * CPS : 0;
  float wreg[RG > 0 ? RG : 1][UPL][H / KL];
  load_resident<RG, KL, UPL, BS, H>(w_hh, H, (long long)NSM * H + j0 + w * UPW, rot, lane, wreg);
  ptx::mbar_wait(&bars[0], 0);
  __syncthreads();
  ptx::cluster_sync_all();  // peers' barriers and state buffers are initialised before anyone writes into them

  // ---- lane identity: after the butterfly this lane owns (unit, batch) ------------------------------
  const int uw = LM::unit(lane), qb = LM::q(lane);
  const int j = j0 + w * UPW + uw;  // hidden unit
  const int b = b0 + qb;            // batch row
  const bool valid = b < B;
  float* gates = p.gates[dir];
  float* extra = p.extra[dir];
  const float bhn = (MODE == B200RNN_GRU) ? p.b_hh[dir][2 * H + j] : 0.f;

  float h_prev = 0.f, c_prev = 0.f, h_sum = 0.f;
  int len_b = T;
  if constexpr (VL) {
    if (valid) len_b = p.lengths[b];
  }
  float gi[G];
#pragma unroll
  for (int g = 0; g < G; ++g) gi[g] = 0.f;
  if (valid && T > 0) {
    const int t0 = dir ? T - 1 : 0;
    const float* gp = gates + ((size_t)t0 * B + b) * GH + j;
#pragma unroll
    for (int g = 0; g < G; ++g) gi[g] = gp[g * H];
  }

  // Global stores of a step (output, saved gates) are DEFERRED into the next step, behind its first chunk: they used to
  // sit between the exchange and the next contraction, i.e. on the serial path of every step (225 cycles).
  float pend_y = 0.f, pend_s0 = 0.f, pend_s1 = 0.f, pend_s2 = 0.f, pend_s3 = 0.f, pend_sx = 0.f;
  auto flush_pending = [&](int tp) {
    if (valid) {
      if (p.y) p.y[(long long)tp * p.y_st + (long long)b * p.y_sb + dir * H + j] = pend_y;
      if (p.training) {
        float* gp = gates + ((size_t)tp * B + b) * GH + j;
        gp[0] = pend_s0;
        gp[H] = pend_s1;
        gp[2 * H] = pend_s2;
        if (G == 4) gp[3 * H] = pend_s3;
        extra[((size_t)tp * B + b) * H + j] = pend_sx;
      }
    }
  };

  for (int step = 0; step < T; ++step) {
    const int t = dir ? (T - 1 - step) : step;
    const int cur = step & 1, nxt = cur ^ 1;
    const float* h_cur = h_s + cur * BS * H;
    float* h_nxt = h_s + nxt * BS * H;
    const uint32_t par = ((step - 1) >> 1) & 1;
#ifdef B200RNN_TRACE
    const bool tr = p.trace != nullptr && blockIdx.x == 0 && lane == 0;  // one row of 8 stamps per (step, warp)
#else
    constexpr bool tr = false;  // build with -DB200RNN_TRACE for the per-phase clock64 timeline (tools/trace_rec.py)
#endif
    long long* trow = p.trace + ((size_t)step * 8 + (w & 7)) * 8;
    if (tr) trow[0] = clock64();

    // FFMA2 (two fp32 FMAs per issue slot) for the GRU only: k-paired (PACK2: float2 = even-k / odd-k partial sums of
    // one output, folded before the butterfly) or batch-paired (PACKB: float2 = two batch rows of one unit, weight as
    // a broadcast 32-bit operand, state kept in the paired shared-memory layout). Measured on the LSTM H=128 forward (same box, round 2):
    // FFMA2 53.6 us vs scalar FFMA 49.5 us per layer - with three distinct 64-bit register operands an FFMA2 issues
    // every 3 cycles (register-file bandwidth), and the 4-gate packed accumulators leave the scheduler less room
    constexpr bool PACKB = PB;
    constexpr bool PACK2 = !PACKB && (MODE == B200RNN_GRU) && RG < 2;
    float2 acc2[PACK2 ? G : 1][UPL][BS];
    float2 acc2b[PACKB ? G : 1][UPL][BS / 2];
    float acc[G][UPL][BS];
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
      for (int au = 0; au < UPL; ++au)
#pragma unroll
        for (int ab = 0; ab < BS; ++ab) {
          acc[g][au][ab] = 0.f;
          if (PACK2) acc2[g][au][ab] = make_float2(0.f, 0.f);
          if (PACKB && ab < BS / 2) acc2b[g][au][ab] = make_float2(0.f, 0.f);
        }
    // contraction over h, one chunk at a time, starting with the slice this CTA produced itself; a chunk is
    // touched only after the slice(s) it belongs to have arrived (per-source mbarriers)
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int ca = (c + rot) % NCH;
      if (step > 0) {
        if (Cfg::ROT) {
          if (c % CPS == 0) ptx::mbar_wait(&bars[1 + cur * C + ca / CPS], par);
        } else {
#pragma unroll
          for (int s2 = 0; s2 < Cfg::SPC; ++s2) ptx::mbar_wait(&bars[1 + cur * C + ca * Cfg::SPC + s2], par);
        }
      }
      if (tr && c < 4) trow[1 + c] = clock64();     // slice of chunk c has arrived (this warp passed its wait)
      if constexpr (PACKB)
        dots_chunk2b<G, RG, KL, UPL, BS, H>(W_s, HS, w * UPW, wreg, h_cur, c, ca, lane, acc2b);
      else if constexpr (PACK2)
        dots_chunk2<G, RG, KL, UPL, BS, H, H>(W_s, HS, w * UPW, wreg, h_cur, c, ca, lane, acc2);
      else
        dots_chunk<G, RG, KL, UPL, BS, H, H>(W_s, HS, w * UPW, wreg, h_cur, c, ca, lane, acc);
      if (c == 0 && step > 0) flush_pending(dir ? (T - step) : (step - 1));  // the previous step's stores
    }
    // every slice of h_step has been consumed by this thread => the barriers of the other buffer are re-armed
    if (tid == 0 && step + 1 < T) {
#pragma unroll
      for (int src = 0; src < C; ++src)
        if (!kLocalSelf || (uint32_t)src != rank)
          ptx::mbar_arrive_expect_tx(&bars[1 + nxt * C + src], (uint32_t)(BS * HS * sizeof(float)));
    }
    if constexpr (PACKB) {
      float red[G];
      warp_transpose_reduce2b<G, KL, UPL, BS>(acc2b, red, lane);
#pragma unroll
      for (int g = 0; g < G; ++g) acc[g][0][0] = red[g];
    } else {
      if constexpr (PACK2) fold_pairs<G, UPL, BS>(acc2, acc);
      warp_transpose_reduce<G, KL, UPL, BS>(acc);
    }
    if (tr) trow[5] = clock64() + (long long)(acc[0][0][0] == 12345.678f);  // butterfly done (value dependence pins it)

    float hnew, s0, s1, s2, s3 = 0.f, sx;
    if (MODE == B200RNN_GRU) {
      const float r = sigmoid_f(gi[0] + acc[0][0][0]);
      const float z = sigmoid_f(gi[1] + acc[1][0][0]);
      const float hn = acc[2][0][0] + bhn;
      const float n = tanh_f(gi[2] + r * hn);
      hnew = n + z * (h_prev - n);
      if constexpr (VL) {
        if (t >= len_b) hnew = h_prev;
      }
      s0 = r; s1 = z; s2 = n; sx = hn;
    } else {
      const float ig = sigmoid_f(gi[0] + acc[0][0][0]);
      const float fg = sigmoid_f(gi[1] + acc[1][0][0]);
      const float gg = tanh_f(gi[2] + acc[2][0][0]);
      const float og = sigmoid_f(gi[G - 1] + acc[G - 1][0][0]);
      float cnew = fg * c_prev + ig * gg;
      hnew = og * tanh_f(cnew);
      if constexpr (VL) {
        if (t >= len_b) {
          cnew = c_prev;
          hnew = h_prev;
        }
      }
      c_prev = cnew;
      s0 = ig; s1 = fg; s2 = gg; s3 = og; sx = cnew;
    }
    h_prev = hnew;
    float yv = hnew;  // what the caller sees at this step
    if constexpr (VL) {
      if (t >= len_b) yv = 0.f;
    }
    h_sum += yv;
    if (tr) trow[6] = clock64() + (long long)(hnew == 12345.678f);          // gate math done

    if (step + 1 < T)
      allgather_units<C, KL, UPL, BS, kLocalSelf, PACKB>(hnew, h_nxt, H, j0 + w * UPW, &bars[1 + nxt * C + rank], lane,
                                                         rank);
    if (tr) trow[7] = clock64();                                            // exchange issued

    // prefetch of the next step's x-projection (long latency, consumed at the next gate math); this step's global
    // stores wait in registers until the next step's first chunk has been issued
    pend_y = yv; pend_s0 = s0; pend_s1 = s1; pend_s2 = s2; pend_s3 = s3; pend_sx = sx;
    if (step == T - 1) flush_pending(t);
    if (valid) {
      if (step == T - 1) {
        p.h_n[((size_t)dir * B + b) * H + j] = hnew;
        if (p.y_pool) p.y_pool[(size_t)b * p.D * H + dir * H + j] = h_sum;
        if (MODE == B200RNN_LSTM && p.c_n) p.c_n[((size_t)dir * B + b) * H + j] = c_prev;
      }
      if (step + 1 < T) {
        const int tn = dir ? (T - 2 - step) : (step + 1);
        const float* gp = gates + ((size_t)tn * B + b) * GH + j;
#pragma unroll
        for (int g = 0; g < G; ++g) gi[g] = gp[g * H];
      }
    }
  }
  ptx::cluster_sync_all();  // nobody exits while a peer could still address its shared memory
}

// =================================================================================================
// backward (BPTT)
// =================================================================================================
// w_prep layout (written by whh_prep_kernel): [C ranks][G][HS][H],
//   w_prep[rank][g][u][jj] = W_hh[g*H + jj][rank*HS + u]
// i.e. for every gate block the transposed slice a CTA needs, contiguous per CTA (TMA bulk copyable).
__global__ void whh_prep_kernel(const float* __restrict__ w_hh, float* __restrict__ out, int G, int H, int C) {
  __shared__ float tile[32][33];
  const int HS = H / C;
  const int tiles_per_g = (H / 32) * (H / 32);
  for (int tix = blockIdx.x; tix < G * tiles_per_g; tix += gridDim.x) {
    const int g = tix / tiles_per_g, rem = tix - g * tiles_per_g;
    const int tj = rem / (H / 32), tk = rem - tj * (H / 32);  // tj: row tile of the gate block, tk: column tile
    for (int i = threadIdx.y; i < 32; i += blockDim.y)
      tile[i][threadIdx.x] = w_hh[((size_t)g * H + tj * 32 + i) * H + tk * 32 + threadIdx.x];
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int col = tk * 32 + i;  // column of W_hh = output unit of the backward contraction
      const int rk = col / HS, u = col - rk * HS;
      out[(((size_t)rk * G + g) * HS + u) * H + tj * 32 + threadIdx.x] = tile[threadIdx.x][i];
    }
    __syncthreads();
  }
}

template <int MODE, int H, int C, int BS, int KL, int UPL, int RG, bool VL = false>
__global__ void __launch_bounds__(RecCfg<MODE, H, C, BS, KL, UPL, RG>::NT, 1)
    rec_bwd_kernel(const RecBwdParams p, const int nslices) {
  using Cfg = RecCfg<MODE, H, C, BS, KL, UPL, RG>;
  using LM = LaneMap<KL, UPL, BS>;
  static_assert(RG <= 1, "the backward kernel keeps at most one gate block in registers");
  // Streamed variant: the last gate block is too large for the register file (H / BS floats per thread, over 64) and
  // is read from global memory (L2: W_hh is small and read by every cluster) in every step instead. Only the LSTM
  // H = 512 backward uses it: there the 16 CTAs of a cluster would each need 256 KB of transposed W_hh on chip.
  constexpr bool STREAM = RG == 1 && UPL * (H / KL) > 64;
  constexpr int G = Cfg::G, GH = Cfg::GH, HS = Cfg::HS, NT = Cfg::NT, UPW = Cfg::UPW, NSM = Cfg::NSM;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* W_s = reinterpret_cast<float*>(smem_raw);   // [NSM][HS][H] transposed gate blocks
  float* d_s = W_s + (size_t)NSM * HS * H;           // [2][BS][G*H] gate gradients of the whole cluster
  uint64_t* bars = reinterpret_cast<uint64_t*>(d_s + 2 * BS * GH);  // [0] weights, [1 + buf*C + src]
  constexpr int NCH = Cfg::NCH, CPS = Cfg::CPS, SPC = Cfg::SPC;

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint32_t rank = ptx::cluster_ctarank();
  const int cid = blockIdx.x / C;
  const int dir = cid / nslices;
  const int slice = cid - dir * nslices;
  const int b0 = slice * BS;
  const int j0 = (int)rank * HS;
  const int B = p.B, T = p.T;
  const float* w_prep = p.w_prep[dir] + (size_t)rank * G * HS * H;

  if (tid == 0) {
    // as in the forward: the own slice is delivered locally (G gate-gradient slices x NW warps arrive per phase)
    for (int i = 0; i < Cfg::NBAR; ++i)
      ptx::mbar_init(&bars[i], (kLocalSelf && i >= 1 && (uint32_t)((i - 1) % C) == rank) ? (uint32_t)(Cfg::NW * G) : 1u);
    ptx::fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0) {
    ptx::mbar_arrive_expect_tx(&bars[0], (uint32_t)Cfg::W_BYTES);
#pragma unroll
    for (int g = 0; g < NSM; ++g)
      ptx::tma_bulk_g2s(W_s + (size_t)g * HS * H, w_prep + (size_t)g * HS * H, (uint32_t)(HS * H * sizeof(float)),
                        &bars[0]);
  }
  for (int i = tid; i < 2 * BS * GH; i += NT) d_s[i] = 0.f;
  const int rot = Cfg::ROT ? (int)rank * CPS : 0;
  float wreg[1][UPL][H / KL];
  if constexpr (!STREAM)
    load_resident<RG, KL, UPL, BS, H>(w_prep + (size_t)NSM * HS * H, HS, (long long)w * UPW, rot, lane, wreg);
  ptx::mbar_wait(&bars[0], 0);
  __syncthreads();
  ptx::cluster_sync_all();

  const int uw = LM::unit(lane), qb = LM::q(lane);
  const int j = j0 + w * UPW + uw;
  const int b = b0 + qb;
  const bool valid = b < B;
  const float* gates = p.gates[dir];
  const float* extra = p.extra[dir];
  float* dgates = p.dgates[dir];

  int len_b = T;
  if constexpr (VL) {
    if (valid) len_b = p.lengths[b];
  }
  float dh_carry = 0.f, dc_carry = 0.f;
  if (valid) {
    if (p.dh_n) dh_carry = p.dh_n[((size_t)dir * B + b) * H + j];
    if (MODE == B200RNN_LSTM && p.dc_n) dc_carry = p.dc_n[((size_t)dir * B + b) * H + j];
  }
  float bsum[G + 1];
#pragma unroll
  for (int g = 0; g <= G; ++g) bsum[g] = 0.f;

  // pooled output (mean / sum over time fused into the caller's graph): every step receives the same gradient row
  const float dy_pooled = (!p.dy && p.dy_pool && valid) ? p.dy_pool[(size_t)b * p.D * H + dir * H + j] * p.dy_scale : 0.f;
  // operands of the current step (prefetched one step ahead)
  float sv[G], sx = 0.f, hp = 0.f, dyv = 0.f;  // saved gates, hn / c_t, h_{prev} / c_{prev}, dy
#pragma unroll
  for (int g = 0; g < G; ++g) sv[g] = 0.f;
  auto load_step = [&](int step) {
    const int t = dir ? step : (T - 1 - step);
    const bool has_prev = step < T - 1;
    const int tp = dir ? t + 1 : t - 1;
    const float* gp = gates + ((size_t)t * B + b) * GH + j;
#pragma unroll
    for (int g = 0; g < G; ++g) sv[g] = gp[g * H];
    sx = extra[((size_t)t * B + b) * H + j];
    dyv = p.dy ? p.dy[(long long)t * p.dy_st + (long long)b * p.dy_sb + dir * H + j] : dy_pooled;
    if (MODE == B200RNN_GRU)
      hp = has_prev ? p.y[(long long)tp * p.y_st + (long long)b * p.y_sb + dir * H + j] : 0.f;
    else
      hp = has_prev ? extra[((size_t)tp * B + b) * H + j] : 0.f;
  };
  if (valid && T > 0) load_step(0);

  for (int step = 0; step < T; ++step) {
    const int t = dir ? step : (T - 1 - step);
    const int buf = step & 1;
    float* d_buf = d_s + buf * BS * GH;
    const bool last = (step == T - 1);
    if (tid == 0 && !last) {
#pragma unroll
      for (int src = 0; src < C; ++src)
        if (!kLocalSelf || (uint32_t)src != rank)
          ptx::mbar_arrive_expect_tx(&bars[1 + buf * C + src], (uint32_t)(BS * G * HS * sizeof(float)));
    }

    // ---- cell backward for (unit j, batch b) ----------------------------------------------------
    float dh = dh_carry + dyv;
    if constexpr (VL) {
      if (t >= len_b) dh = dh_carry;  // the output of a frozen step is the constant 0: its dy reaches nothing
    }
    float dg[G], direct, dhn = 0.f;
    if (MODE == B200RNN_GRU) {
      const float r = sv[0], z = sv[1], n = sv[2], hn = sx;
      const float dn = dh * (1.f - z) * (1.f - n * n);
      const float dz = dh * (hp - n) * z * (1.f - z);
      const float dr = dn * hn * r * (1.f - r);
      dhn = dn * r;
      dg[0] = dr; dg[1] = dz; dg[2] = dn;
      direct = dh * z;
    } else {
      const float ig = sv[0], fg = sv[1], gg = sv[2], og = sv[G - 1];
      const float tc = tanh_f(sx);
      const float dout = dh * tc * og * (1.f - og);
      const float dc = dc_carry + dh * og * (1.f - tc * tc);
      dg[0] = dc * gg * ig * (1.f - ig);
      dg[1] = dc * hp * fg * (1.f - fg);
      dg[2] = dc * ig * (1.f - gg * gg);
      dg[G - 1] = dout;
      const float dc_next = dc * fg;
      direct = 0.f;
      if constexpr (VL) {
        if (t >= len_b) direct = dh;  // frozen step: dh and dc pass straight through
        else dc_carry = dc_next;
      } else {
        dc_carry = dc_next;
      }
    }
    if constexpr (VL) {
      if (t >= len_b) {
#pragma unroll
        for (int g = 0; g < G; ++g) dg[g] = 0.f;
        dhn = 0.f;
        if (MODE == B200RNN_GRU) direct = dh;
      }
    }
    if (valid) {
#pragma unroll
      for (int g = 0; g < G; ++g) bsum[g] += dg[g];
      bsum[G] += dhn;
    }

    if (!last) {
      // all-gather the recurrent-side gate gradient (GRU: n-gate part is dn*r) into every peer CTA
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float v = dg[g];
        if (MODE == B200RNN_GRU && g == 2) v = dhn;
        if (!valid) v = 0.f;
        allgather_units<C, KL, UPL, BS, kLocalSelf>(v, d_buf, GH, g * H + j0 + w * UPW, &bars[1 + buf * C + rank],
                                                    lane, rank);
      }
    }

    if (valid) {
      float* gp = dgates + ((size_t)t * B + b) * GH + j;
#pragma unroll
      for (int g = 0; g < G; ++g) gp[g * H] = dg[g];
      if (MODE == B200RNN_GRU) p.dghn[dir][((size_t)t * B + b) * H + j] = dhn;
    }
    if (last) break;
    if (valid) load_step(step + 1);
    const uint32_t par = (step >> 1) & 1;

    // ---- dh_{prev}[b][j] = direct + sum_col dgh[b][col] * W_hh[col][j], one gate block of columns at a time ----
    // FFMA2: even-k / odd-k partial sums in one float2 accumulator (one issue slot per two FMAs), folded before the
    // butterfly - the scalar FFMA pipe retires one warp instruction per two cycles and SMSP
    float2 acc2[1][UPL][BS];
    float acc[1][UPL][BS];
#pragma unroll
    for (int au = 0; au < UPL; ++au)
#pragma unroll
      for (int ab = 0; ab < BS; ++ab) acc2[0][au][ab] = make_float2(0.f, 0.f);
    // chunk by chunk over the source CTAs (own slice first); a source's G gate-gradient slices share one barrier
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int ca = (c + rot) % NCH;
      if (Cfg::ROT) {
        if (c % CPS == 0) ptx::mbar_wait(&bars[1 + buf * C + ca / CPS], par);
      } else {
#pragma unroll
        for (int s2 = 0; s2 < SPC; ++s2) ptx::mbar_wait(&bars[1 + buf * C + ca * SPC + s2], par);
      }
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (g < NSM)
          dots_chunk2<1, 0, KL, UPL, BS, H, GH>(W_s + (size_t)g * HS * H, 0, w * UPW, wreg, d_buf + g * H, c, ca,
                                                lane, acc2);
        else if constexpr (STREAM)
          dots_chunk2<1, 0, KL, UPL, BS, H, GH>(w_prep + (size_t)NSM * HS * H, 0, w * UPW, wreg, d_buf + g * H, c,
                                                ca, lane, acc2);
        else
          dots_chunk2<1, 1, KL, UPL, BS, H, GH>(W_s, 0, 0, wreg, d_buf + g * H, c, ca, lane, acc2);
      }
    }
    fold_pairs<1, UPL, BS>(acc2, acc);
    warp_transpose_reduce<1, KL, UPL, BS>(acc);
    dh_carry = direct + acc[0][0][0];
  }

  // ---- per-slice bias-gradient partials: sum over this slice's batch rows (the low lane bits) -------------
#pragma unroll
  for (int g = 0; g <= G; ++g) {
    float v = bsum[g];
#pragma unroll
    for (int off = 1; off < BS; off <<= 1) v += __shfl_xor_sync(FULLMASK, v, off);
    bsum[g] = v;
  }
  if (qb == 0) {
    float* out = p.dbias_part[dir] + (size_t)slice * (G + 1) * H;
#pragma unroll
    for (int g = 0; g < G; ++g) out[g * H + j] = bsum[g];
    out[G * H + j] = bsum[G];
  }
  ptx::cluster_sync_all();
}

// =================================================================================================
// launchers
// =================================================================================================
template <typename K>
int prepare_kernel(K kernel, size_t smem, int C) {
  struct Done {
    const void* k;
    int dev;
  };
  static std::mutex mu;  // forward and autograd-backward threads both launch
  static Done done[256];
  static int ndone = 0;
  const int dev = current_device();
  std::lock_guard<std::mutex> lk(mu);
  for (int i = 0; i < ndone; ++i)
    if (done[i].k == (const void*)kernel && done[i].dev == dev) return B200RNN_OK;
  B200_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // clusters above the portable size of 8 (the 16-CTA clusters of H = 512) have to be allowed explicitly
  if (C > 8) B200_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  if (ndone < 256) done[ndone++] = Done{(const void*)kernel, dev};
  return B200RNN_OK;
}

template <typename K, typename P>
int launch_clustered(K kernel, const P& params, int nslices, int nclusters, int C, int NT, size_t smem,
                     cudaStream_t stream, int prof_kind) {
  int rc = prepare_kernel(kernel, smem, C);
  if (rc) return rc;
  ProfScope prof(prof_kind, stream);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(nclusters * C), 1, 1);
  cfg.blockDim = dim3((unsigned)NT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, params, nslices));
  count_launch();
  return B200RNN_OK;
}

// how many clusters of this kernel can be resident at once (cached per kernel)
template <typename K>
int max_active_clusters(K kernel, int C, int NT, size_t smem) {
  struct Entry {
    const void* k;
    int dev, n;
  };
  static std::mutex mu;
  static Entry cache[256];
  static int ncache = 0;
  const int dev = current_device();
  {
    std::lock_guard<std::mutex> lk(mu);
    for (int i = 0; i < ncache; ++i)
      if (cache[i].k == (const void*)kernel && cache[i].dev == dev) return cache[i].n;
  }
  if (prepare_kernel(kernel, smem, C) != B200RNN_OK) return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(C * 148), 1, 1);
  cfg.blockDim = dim3((unsigned)NT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  std::lock_guard<std::mutex> lk(mu);
  if (ncache < 256) cache[ncache++] = Entry{(const void*)kernel, dev, n};
  return n;
}

// A non-portable cluster (C > 8) needs C free SMs in one GPC: a device partitioned below that (MIG, a green context)
// reports room for no cluster at all. Such a launch would fail; report it as unsupported instead.
template <typename K>
bool cluster_fits(K kernel, int C, int NT, size_t smem, int* rc) {
  if (max_active_clusters(kernel, C, NT, smem) > 0) return true;
  set_error("recurrence: this device cannot hold one %d-CTA cluster (%zu B shared memory per CTA)", C, smem);
  *rc = B200RNN_ERR_UNSUPPORTED;
  return false;
}

template <int MODE, int H, int C, int BS, int KL, int UPL, int RG, bool PB = false>
bool try_fwd(const RecFwdParams& p, cudaStream_t s, bool force, int* rc) {
  using Cfg = RecCfg<MODE, H, C, BS, KL, UPL, RG>;
  static_assert(Cfg::FWD_SMEM <= MAX_SMEM, "forward config does not fit an SM");
  auto k = p.lengths ? rec_fwd_kernel<MODE, H, C, BS, KL, UPL, RG, true, PB>
                     : rec_fwd_kernel<MODE, H, C, BS, KL, UPL, RG, false, PB>;
  const int nslices = (p.B + BS - 1) / BS;
  const int nclusters = nslices * p.D;
  static const bool debug = getenv("B200RNN_DEBUG") != nullptr;
  if (debug)
    fprintf(stderr, "[b200rnn] fwd cfg C=%d BS=%d KL=%d UPL=%d RG=%d: need %d clusters, capacity %d, smem %zu\n", C, BS,
            KL, UPL, RG, nclusters, max_active_clusters(k, C, Cfg::NT, Cfg::FWD_SMEM), (size_t)Cfg::FWD_SMEM);
  if (!force && nclusters > max_active_clusters(k, C, Cfg::NT, Cfg::FWD_SMEM)) return false;
  if (C > 8 && !cluster_fits(k, C, Cfg::NT, Cfg::FWD_SMEM, rc)) return true;
  *rc = launch_clustered(k, p, nslices, nclusters, C, Cfg::NT, Cfg::FWD_SMEM, s, PROF_REC_FWD);
  return true;
}

template <int MODE, int H, int C, int BS, int KL, int UPL, int RG>
bool try_bwd(RecBwdParams& p, cudaStream_t s, bool force, int* rc) {
  using Cfg = RecCfg<MODE, H, C, BS, KL, UPL, RG>;
  static_assert(Cfg::BWD_SMEM <= MAX_SMEM, "backward config does not fit an SM");
  auto k = p.lengths ? rec_bwd_kernel<MODE, H, C, BS, KL, UPL, RG, true> : rec_bwd_kernel<MODE, H, C, BS, KL, UPL, RG, false>;
  const int nslices = (p.B + BS - 1) / BS;
  const int nclusters = nslices * p.D;
  if (!force && nclusters > max_active_clusters(k, C, Cfg::NT, Cfg::BWD_SMEM)) return false;
  if (C > 8 && !cluster_fits(k, C, Cfg::NT, Cfg::BWD_SMEM, rc)) return true;
  // transposed, per-CTA contiguous copy of W_hh for this cluster width
  for (int d = 0; d < p.D; ++d) {
    whh_prep_kernel<<<148, dim3(32, 8), 0, s>>>(p.w_hh[d], p.w_prep[d], Cfg::G, H, C);
    if (cudaGetLastError() != cudaSuccess) {
      set_error("whh_prep launch failed");
      *rc = B200RNN_ERR_CUDA;
      return true;
    }
    count_launch();
  }
  p.nslices_out = nslices;
  *rc = launch_clustered(k, p, nslices, nclusters, C, Cfg::NT, Cfg::BWD_SMEM, s, PROF_REC_BWD);
  return true;
}

// Batch-size-aware dispatch (measured on one box, GRU H=256, T=120, per layer launch; profiles/README.md):
//   B = 128 : FFMA <C=4,BS=4> 222 us (215 us with the batch-paired FFMA2 form)
//   B =  64 : FFMA <C=4,BS=4> 215 us (64 CTAs: 43 % of the chip) | FFMA <C=4,BS=2> 175 us (128 CTAs, half the FFMA per step)
//   B <= 48 : FFMA <C=4,BS=4> 209 us | FFMA <C=4,BS=2> 170 us
// so: clusters of 2 batch rows whenever they fit one wave (B <= ~72), clusters of 4 above.
}  // namespace

// smallest BS any backward config uses is 2
int rec_bwd_max_slices(int B) { return (B + 1) / 2; }

// Candidates are ordered by batch rows per cluster; the first one whose clusters are all co-resident
// (one wave => every sequence advances in lock step) wins, else the widest one runs in several waves.
// Template arguments: <MODE, H, C, BS, KL, UPL, RG>.
int launch_rec_fwd(const RecFwdParams& p, cudaStream_t s) {
  int rc = B200RNN_OK;
  if (p.B <= 0 || p.T <= 0) return rc;
  // One tuned config per shape (B200, round-1/2 A/B runs in profiles/README.md) plus a wider-batch fallback that runs
  // in several waves when the batch needs more clusters than fit the chip.
  if (p.mode == B200RNN_GRU && p.H == 256) {
    // half-filled chip (B <= 74, e.g. BASELINE c2 with B = 64): clusters of 2 batch rows use twice the SMs with half the
    // FFMA work per step (all three gate blocks in shared memory, 4 warps per CTA)
    if (p.B <= 74 && try_fwd<B200RNN_GRU, 256, 4, 2, 16, 8, 0>(p, s, false, &rc)) return rc;
    // batch-paired FFMA2 (rnn_core.cuh dots_chunk2b): 215 us at B=128, T=120 against 222 us for the k-paired form on
    // the same box. The same change measured SLOWER for the 2-row clusters (0.408 vs 0.397 ms per 2-layer forward at
    // B=64) and with two gate blocks in registers (0.549 vs 0.539 ms), so only this config uses it.
    if (try_fwd<B200RNN_GRU, 256, 4, 4, 16, 4, 1, true>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_GRU, 256, 8, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_GRU && p.H == 128) {
    if (try_fwd<B200RNN_GRU, 128, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_GRU, 128, 4, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 256) {
    // batch-paired FFMA2: 0.238 vs 0.242 ms per 2-layer BiLSTM forward (B=64, T=30) for the scalar-FFMA form
    if (try_fwd<B200RNN_LSTM, 256, 4, 4, 16, 4, 1, true>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_LSTM, 256, 8, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 128) {
    // scalar FFMA: the batch-paired FFMA2 form measured 0.185 vs 0.180 ms per 2-layer BiLSTM forward (B=128, T=30)
    if (try_fwd<B200RNN_LSTM, 128, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_LSTM, 128, 4, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  // H = 64: the H = 128 configs at half the width (H % (4*KL) == 0 caps KL at 16); W_hh is 48 / 64 KB per direction
  if (p.mode == B200RNN_GRU && p.H == 64) {
    if (try_fwd<B200RNN_GRU, 64, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_GRU, 64, 2, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 64) {
    if (try_fwd<B200RNN_LSTM, 64, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_fwd<B200RNN_LSTM, 64, 2, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  // H = 512: 16-CTA clusters (HS = 32 units per CTA), the largest that exists; nothing wider to fall back to, so the
  // batch runs in as many waves as it needs. GRU: all three gate blocks in shared memory (213 504 B); LSTM: three in
  // shared memory (229 888 B), the fourth in registers (64 floats per thread)
  if (p.mode == B200RNN_GRU && p.H == 512) {
    try_fwd<B200RNN_GRU, 512, 16, 4, 16, 4, 0>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 512) {
    try_fwd<B200RNN_LSTM, 512, 16, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  set_error("recurrence: unsupported (mode=%d, hidden_size=%d); built for hidden_size 64, 128, 256 and 512", p.mode,
            p.H);
  return B200RNN_ERR_UNSUPPORTED;
}

int launch_rec_bwd(RecBwdParams& p, cudaStream_t s) {
  int rc = B200RNN_OK;
  if (p.B <= 0 || p.T <= 0) return rc;
  // K across all 32 lanes with 8 units per lane halves the redundant reads of the [BS][G*H] gradient vector, which
  // (not the weights) dominates the shared-memory traffic of the backward contraction: 303 -> 278 us (GRU H=256)
  if (p.mode == B200RNN_GRU && p.H == 256) {
    if (p.B <= 74 && try_bwd<B200RNN_GRU, 256, 4, 2, 16, 8, 0>(p, s, false, &rc)) return rc;
    if (try_bwd<B200RNN_GRU, 256, 4, 4, 32, 8, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_GRU, 256, 8, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_GRU && p.H == 128) {
    if (try_bwd<B200RNN_GRU, 128, 2, 4, 32, 8, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_GRU, 128, 4, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 256) {
    if (try_bwd<B200RNN_LSTM, 256, 4, 4, 32, 8, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_LSTM, 256, 8, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 128) {
    if (try_bwd<B200RNN_LSTM, 128, 2, 4, 32, 8, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_LSTM, 128, 4, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_GRU && p.H == 64) {
    if (try_bwd<B200RNN_GRU, 64, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_GRU, 64, 2, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 64) {
    if (try_bwd<B200RNN_LSTM, 64, 2, 4, 16, 4, 1>(p, s, false, &rc)) return rc;
    try_bwd<B200RNN_LSTM, 64, 2, 8, 16, 2, 1>(p, s, true, &rc);
    return rc;
  }
  // H = 512, 16-CTA clusters. GRU: two transposed gate blocks in shared memory, one in registers (229 888 B). LSTM: no
  // config holds all four blocks on chip (256 KB per CTA); three sit in shared memory and the fourth is streamed from
  // L2 in every step (rec_bwd_kernel's STREAM variant, 64 KB per CTA per step), 2 batch rows per cluster (229 888 B)
  if (p.mode == B200RNN_GRU && p.H == 512) {
    try_bwd<B200RNN_GRU, 512, 16, 8, 32, 4, 1>(p, s, true, &rc);
    return rc;
  }
  if (p.mode == B200RNN_LSTM && p.H == 512) {
    try_bwd<B200RNN_LSTM, 512, 16, 2, 8, 4, 1>(p, s, true, &rc);
    return rc;
  }
  set_error("recurrence backward: unsupported (mode=%d, hidden_size=%d); built for hidden_size 64, 128, 256 and 512",
            p.mode, p.H);
  return B200RNN_ERR_UNSUPPORTED;
}

}  // namespace b200rnn
