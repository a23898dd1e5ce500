// rnn_kernels.cuh — host-side launch interface of the persistent recurrence kernels (K2-K5).
#pragma once
#include "common.cuh"

namespace b200rnn {

// One launch runs ALL directions of one layer: grid = D * nslices clusters of C CTAs.
struct RecFwdParams {
  int mode, B, T, H, D;
  int training;              // save activated gates + hn/c for backward
  const float* w_hh[2];      // per direction [G*H, H]
  const float* b_hh[2];      // per direction [G*H]  (GRU: only the n third is read; r,z are pre-folded)
  float* gates[2];           // per direction [T,B,G*H]; in: x-projection + folded biases; out: activated gates
  float* extra[2];           // per direction [T,B,H]; GRU: W_hn h + b_hn ; LSTM: c_t   (training only)
  float* y;                  // layer output, element (t,b,d*H+j) at t*y_st + b*y_sb + d*H + j (NULL: not written)
  long long y_st, y_sb;
  float* y_pool;             // optional [B, D*H]: sum over t of the layer output (fused pooling epilogue)
  float* h_n;                // [D,B,H] of this layer
  float* c_n;                // [D,B,H] of this layer (LSTM) or NULL
  long long* trace;          // debug: per-step phase timestamps of CTA 0 / warp 0 (NULL = off), [T][8]
  const int* lengths;        // optional [B]: valid steps per sequence (PackedSequence semantics); NULL = all T
};

struct RecBwdParams {
  int mode, B, T, H, D;
  const float* w_hh[2];      // per direction weight_hh [G*H, H]
  float* w_prep[2];          // per direction scratch, G*H*H floats: per-CTA transposed slices (filled by the launcher)
  const float* gates[2];     // saved activated gates [T,B,G*H]
  const float* extra[2];     // GRU hn / LSTM c, [T,B,H]
  const float* y;            // this layer's forward output (h_t), strided
  long long y_st, y_sb;
  const float* dy;           // gradient of this layer's output, strided (NULL: use dy_pool)
  long long dy_st, dy_sb;
  const float* dy_pool;      // [B, D*H]: gradient of the time-POOLED output, broadcast over the steps inside the kernel
  float dy_scale;            //           (x dy_scale): the [T,B,D*H] gradient of a mean / sum over time never exists
  const float* dh_n;         // [D,B,H] or NULL
  const float* dc_n;         // [D,B,H] or NULL
  float* dgates[2];          // out: [T,B,G*H] gradient w.r.t. the x-projection (dGi)
  float* dghn[2];            // out (GRU only): [T,B,H] gradient w.r.t. (W_hn h + b_hn) = dn * r
  float* dbias_part[2];      // out: [nslices][(G+1)*H] per-slice column sums (rows 0..G*H: dGi; GRU tail H: dghn)
  int nslices_out;           // filled by the launcher
  const int* lengths;        // optional [B], as in the forward
};

// number of batch slices the launcher will use for this shape (needed to size dbias_part)
int rec_bwd_max_slices(int B);

int launch_rec_fwd(const RecFwdParams& p, cudaStream_t stream);
int launch_rec_bwd(RecBwdParams& p, cudaStream_t stream);

}  // namespace b200rnn
