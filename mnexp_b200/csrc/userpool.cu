// User-encoder heads of the cook / sigmoid families that are not a plain GRU: attention pooling over a short sequence of
// vectors, AlphaAdd, strided row adds, and the masked Keras-2.2 LSTM recurrence.
//
// Reference call sites: task/cook.py:158-160 ('iatt': SimpleAttentionMaskSupport()(Masking()(ch))), :177-184 ('atgru':
// the same layer over the two-step sequence [GRU output, id vector]), :185-187 ('algru': models.AlphaAdd,
// models.py:540-554), :161-163 ('ilstm': keras.layers.LSTM), :177-183 ('inagru'); task/paper.py:206-208 ('att').
// Layer arithmetic: models.py:474-489 (a = tanh(x.k + b); e = exp(a) * mask; w = e / (sum e + 1e-7); out = sum_t w_t x_t).
//
// All of it is B x W x D work on a few hundred KB: one CTA per batch row, fixed-order sums (bit-reproducible), parameter
// gradients as per-row partials that lstur_colsum folds in a fixed order.
#include "common.cuh"

namespace lstur {

// ---- attention pooling over W vectors of width D per batch row
__global__ void seq_attn_fwd_kernel(int B, int W, int D, const float* __restrict__ H, const float* __restrict__ m,
                                    const float* __restrict__ kw, const float* __restrict__ bias,
                                    float* __restrict__ out, long long ldo, float* __restrict__ a_out,
                                    float* __restrict__ w_out) {
  extern __shared__ float se[];   // [W]
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wi = tid >> 5, nw = blockDim.x >> 5;
  const float* Hb = H + (long long)b * W * D;
  const float bb = bias[0];
  for (int t = wi; t < W; t += nw) {
    float acc = 0.f;
    for (int k = lane; k < D; k += 32) acc = fmaf(Hb[(long long)t * D + k], kw[k], acc);
    acc = warp_sum(acc);
    if (lane == 0) {
      const float a = tanhf(acc + bb);
      se[t] = expf(a) * m[(long long)b * W + t];
      if (a_out) a_out[(long long)b * W + t] = a;
    }
  }
  __syncthreads();
  float S = 0.f;
  for (int t = 0; t < W; ++t) S += se[t];
  const float inv = 1.f / (S + 1e-7f);
  if (w_out)
    for (int t = tid; t < W; t += blockDim.x) w_out[(long long)b * W + t] = se[t] * inv;
  for (int k = tid; k < D; k += blockDim.x) {
    float acc = 0.f;
    for (int t = 0; t < W; ++t) acc = fmaf(se[t] * inv, Hb[(long long)t * D + k], acc);
    out[(long long)b * ldo + k] = acc;
  }
}

// d w_t = dout . x_t;  c = sum_t w_t d w_t;  d a_t = (d w_t - c) w_t;  d pre_t = d a_t (1 - a_t^2);
// d x_t = keep_t (w_t dout + d pre_t k);  partial[b] = [ sum_t d pre_t x_t (D) | sum_t d pre_t ]
__global__ void seq_attn_bwd_kernel(int B, int W, int D, const float* __restrict__ H, const float* __restrict__ kw,
                                    const float* __restrict__ a_in, const float* __restrict__ w_in,
                                    const float* __restrict__ dout, long long ldd, const float* __restrict__ keep,
                                    float* __restrict__ dH, float* __restrict__ partial) {
  extern __shared__ float sm[];
  float* sdw = sm;         // [W]  d w_t, then d pre_t
  float* sw = sm + W;      // [W]  w_t
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wi = tid >> 5, nw = blockDim.x >> 5;
  const float* Hb = H + (long long)b * W * D;
  const float* db = dout + (long long)b * ldd;
  for (int t = wi; t < W; t += nw) {
    float acc = 0.f;
    for (int k = lane; k < D; k += 32) acc = fmaf(Hb[(long long)t * D + k], db[k], acc);
    acc = warp_sum(acc);
    if (lane == 0) {
      sdw[t] = acc;
      sw[t] = w_in[(long long)b * W + t];
    }
  }
  __syncthreads();
  float c = 0.f;
  for (int t = 0; t < W; ++t) c = fmaf(sw[t], sdw[t], c);
  __syncthreads();
  for (int t = tid; t < W; t += blockDim.x) {
    const float a = a_in[(long long)b * W + t];
    sdw[t] = (sdw[t] - c) * sw[t] * (1.f - a * a);
  }
  __syncthreads();
  for (int k = tid; k < D; k += blockDim.x) {
    const float dk = db[k], kk = kw[k];
    float acc = 0.f;
    for (int t = 0; t < W; ++t) {
      const float kp = keep ? keep[(long long)b * W + t] : 1.f;
      dH[((long long)b * W + t) * D + k] = kp * fmaf(sw[t], dk, sdw[t] * kk);
      acc = fmaf(sdw[t], Hb[(long long)t * D + k], acc);
    }
    partial[(long long)b * (D + 1) + k] = acc;
  }
  if (tid == 0) {
    float acc = 0.f;
    for (int t = 0; t < W; ++t) acc += sdw[t];
    partial[(long long)b * (D + 1) + D] = acc;
  }
}

// mask[r] = any_k(x[r, k] != 0)   (keras Masking())
__global__ void rows_nonzero_kernel(long long rows, int D, const float* __restrict__ x, long long ld, float* __restrict__ mask) {
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  int nz = 0;
  for (int k = lane; k < D; k += 32) nz |= (x[r * ld + k] != 0.f);
  nz = warp_or(nz);
  if (lane == 0) mask[r] = nz ? 1.f : 0.f;
}

// key[b] = first step t with mask[b, t] != 0 (W if the whole row is masked): the sort key that groups batch rows of similar
// history length into the same 32-row tile of the recurrence kernels
__global__ void first_live_step_kernel(int B, int W, const float* __restrict__ m, int* __restrict__ key) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  int first = W;
  for (int t0 = 0; t0 < W && first == W; t0 += 32) {
    const int t = t0 + lane;
    const unsigned bal = __ballot_sync(0xffffffffu, t < W && m[(long long)b * W + t] != 0.f);
    if (bal) first = t0 + __ffs(bal) - 1;
  }
  if (lane == 0) key[b] = first;
}

// out[r, :cols] = bias[:cols] (or 0) for the rows with flags[r] == want   (one warp per row)
__global__ void fill_rows_where_kernel(int rows, int cols, const int* __restrict__ flags, int want,
                                       const float* __restrict__ bias, float* __restrict__ out, long long ld) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows || flags[r] != want) return;
  for (int k = lane; k < cols; k += 32) out[(long long)r * ld + k] = bias ? bias[k] : 0.f;
}

// y[r, :] = ay * y[r, :] + ax * x[r, :]   (strided rows)
__global__ void add_rows_kernel(int rows, int D, float ax, const float* __restrict__ x, long long ldx, float ay,
                                float* __restrict__ y, long long ldy) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int r = (int)(i / D), k = (int)(i % D);
  if (r >= rows) return;
  const float yv = ay == 0.f ? 0.f : ay * y[(long long)r * ldy + k];
  y[(long long)r * ldy + k] = fmaf(ax, x[(long long)r * ldx + k], yv);
}

// models.AlphaAdd (models.py:540-554): out = alpha a + (1 - alpha) b
__global__ void alpha_add_fwd_kernel(int rows, int D, const float* __restrict__ alpha, const float* __restrict__ a,
                                     long long lda, const float* __restrict__ b, long long ldb, float* __restrict__ out,
                                     long long ldo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int r = (int)(i / D), k = (int)(i % D);
  if (r >= rows) return;
  const float al = alpha[0];
  out[(long long)r * ldo + k] = al * a[(long long)r * lda + k] + (1.f - al) * b[(long long)r * ldb + k];
}
// d a = alpha dout, d b = (1 - alpha) dout, row_partial[r] = sum_k dout (a - b)   (one warp per row)
__global__ void alpha_add_bwd_kernel(int rows, int D, const float* __restrict__ alpha, const float* __restrict__ a,
                                     long long lda, const float* __restrict__ b, long long ldb,
                                     const float* __restrict__ dout, long long ldd, float* __restrict__ da,
                                     long long ldda, float* __restrict__ db, long long lddb, float* __restrict__ row_partial) {
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float al = alpha[0];
  float acc = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float g = dout[r * ldd + k];
    da[r * ldda + k] = al * g;
    db[r * lddb + k] = (1.f - al) * g;
    acc = fmaf(g, a[r * lda + k] - b[r * ldb + k], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) row_partial[r] = acc;
}

// keras.constraints.MinMaxNorm(min, max, rate=1, axis=0) on an (n,)-shaped weight: every element is its own norm, so
// w <- w * clip(|w|, min, max) / (1e-7 + |w|)   (applied after the optimizer update, as Keras does)
__global__ void minmaxnorm_kernel(int n, float lo, float hi, float* __restrict__ w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float nr = fabsf(w[i]);
  w[i] = w[i] * (fminf(fmaxf(nr, lo), hi) / (1e-7f + nr));
}

// ---- softmax + keras categorical_crossentropy against integer class labels (the one-hot targets of the auxiliary vertical
// classifier, task/paper.py:899-902, 973-990, and of the vertical model of ...VertAlt, :1128-1136).  One warp per row, any
// class count: p = softmax(logits); q = p / sum p; loss = -log clip(q_label, 1e-7, 1 - 1e-7); the gradient is zero through
// a saturated clip; d logits_k = scale * p_k (g_k - sum_j g_j p_j) with g_label = -1 / q_label.
__global__ void softmax_ce_labels_kernel(long long n, int nc, const float* __restrict__ logits, const int* __restrict__ label,
                                         float* __restrict__ probs, float* __restrict__ loss_rows,
                                         float* __restrict__ dlogits, float scale) {
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= n) return;
  const float* x = logits + r * nc;
  float mx = -INFINITY;
  for (int k = lane; k < nc; k += 32) mx = fmaxf(mx, x[k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float se = 0.f;
  for (int k = lane; k < nc; k += 32) se += expf(x[k] - mx);
  se = warp_sum(se);
  float sp = 0.f;
  for (int k = lane; k < nc; k += 32) sp += expf(x[k] - mx) / se;
  sp = warp_sum(sp);
  int y = label[r];
  if (y < 0 || y >= nc) y = 0;
  const float py = expf(x[y] - mx) / se, qy = py / sp;
  const bool inrange = qy >= 1e-7f && qy <= 1.f - 1e-7f;
  if (lane == 0 && loss_rows) loss_rows[r] = -logf(fminf(fmaxf(qy, 1e-7f), 1.f - 1e-7f));
  const float g = inrange ? -1.f / qy : 0.f, gp = g * py;
  for (int k = lane; k < nc; k += 32) {
    const float p = expf(x[k] - mx) / se;
    if (probs) probs[r * nc + k] = p;
    if (dlogits) dlogits[r * nc + k] = scale * p * ((k == y ? g : 0.f) - gp);
  }
}

// g[i] = y[i] > 0 ? g[i] : 0   (backward of a relu Dense given its output)
__global__ void relu_bwd_kernel(long long n, const float* __restrict__ y, float* __restrict__ g) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(y[i] > 0.f)) g[i] = 0.f;
}

// mean of x (fixed order) into out[0]
__global__ void mean_rows_kernel(long long n, const float* __restrict__ x, float* __restrict__ out) {
  __shared__ float s[256];
  float acc = 0.f;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) acc += x[i];
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = s[0] / (float)n;
}

// ---- masked Keras-2.2 LSTM (task/cook.py:161-163): gate order i, f, c, o; hard_sigmoid recurrent activation;
// c' = f c + i tanh(a_c); h' = o tanh(c'); masked steps carry (h, c); output = last h.  Same thread mapping as the
// streaming GRU kernels (gru.cu): one CTA owns BT batch rows, thread j owns unit j of every row.
constexpr int LSTM_BT = 8;

__device__ __forceinline__ float lstm_act(float x, int act) {
  return act == LSTUR_ACT_HARD_SIGMOID ? hard_sigmoid_f(x) : 1.f / (1.f + expf(-x));
}
__device__ __forceinline__ float lstm_act_grad(float y, int act) {
  return act == LSTUR_ACT_HARD_SIGMOID ? ((y > 0.f && y < 1.f) ? 0.2f : 0.f) : y * (1.f - y);
}

template <int BT>
__device__ __forceinline__ void lstm_fwd_body(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                                              const float* __restrict__ Wh, int act, float* __restrict__ hT, long long ldo,
                                              float* __restrict__ SI, float* __restrict__ SF, float* __restrict__ SG,
                                              float* __restrict__ SO, float* __restrict__ SCP, float* __restrict__ SHP,
                                              float* __restrict__ STC) {
  extern __shared__ float sm[];   // [BT][G] previous h
  const int j = threadIdx.x, b0 = blockIdx.x * BT;
  const bool act_j = j < G;
  const int G4 = 4 * G;
  float h[BT], c[BT];
#pragma unroll
  for (int i = 0; i < BT; ++i) {
    h[i] = 0.f; c[i] = 0.f;
    if (act_j) sm[i * G + j] = 0.f;
  }
  __syncthreads();
  for (int t = 0; t < W; ++t) {
    unsigned mbits = 0;
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B && gm[(long long)b * W + t] != 0.f) mbits |= 1u << i;
    }
    float a[4][BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      bool ok = act_j && b < B && mbits;
#pragma unroll
      for (int q = 0; q < 4; ++q) a[q][i] = ok ? XW[((long long)b * W + t) * G4 + q * G + j] : 0.f;
    }
    if (act_j && mbits) {
      for (int k = 0; k < G; ++k) {
        float w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] = __ldg(Wh + (long long)k * G4 + q * G + j);
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          const float hv = sm[i * G + k];
#pragma unroll
          for (int q = 0; q < 4; ++q) a[q][i] = fmaf(hv, w[q], a[q][i]);
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      const bool on = (mbits >> i) & 1u;
      const float gi = lstm_act(a[0][i], act), gf = lstm_act(a[1][i], act), gg = tanhf(a[2][i]), go = lstm_act(a[3][i], act);
      const float cn = gf * c[i] + gi * gg;
      const float tc = tanhf(cn);
      if (SI && act_j && b < B) {
        long long o = ((long long)b * W + t) * G + j;
        SI[o] = on ? gi : 0.f; SF[o] = on ? gf : 0.f; SG[o] = on ? gg : 0.f; SO[o] = on ? go : 0.f;
        STC[o] = on ? tc : 0.f; SCP[o] = c[i]; SHP[o] = h[i];
      }
      if (on) { c[i] = cn; h[i] = go * tc; }
      if (act_j) sm[i * G + j] = h[i];
    }
    __syncthreads();
  }
  if (act_j) {
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B) hT[(long long)b * ldo + j] = h[i];
    }
  }
}

// BPTT: dA (B,W,4G) in gate order i,f,c,o (zero on masked steps).  WhT = Wh transposed (4G, G).
template <int BT>
__device__ __forceinline__ void lstm_bwd_body(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ SI,
                                              const float* __restrict__ SF, const float* __restrict__ SG,
                                              const float* __restrict__ SO, const float* __restrict__ SCP,
                                              const float* __restrict__ STC, const float* __restrict__ WhT, int act,
                                              const float* __restrict__ dhT, long long lddh, float* __restrict__ dA) {
  extern __shared__ float sm[];   // [4][BT][G] gate pre-activation gradients of this step
  const int k = threadIdx.x, b0 = blockIdx.x * BT;
  const bool act_k = k < G;
  const int G4 = 4 * G;
  float dh[BT], dc[BT];
#pragma unroll
  for (int i = 0; i < BT; ++i) {
    int b = b0 + i;
    dh[i] = (act_k && b < B) ? dhT[(long long)b * lddh + k] : 0.f;
    dc[i] = 0.f;
  }
  for (int t = W - 1; t >= 0; --t) {
    unsigned mbits = 0;
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B && gm[(long long)b * W + t] != 0.f) mbits |= 1u << i;
    }
    float dcp[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      const bool on = act_k && b < B && ((mbits >> i) & 1u);
      const long long o = ((long long)b * W + t) * G + k;
      const float gi = on ? SI[o] : 0.f, gf = on ? SF[o] : 0.f, gg = on ? SG[o] : 0.f, go = on ? SO[o] : 0.f;
      const float tc = on ? STC[o] : 0.f, cp = on ? SCP[o] : 0.f;
      const float dcn = dc[i] + dh[i] * go * (1.f - tc * tc);
      const float dai = on ? dcn * gg * lstm_act_grad(gi, act) : 0.f;
      const float daf = on ? dcn * cp * lstm_act_grad(gf, act) : 0.f;
      const float dag = on ? dcn * gi * (1.f - gg * gg) : 0.f;
      const float dao = on ? dh[i] * tc * lstm_act_grad(go, act) : 0.f;
      dcp[i] = dcn * gf;
      if (act_k) {
        sm[(0 * BT + i) * G + k] = dai; sm[(1 * BT + i) * G + k] = daf;
        sm[(2 * BT + i) * G + k] = dag; sm[(3 * BT + i) * G + k] = dao;
        if (b < B) {
          const long long oa = ((long long)b * W + t) * G4;
          dA[oa + k] = dai; dA[oa + G + k] = daf; dA[oa + 2 * G + k] = dag; dA[oa + 3 * G + k] = dao;
        }
      }
    }
    __syncthreads();
    float dhp[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) dhp[i] = 0.f;
    if (act_k && mbits) {
      for (int q = 0; q < 4; ++q)
        for (int j = 0; j < G; ++j) {
          const float w = __ldg(WhT + (long long)(q * G + j) * G + k);
#pragma unroll
          for (int i = 0; i < BT; ++i) dhp[i] = fmaf(sm[(q * BT + i) * G + j], w, dhp[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < BT; ++i)
      if ((mbits >> i) & 1u) { dh[i] = dhp[i]; dc[i] = dcp[i]; }
    __syncthreads();
  }
}

// Two instances of each kernel, as for the streaming GRU (gru.cu): LSTM_BT = 8 rows per CTA for the widths its register
// count can launch with one thread per unit, the _wide one (4 rows, __launch_bounds__(1024)) for every wider G <= 1024.
constexpr int LSTM_BT_WIDE = 4;

template <int BT>
__global__ void lstm_fwd_kernel(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                                const float* __restrict__ Wh, int act, float* __restrict__ hT, long long ldo,
                                float* __restrict__ SI, float* __restrict__ SF, float* __restrict__ SG,
                                float* __restrict__ SO, float* __restrict__ SCP, float* __restrict__ SHP,
                                float* __restrict__ STC) {
  lstm_fwd_body<BT>(B, W, G, XW, gm, Wh, act, hT, ldo, SI, SF, SG, SO, SCP, SHP, STC);
}
__global__ void __launch_bounds__(1024)
lstm_fwd_kernel_wide(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                     const float* __restrict__ Wh, int act, float* __restrict__ hT, long long ldo, float* __restrict__ SI,
                     float* __restrict__ SF, float* __restrict__ SG, float* __restrict__ SO, float* __restrict__ SCP,
                     float* __restrict__ SHP, float* __restrict__ STC) {
  lstm_fwd_body<LSTM_BT_WIDE>(B, W, G, XW, gm, Wh, act, hT, ldo, SI, SF, SG, SO, SCP, SHP, STC);
}

template <int BT>
__global__ void lstm_bwd_kernel(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ SI,
                                const float* __restrict__ SF, const float* __restrict__ SG, const float* __restrict__ SO,
                                const float* __restrict__ SCP, const float* __restrict__ STC,
                                const float* __restrict__ WhT, int act, const float* __restrict__ dhT, long long lddh,
                                float* __restrict__ dA) {
  lstm_bwd_body<BT>(B, W, G, gm, SI, SF, SG, SO, SCP, STC, WhT, act, dhT, lddh, dA);
}
__global__ void __launch_bounds__(1024)
lstm_bwd_kernel_wide(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ SI,
                     const float* __restrict__ SF, const float* __restrict__ SG, const float* __restrict__ SO,
                     const float* __restrict__ SCP, const float* __restrict__ STC, const float* __restrict__ WhT, int act,
                     const float* __restrict__ dhT, long long lddh, float* __restrict__ dA) {
  lstm_bwd_body<LSTM_BT_WIDE>(B, W, G, gm, SI, SF, SG, SO, SCP, STC, WhT, act, dhT, lddh, dA);
}

}  // namespace lstur

using namespace lstur;

extern "C" int lstur_seq_attn_fwd(int B, int W, int D, const float* H, const float* mask, const float* att_w,
                                  const float* att_b, float* out, long long ldo, float* a_out, float* w_out,
                                  cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && W <= 4096 && D > 0 && H && mask && att_w && att_b && out && ldo >= D, "lstur_seq_attn_fwd");
  if (B == 0) return LSTUR_OK;
  seq_attn_fwd_kernel<<<B, 128, (size_t)W * sizeof(float), stream>>>(B, W, D, H, mask, att_w, att_b, out, ldo, a_out, w_out);
  LSTUR_CHECK_LAUNCH("lstur_seq_attn_fwd");
  return LSTUR_OK;
}

extern "C" int lstur_seq_attn_bwd(int B, int W, int D, const float* H, const float* att_w, const float* a_in,
                                  const float* w_in, const float* dout, long long ldd, const float* keep, float* dH,
                                  float* partial, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && W <= 4096 && D > 0 && H && att_w && a_in && w_in && dout && dH && partial, "lstur_seq_attn_bwd");
  if (B == 0) return LSTUR_OK;
  seq_attn_bwd_kernel<<<B, 128, (size_t)2 * W * sizeof(float), stream>>>(B, W, D, H, att_w, a_in, w_in, dout, ldd, keep, dH, partial);
  LSTUR_CHECK_LAUNCH("lstur_seq_attn_bwd");
  return LSTUR_OK;
}

extern "C" int lstur_rows_nonzero(long long rows, int D, const float* x, long long ld, float* mask, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && D > 0 && (rows == 0 || (x && mask)), "lstur_rows_nonzero");
  if (rows == 0) return LSTUR_OK;
  rows_nonzero_kernel<<<cdiv(rows, 8), 256, 0, stream>>>(rows, D, x, ld, mask);
  LSTUR_CHECK_LAUNCH("lstur_rows_nonzero");
  return LSTUR_OK;
}

extern "C" int lstur_first_live_step(int B, int W, const float* mask, int* key, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && (B == 0 || (mask && key)), "lstur_first_live_step");
  if (B == 0) return LSTUR_OK;
  first_live_step_kernel<<<cdiv(B, 8), 256, 0, stream>>>(B, W, mask, key);
  LSTUR_CHECK_LAUNCH("lstur_first_live_step");
  return LSTUR_OK;
}

extern "C" int lstur_fill_rows_where(int rows, int cols, const int* flags, int want, const float* bias, float* out,
                                     long long ld, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && cols > 0 && (rows == 0 || (flags && out)), "lstur_fill_rows_where");
  if (rows == 0) return LSTUR_OK;
  fill_rows_where_kernel<<<cdiv(rows, 8), 256, 0, stream>>>(rows, cols, flags, want, bias, out, ld);
  LSTUR_CHECK_LAUNCH("lstur_fill_rows_where");
  return LSTUR_OK;
}

extern "C" int lstur_add_rows(int rows, int D, float ax, const float* x, long long ldx, float ay, float* y, long long ldy,
                              cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && D > 0 && (rows == 0 || (x && y)), "lstur_add_rows");
  if (rows == 0) return LSTUR_OK;
  add_rows_kernel<<<cdiv((long long)rows * D, 256), 256, 0, stream>>>(rows, D, ax, x, ldx, ay, y, ldy);
  LSTUR_CHECK_LAUNCH("lstur_add_rows");
  return LSTUR_OK;
}

extern "C" int lstur_alpha_add_fwd(int rows, int D, const float* alpha, const float* a, long long lda, const float* b,
                                   long long ldb, float* out, long long ldo, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && D > 0 && alpha && (rows == 0 || (a && b && out)), "lstur_alpha_add_fwd");
  if (rows == 0) return LSTUR_OK;
  alpha_add_fwd_kernel<<<cdiv((long long)rows * D, 256), 256, 0, stream>>>(rows, D, alpha, a, lda, b, ldb, out, ldo);
  LSTUR_CHECK_LAUNCH("lstur_alpha_add_fwd");
  return LSTUR_OK;
}

extern "C" int lstur_alpha_add_bwd(int rows, int D, const float* alpha, const float* a, long long lda, const float* b,
                                   long long ldb, const float* dout, long long ldd, float* da, long long ldda, float* db,
                                   long long lddb, float* row_partial, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && D > 0 && alpha && (rows == 0 || (a && b && dout && da && db && row_partial)), "lstur_alpha_add_bwd");
  if (rows == 0) return LSTUR_OK;
  alpha_add_bwd_kernel<<<cdiv(rows, 8), 256, 0, stream>>>(rows, D, alpha, a, lda, b, ldb, dout, ldd, da, ldda, db, lddb, row_partial);
  LSTUR_CHECK_LAUNCH("lstur_alpha_add_bwd");
  return LSTUR_OK;
}

extern "C" int lstur_softmax_ce_labels(long long n, int n_classes, const float* logits, const int* label, float* probs,
                                       float* loss_rows, float* loss_mean, float* dlogits, float scale, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && n_classes >= 1 && (n == 0 || (logits && label)), "lstur_softmax_ce_labels");
  LSTUR_REQUIRE(loss_mean == nullptr || loss_rows != nullptr, "lstur_softmax_ce_labels");
  if (n == 0) return LSTUR_OK;
  softmax_ce_labels_kernel<<<cdiv(n, 8), 256, 0, stream>>>(n, n_classes, logits, label, probs, loss_rows, dlogits, scale);
  LSTUR_CHECK_LAUNCH("lstur_softmax_ce_labels");
  if (loss_mean) {
    mean_rows_kernel<<<1, 256, 0, stream>>>(n, loss_rows, loss_mean);
    LSTUR_CHECK_LAUNCH("lstur_softmax_ce_labels(mean)");
  }
  return LSTUR_OK;
}

extern "C" int lstur_relu_bwd(long long n, const float* y, float* g, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && (n == 0 || (y && g)), "lstur_relu_bwd");
  if (n == 0) return LSTUR_OK;
  relu_bwd_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, y, g);
  LSTUR_CHECK_LAUNCH("lstur_relu_bwd");
  return LSTUR_OK;
}

extern "C" int lstur_minmaxnorm(int n, float lo, float hi, float* w, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && lo <= hi && (n == 0 || w), "lstur_minmaxnorm");
  if (n == 0) return LSTUR_OK;
  minmaxnorm_kernel<<<cdiv(n, 128), 128, 0, stream>>>(n, lo, hi, w);
  LSTUR_CHECK_LAUNCH("lstur_minmaxnorm");
  return LSTUR_OK;
}

extern "C" int lstur_lstm_fwd(int B, int W, int G, const float* XW, const float* gm, const float* Wh, int rec_act,
                              float* hT, long long ldo, float* SI, float* SF, float* SG, float* SO, float* SCP, float* SHP,
                              float* STC, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && G > 0 && G <= 1024 && XW && gm && Wh && hT, "lstur_lstm_fwd");
  LSTUR_REQUIRE((SI && SF && SG && SO && SCP && SHP && STC) || (!SI && !SF && !SG && !SO && !SCP && !SHP && !STC), "lstur_lstm_fwd");
  if (B == 0) return LSTUR_OK;
  static const int narrow_max = kernel_max_threads((const void*)lstm_fwd_kernel<LSTM_BT>);
  const int threads = cdiv(G, 32) * 32;
  const int bt = threads <= narrow_max ? LSTM_BT : LSTM_BT_WIDE;
  const void* fn = bt == LSTM_BT ? (const void*)lstm_fwd_kernel<LSTM_BT> : (const void*)lstm_fwd_kernel_wide;
  const size_t smem = (size_t)bt * G * sizeof(float);
  if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (bt == LSTM_BT)
    lstm_fwd_kernel<LSTM_BT><<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, XW, gm, Wh, rec_act, hT, ldo, SI, SF, SG, SO,
                                                                      SCP, SHP, STC);
  else
    lstm_fwd_kernel_wide<<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, XW, gm, Wh, rec_act, hT, ldo, SI, SF, SG, SO, SCP,
                                                                  SHP, STC);
  LSTUR_CHECK_LAUNCH("lstur_lstm_fwd");
  return LSTUR_OK;
}

extern "C" int lstur_lstm_bwd(int B, int W, int G, const float* gm, const float* SI, const float* SF, const float* SG,
                              const float* SO, const float* SCP, const float* STC, const float* WhT, int rec_act,
                              const float* dhT, long long lddh, float* dA, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && G > 0 && G <= 1024 && gm && SI && SF && SG && SO && SCP && STC && WhT && dhT && dA, "lstur_lstm_bwd");
  if (B == 0) return LSTUR_OK;
  static const int narrow_max = kernel_max_threads((const void*)lstm_bwd_kernel<LSTM_BT>);
  const int threads = cdiv(G, 32) * 32;
  const int bt = threads <= narrow_max ? LSTM_BT : LSTM_BT_WIDE;
  const void* fn = bt == LSTM_BT ? (const void*)lstm_bwd_kernel<LSTM_BT> : (const void*)lstm_bwd_kernel_wide;
  const size_t smem = (size_t)4 * bt * G * sizeof(float);
  if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (bt == LSTM_BT)
    lstm_bwd_kernel<LSTM_BT><<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, gm, SI, SF, SG, SO, SCP, STC, WhT, rec_act, dhT,
                                                                      lddh, dA);
  else
    lstm_bwd_kernel_wide<<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, gm, SI, SF, SG, SO, SCP, STC, WhT, rec_act, dhT, lddh,
                                                                  dA);
  LSTUR_CHECK_LAUNCH("lstur_lstm_bwd");
  return LSTUR_OK;
}
