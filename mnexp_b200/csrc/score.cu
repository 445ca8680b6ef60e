// Dot-product click scorer + (1+K)-way softmax + Keras categorical cross-entropy, fused fwd+bwd;
// and the sigmoid scoring head of the test model.
//
// Reference: _score_model 'dot' task/paper.py:446-447; softmax over the concatenated
// logits :460-464; loss=keras.losses.categorical_crossentropy :657 — on probabilities:
// p <- p/sum(p); p <- clip(p,1e-7,1-1e-7); l = -sum_j y_j log p_j; mean over batch [K]
// (SURVEY.md §9.5-9.6).  Test head: sigmoid(score) task/paper.py:661-665.
#include "common.cuh"

namespace lstur {

// One warp per batch row; lane c owns candidate c (C <= 32).
__global__ void score_softmax_ce_kernel(int B, int C, int D, const float* __restrict__ u, long long ldu,
                                        const float* __restrict__ d, long long ldd, const float* __restrict__ label,
                                        float* __restrict__ logits, float* __restrict__ probs,
                                        float* __restrict__ loss_rows, float* __restrict__ du, long long lddu,
                                        float* __restrict__ dd, long long lddd, float grad_scale) {
  int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* ub = u + (long long)b * ldu;
  float s_mine = -INFINITY;
  for (int c = 0; c < C; ++c) {
    const float* dc = d + ((long long)b * C + c) * ldd;
    float acc = 0.f;
    for (int k = lane; k < D; k += 32) acc = fmaf(ub[k], dc[k], acc);
    acc = warp_sum(acc);
    if (lane == c) s_mine = acc;
  }
  float mx = s_mine;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float e = lane < C ? expf(s_mine - mx) : 0.f;
  float p = e / warp_sum(e);
  float y = lane < C ? (label ? label[(long long)b * C + lane] : (lane == 0 ? 1.f : 0.f)) : 0.f;
  float q = p / warp_sum(p);  // keras renormalises before the clip
  bool inrange = (q >= 1e-7f) && (q <= 1.f - 1e-7f);
  float qc = fminf(fmaxf(q, 1e-7f), 1.f - 1e-7f);
  float l = lane < C ? -y * logf(qc) : 0.f;
  l = warp_sum(l);
  if (lane < C) {
    if (logits) logits[(long long)b * C + lane] = s_mine;
    if (probs) probs[(long long)b * C + lane] = p;
  }
  if (lane == 0 && loss_rows) loss_rows[b] = l;
  if (!du) return;
  // g_j = dL/dp_j = -y_j/p_j inside the clip range, else 0;  ds_k = p_k (g_k - sum_j g_j p_j)
  float g = (lane < C && inrange && y != 0.f) ? -y / q : 0.f;
  float gp = warp_sum(g * p);
  float ds = lane < C ? p * (g - gp) * grad_scale : 0.f;
  float* dub = du + (long long)b * lddu;
  for (int k0 = 0; k0 < D; k0 += 32) {
    int k = k0 + lane;
    float uk = k < D ? ub[k] : 0.f, acc = 0.f;
    for (int c = 0; c < C; ++c) {
      float dsc = __shfl_sync(0xffffffffu, ds, c);
      if (k < D) {
        acc = fmaf(dsc, d[((long long)b * C + c) * ldd + k], acc);
        dd[((long long)b * C + c) * lddd + k] = dsc * uk;
      }
    }
    if (k < D) dub[k] = acc;
  }
}

// out[i] = sigmoid(u[row(i)] . d[i]),  row(i) = i / C.  One warp per pair.
__global__ void score_sigmoid_kernel(long long n, int C, int D, const float* __restrict__ u, long long ldu,
                                     const float* __restrict__ d, long long ldd, float* __restrict__ out,
                                     int apply_sigmoid) {
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float* ub = u + (i / C) * ldu;
  const float* di = d + i * ldd;
  float acc = 0.f;
  for (int k = lane; k < D; k += 32) acc = fmaf(ub[k], di[k], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[i] = apply_sigmoid ? 1.f / (1.f + expf(-acc)) : acc;
}

// Ragged test head: one warp per pair j, out[j] = sigmoid(u[pair_row[j]] . d[pair_doc ? pair_doc[j] : j]); the sum runs
// in the lane order of score_sigmoid_kernel.
__global__ void score_sigmoid_ragged_kernel(long long n, int D, const int* __restrict__ pair_row, const float* __restrict__ u,
                                            long long ldu, const int* __restrict__ pair_doc, const float* __restrict__ d,
                                            long long ldd, float* __restrict__ out) {
  const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= n) return;
  const float* ub = u + (long long)pair_row[j] * ldu;
  const float* dj = d + (pair_doc ? (long long)pair_doc[j] : j) * ldd;
  float acc = 0.f;
  for (int k = lane; k < D; k += 32) acc = fmaf(ub[k], dj[k], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[j] = 1.f / (1.f + expf(-acc));
}
// CSR offsets (n_rows + 1, starting anywhere) -> row_of[j - offsets[0]] = the row that pair j belongs to; one warp per row
__global__ void csr_rows_kernel(int n_rows, const int* __restrict__ offsets, int* __restrict__ row_of) {
  const int r = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const int base = offsets[0], e = offsets[r + 1] - base;
  for (int j = offsets[r] - base + lane; j < e; j += 32) row_of[j] = r;
}

__global__ void mean_kernel(int n, const float* __restrict__ x, float* __restrict__ out) {
  __shared__ float s[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += x[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) out[0] = v / (float)n;
  }
}


// Per-impression ranking metrics (task/paper.py:497-524 via utils.py:106-124 and sklearn roc_auc_score): one CTA per
// impression, O(C^2) rank counting (C = candidates of the impression, a few hundred at most).  Order = descending score,
// ties by descending index (np.argsort(s)[::-1] with a stable sort).  out[i] = {auc, ndcg@10, ndcg@5, mrr}; an impression
// without a positive or without a negative yields NaN where the host formulas divide by zero.
__global__ void ranking_metrics_kernel(int n_impr, const int* __restrict__ offsets, const float* __restrict__ scores,
                                       const float* __restrict__ labels, float* __restrict__ out) {
  const int imp = blockIdx.x;
  if (imp >= n_impr) return;
  const int beg = offsets[imp], C = offsets[imp + 1] - beg;
  const float* s = scores + beg;
  const float* y = labels + beg;
  double auc_num = 0.0, dcg10 = 0.0, dcg5 = 0.0, idcg10 = 0.0, idcg5 = 0.0, rr = 0.0, ysum = 0.0, npos = 0.0, nneg = 0.0;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    const float si = s[i], yi = y[i];
    int rank = 0, irank = 0;          // position in the score order / in the ideal (label) order
    double wins = 0.0;
    for (int j = 0; j < C; ++j) {
      const float sj = s[j], yj = y[j];
      rank += (sj > si) || (sj == si && j > i);
      irank += (yj > yi) || (yj == yi && j > i);
      if (yi > 0.f && !(yj > 0.f)) wins += si > sj ? 1.0 : (si == sj ? 0.5 : 0.0);
    }
    const double gain = exp2((double)yi) - 1.0;
    if (rank < 10) dcg10 += gain / log2((double)rank + 2.0);
    if (rank < 5) dcg5 += gain / log2((double)rank + 2.0);
    if (irank < 10) idcg10 += gain / log2((double)irank + 2.0);
    if (irank < 5) idcg5 += gain / log2((double)irank + 2.0);
    rr += (double)yi / ((double)rank + 1.0);
    ysum += (double)yi;
    if (yi > 0.f) { npos += 1.0; auc_num += wins; } else { nneg += 1.0; }
  }
  __shared__ double red[9][32];
  double vals[9] = {auc_num, dcg10, dcg5, idcg10, idcg5, rr, ysum, npos, nneg};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    double v = vals[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t[9];
    const int nw = blockDim.x >> 5;
    for (int k = 0; k < 9; ++k) {
      t[k] = 0.0;
      for (int w = 0; w < nw; ++w) t[k] += red[k][w];
    }
    out[4 * imp + 0] = (float)(t[0] / (t[7] * t[8]));
    out[4 * imp + 1] = (float)(t[1] / t[3]);
    out[4 * imp + 2] = (float)(t[2] / t[4]);
    out[4 * imp + 3] = (float)(t[5] / t[6]);
  }
}

// ---- 'dnn' / 'ddot' scorers (task/paper.py:448-455, task/cook.py:206-209) and the masked mean of 'niavg'
// (models.py:422-441): small row-wise kernels around the dense GEMMs.

// out[(b,c)] = [u[b] (U) ‖ d[(b,c)] (D)]
// pair_row (nullable): the user row of pair i comes from a ragged list (pair_row[i]) instead of i / C
__global__ void pair_concat_kernel(long long n_pairs, int C, int U, int D, const float* __restrict__ u, long long ldu,
                                   const float* __restrict__ d, long long ldd, float* __restrict__ out,
                                   const int* __restrict__ pair_row) {
  const int K = U + D;
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / K;
  const int k = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) % K);
  if (i >= n_pairs) return;
  const long long r = pair_row ? (long long)pair_row[i] : i / C;
  out[i * K + k] = k < U ? u[r * ldu + k] : d[i * ldd + (k - U)];
}
// du[b] = sum_c dcat[(b,c), :U] (fixed order);  dd[(b,c)] = dcat[(b,c), U:]
__global__ void pair_split_kernel(int B, int C, int U, int D, const float* __restrict__ dcat, float* __restrict__ du,
                                  long long lddu, float* __restrict__ dd, long long lddd) {
  const int K = U + D;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / K), k = (int)(idx % K);
  if (b >= B) return;
  if (k < U) {
    float acc = 0.f;
    for (int c = 0; c < C; ++c) acc += dcat[((long long)b * C + c) * K + k];
    du[(long long)b * lddu + k] = acc;
  } else {
    for (int c = 0; c < C; ++c) dd[((long long)b * C + c) * lddd + (k - U)] = dcat[((long long)b * C + c) * K + k];
  }
}
// out[i] = h[i] . w + bias[0]; one warp per row
__global__ void rowdot_bias_kernel(long long n, int H, const float* __restrict__ h, const float* __restrict__ w,
                                   const float* __restrict__ bias, float* __restrict__ out) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  float acc = 0.f;
  for (int k = lane; k < H; k += 32) acc = fmaf(h[i * H + k], w[k], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[i] = acc + (bias ? bias[0] : 0.f);
}
// backward of  logit = relu_hid . w2 + b2:  dhid = (hid > 0) dl w2;  whid = dl hid (column sums = d w2)
__global__ void dnn_out_bwd_kernel(long long n, int H, const float* __restrict__ hid, const float* __restrict__ w2,
                                   const float* __restrict__ dl, float* __restrict__ dhid, float* __restrict__ whid) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * H) return;
  const long long i = idx / H;
  const int k = (int)(idx % H);
  const float hv = hid[idx], g = dl[i];
  dhid[idx] = hv > 0.f ? g * w2[k] : 0.f;
  whid[idx] = g * hv;
}
__global__ void fill_kernel(long long n, float v, float* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}
__global__ void tanh_fwd_kernel(long long n, float* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = tanhf(x[i]);
}
__global__ void tanh_bwd_kernel(long long n, const float* __restrict__ y, float* __restrict__ g) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) g[i] *= 1.f - y[i] * y[i];
}
// GlobalAveragePoolingMaskSupport: out[b] = sum_t H[b,t,:] / (sum_t m[b,t] + 1e-7)
__global__ void masked_mean_fwd_kernel(int B, int W, int D, const float* __restrict__ H, const float* __restrict__ m,
                                       float* __restrict__ out, long long ldo) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / D), k = (int)(idx % D);
  if (b >= B) return;
  float acc = 0.f, cnt = 0.f;
  for (int t = 0; t < W; ++t) {
    acc += H[((long long)b * W + t) * D + k];
    cnt += m[(long long)b * W + t];
  }
  out[(long long)b * ldo + k] = acc / (cnt + 1e-7f);
}
// dH[b,t,:] = keep[b,t] * dout[b] / (sum_t m[b,t] + 1e-7)   (keep = the history mask multiplied in before the layer)
__global__ void masked_mean_bwd_kernel(int B, int W, int D, const float* __restrict__ dout, long long ldd,
                                       const float* __restrict__ m, const float* __restrict__ keep,
                                       float* __restrict__ dH) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / D), k = (int)(idx % D);
  if (b >= B) return;
  float cnt = 0.f;
  for (int t = 0; t < W; ++t) cnt += m[(long long)b * W + t];
  const float g = dout[(long long)b * ldd + k] / (cnt + 1e-7f);
  for (int t = 0; t < W; ++t) dH[((long long)b * W + t) * D + k] = keep[(long long)b * W + t] * g;
}

// ---- sigmoid-family head (Seq2VecPaper / Seq2VecPaperDot / Seq2VecPaperId, task/paper.py:222-262): p = sigmoid(s) and
// the weighted binary cross-entropy Seq2Vec.loss (task/seq2vec.py:213-216):
//   L = -0.5 (1+K) mean_i [ y_i log(p_i + 1e-8) gain + (1 - y_i) log(1 - p_i + 1e-8) / K ]
__global__ void bce_fwd_kernel(long long n, const float* __restrict__ s, const float* __restrict__ y, float gain, float K,
                               float* __restrict__ p_out, float* __restrict__ loss_rows) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float p = 1.f / (1.f + expf(-s[i]));
  if (p_out) p_out[i] = p;
  if (loss_rows) loss_rows[i] = -0.5f * (1.f + K) * (y[i] * logf(p + 1e-8f) * gain + (1.f - y[i]) * logf(1.f - p + 1e-8f) / K);
}
// ds_i = grad_scale * dL_i/dp_i * p (1 - p)
__global__ void bce_bwd_kernel(long long n, const float* __restrict__ s, const float* __restrict__ y, float gain, float K,
                               float grad_scale, float* __restrict__ ds) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float p = 1.f / (1.f + expf(-s[i]));
  const float dp = -0.5f * (1.f + K) * (y[i] * gain / (p + 1e-8f) - (1.f - y[i]) / (K * (1.f - p + 1e-8f)));
  ds[i] = grad_scale * dp * p * (1.f - p);
}
// backward of s[(b,c)] = u[b] . d[(b,c)]:  du[b] = sum_c ds d (fixed order), dd[(b,c)] = ds u[b]
__global__ void dot_score_bwd_kernel(int B, int C, int D, const float* __restrict__ u, long long ldu,
                                     const float* __restrict__ d, long long ldd, const float* __restrict__ ds,
                                     float* __restrict__ du, long long lddu, float* __restrict__ dd, long long lddd) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / D), k = (int)(idx % D);
  if (b >= B) return;
  const float uk = u[(long long)b * ldu + k];
  float acc = 0.f;
  for (int c = 0; c < C; ++c) {
    const float g = ds[(long long)b * C + c];
    acc = fmaf(g, d[((long long)b * C + c) * ldd + k], acc);
    dd[((long long)b * C + c) * lddd + k] = g * uk;
  }
  du[(long long)b * lddu + k] = acc;
}

}  // namespace lstur

using namespace lstur;

// u (B,D) ld=ldu; d (B*C, D) ld=ldd; label (B,C) or NULL (positive = column 0).
// du/dd may be NULL for forward only.  grad_scale = 1/global_batch.
extern "C" int lstur_score_softmax_ce(int B, int C, int D, const float* u, long long ldu, const float* d, long long ldd,
                                      const float* label, float* logits, float* probs, float* loss_rows,
                                      float* loss_mean, float* du, long long lddu, float* dd, long long lddd,
                                      float grad_scale, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && C >= 1 && C <= 32 && D > 0, "lstur_score_softmax_ce");
  LSTUR_REQUIRE((du == nullptr) == (dd == nullptr), "lstur_score_softmax_ce");
  LSTUR_REQUIRE(loss_mean == nullptr || loss_rows != nullptr, "lstur_score_softmax_ce");
  if (B == 0) return LSTUR_OK;
  score_softmax_ce_kernel<<<cdiv((long long)B * 32, 128), 128, 0, stream>>>(B, C, D, u, ldu, d, ldd, label, logits, probs,
                                                                          loss_rows, du, lddu, dd, lddd, grad_scale);
  LSTUR_CHECK_LAUNCH("lstur_score_softmax_ce");
  if (loss_mean) {
    mean_kernel<<<1, 256, 0, stream>>>(B, loss_rows, loss_mean);
    LSTUR_CHECK_LAUNCH("lstur_score_softmax_ce(mean)");
  }
  return LSTUR_OK;
}

extern "C" int lstur_score_sigmoid(long long n_pairs, int C, int D, const float* u, long long ldu, const float* d,
                                   long long ldd, float* out, int apply_sigmoid, cudaStream_t stream) {
  LSTUR_REQUIRE(n_pairs >= 0 && C >= 1 && D > 0, "lstur_score_sigmoid");
  if (n_pairs == 0) return LSTUR_OK;
  score_sigmoid_kernel<<<cdiv(n_pairs * 32, 256), 256, 0, stream>>>(n_pairs, C, D, u, ldu, d, ldd, out, apply_sigmoid);
  LSTUR_CHECK_LAUNCH("lstur_score_sigmoid");
  return LSTUR_OK;
}

// AUC / nDCG@10 / nDCG@5 / MRR of every impression (offsets: n_impr+1 prefix sums into scores / labels), the evaluation
// loop of Seq2VecPaperSoftmax.callback (task/paper.py:497-524).  out: (n_impr, 4).
extern "C" int lstur_ranking_metrics(int n_impr, const int* offsets, const float* scores, const float* labels, float* out,
                                     cudaStream_t stream) {
  LSTUR_REQUIRE(n_impr >= 0 && (n_impr == 0 || (offsets && scores && labels && out)), "lstur_ranking_metrics");
  if (n_impr == 0) return LSTUR_OK;
  ranking_metrics_kernel<<<n_impr, 128, 0, stream>>>(n_impr, offsets, scores, labels, out);
  LSTUR_CHECK_LAUNCH("lstur_ranking_metrics");
  return LSTUR_OK;
}

extern "C" int lstur_score_sigmoid_ragged(long long n_pairs, int D, const int* pair_row, const float* u, long long ldu,
                                          const int* pair_doc, const float* d, long long ldd, float* out,
                                          cudaStream_t stream) {
  LSTUR_REQUIRE(n_pairs >= 0 && D > 0 && (n_pairs == 0 || (pair_row && u && d && out)), "lstur_score_sigmoid_ragged");
  if (n_pairs == 0) return LSTUR_OK;
  score_sigmoid_ragged_kernel<<<cdiv(n_pairs * 32, 256), 256, 0, stream>>>(n_pairs, D, pair_row, u, ldu, pair_doc, d, ldd,
                                                                            out);
  LSTUR_CHECK_LAUNCH("lstur_score_sigmoid_ragged");
  return LSTUR_OK;
}
extern "C" int lstur_csr_rows(int n_rows, const int* offsets, int* row_of, cudaStream_t stream) {
  LSTUR_REQUIRE(n_rows >= 0 && (n_rows == 0 || (offsets && row_of)), "lstur_csr_rows");
  if (n_rows == 0) return LSTUR_OK;
  csr_rows_kernel<<<cdiv((long long)n_rows * 32, 256), 256, 0, stream>>>(n_rows, offsets, row_of);
  LSTUR_CHECK_LAUNCH("lstur_csr_rows");
  return LSTUR_OK;
}

extern "C" int lstur_pair_concat(long long n_pairs, int C, int U, int D, const float* u, long long ldu, const float* d,
                                 long long ldd, float* out, const int* pair_row, cudaStream_t stream) {
  LSTUR_REQUIRE(n_pairs >= 0 && C >= 1 && U > 0 && D > 0 && u && d && out, "lstur_pair_concat");
  if (n_pairs == 0) return LSTUR_OK;
  pair_concat_kernel<<<cdiv(n_pairs * (U + D), 256), 256, 0, stream>>>(n_pairs, C, U, D, u, ldu, d, ldd, out, pair_row);
  LSTUR_CHECK_LAUNCH("lstur_pair_concat");
  return LSTUR_OK;
}
extern "C" int lstur_pair_split(int B, int C, int U, int D, const float* dcat, float* du, long long lddu, float* dd,
                                long long lddd, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && C >= 1 && U > 0 && D > 0 && dcat && du && dd, "lstur_pair_split");
  if (B == 0) return LSTUR_OK;
  pair_split_kernel<<<cdiv((long long)B * (U + D), 256), 256, 0, stream>>>(B, C, U, D, dcat, du, lddu, dd, lddd);
  LSTUR_CHECK_LAUNCH("lstur_pair_split");
  return LSTUR_OK;
}
extern "C" int lstur_rowdot_bias(long long n, int H, const float* h, const float* w, const float* bias, float* out,
                                 cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && H > 0 && h && w && out, "lstur_rowdot_bias");
  if (n == 0) return LSTUR_OK;
  rowdot_bias_kernel<<<cdiv(n * 32, 256), 256, 0, stream>>>(n, H, h, w, bias, out);
  LSTUR_CHECK_LAUNCH("lstur_rowdot_bias");
  return LSTUR_OK;
}
extern "C" int lstur_dnn_out_bwd(long long n, int H, const float* hid, const float* w2, const float* dlogit, float* dhid,
                                 float* whid, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && H > 0 && hid && w2 && dlogit && dhid && whid, "lstur_dnn_out_bwd");
  if (n == 0) return LSTUR_OK;
  dnn_out_bwd_kernel<<<cdiv(n * H, 256), 256, 0, stream>>>(n, H, hid, w2, dlogit, dhid, whid);
  LSTUR_CHECK_LAUNCH("lstur_dnn_out_bwd");
  return LSTUR_OK;
}
extern "C" int lstur_tanh_fwd(long long n, float* x, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && (n == 0 || x), "lstur_tanh_fwd");
  if (n == 0) return LSTUR_OK;
  tanh_fwd_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, x);
  LSTUR_CHECK_LAUNCH("lstur_tanh_fwd");
  return LSTUR_OK;
}
extern "C" int lstur_tanh_bwd(long long n, const float* y, float* g, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && (n == 0 || (y && g)), "lstur_tanh_bwd");
  if (n == 0) return LSTUR_OK;
  tanh_bwd_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, y, g);
  LSTUR_CHECK_LAUNCH("lstur_tanh_bwd");
  return LSTUR_OK;
}
extern "C" int lstur_masked_mean_fwd(int B, int W, int D, const float* H, const float* mask, float* out, long long ldo,
                                     cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && D > 0 && H && mask && out, "lstur_masked_mean_fwd");
  if (B == 0) return LSTUR_OK;
  masked_mean_fwd_kernel<<<cdiv((long long)B * D, 256), 256, 0, stream>>>(B, W, D, H, mask, out, ldo);
  LSTUR_CHECK_LAUNCH("lstur_masked_mean_fwd");
  return LSTUR_OK;
}
extern "C" int lstur_masked_mean_bwd(int B, int W, int D, const float* dout, long long ldd, const float* mask,
                                     const float* keep, float* dH, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && D > 0 && dout && mask && keep && dH, "lstur_masked_mean_bwd");
  if (B == 0) return LSTUR_OK;
  masked_mean_bwd_kernel<<<cdiv((long long)B * D, 256), 256, 0, stream>>>(B, W, D, dout, ldd, mask, keep, dH);
  LSTUR_CHECK_LAUNCH("lstur_masked_mean_bwd");
  return LSTUR_OK;
}
extern "C" int lstur_fill(long long n, float v, float* x, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && (n == 0 || x), "lstur_fill");
  if (n == 0) return LSTUR_OK;
  fill_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, v, x);
  LSTUR_CHECK_LAUNCH("lstur_fill");
  return LSTUR_OK;
}

extern "C" int lstur_bce_loss(long long n, const float* scores, const float* label, float gain, int negative_samples,
                              float* probs, float* loss_rows, float* loss_mean, float* dscores, float grad_scale,
                              cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && negative_samples >= 1 && (n == 0 || (scores && label)), "lstur_bce_loss");
  LSTUR_REQUIRE(loss_mean == nullptr || loss_rows != nullptr, "lstur_bce_loss");
  if (n == 0) return LSTUR_OK;
  if (probs || loss_rows) {
    bce_fwd_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, scores, label, gain, (float)negative_samples, probs, loss_rows);
    LSTUR_CHECK_LAUNCH("lstur_bce_loss(fwd)");
  }
  if (loss_mean) {
    mean_kernel<<<1, 256, 0, stream>>>((int)n, loss_rows, loss_mean);
    LSTUR_CHECK_LAUNCH("lstur_bce_loss(mean)");
  }
  if (dscores) {
    bce_bwd_kernel<<<cdiv(n, 256), 256, 0, stream>>>(n, scores, label, gain, (float)negative_samples, grad_scale, dscores);
    LSTUR_CHECK_LAUNCH("lstur_bce_loss(bwd)");
  }
  return LSTUR_OK;
}
extern "C" int lstur_dot_score_bwd(int B, int C, int D, const float* u, long long ldu, const float* d, long long ldd,
                                   const float* dscores, float* du, long long lddu, float* dd, long long lddd,
                                   cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && C >= 1 && D > 0 && u && d && dscores && du && dd, "lstur_dot_score_bwd");
  if (B == 0) return LSTUR_OK;
  dot_score_bwd_kernel<<<cdiv((long long)B * D, 256), 256, 0, stream>>>(B, C, D, u, ldu, d, ldd, dscores, du, lddu, dd, lddd);
  LSTUR_CHECK_LAUNCH("lstur_dot_score_bwd");
  return LSTUR_OK;
}
