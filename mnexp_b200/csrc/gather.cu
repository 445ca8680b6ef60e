// Integer / gather kernels of the LSTUR path (HBM-bound byte movers).
//
//  token_gather      Window.get_title / np.stack([docs[i].title …])       task/seq2vec.py:25-30, task/paper.py:538-541
//  embed_gather      keras Embedding(mask_zero=False) + Dropout            task/paper.py:132-138,142,147
//  hist_mask_apply   models.ComputeMasking(0) + multiply + Masking()       models.py:25-27, task/paper.py:644-645,592
//  row_gather        user-ID Embedding lookup                              task/paper.py:589-591
//  vert_concat       [title ‖ Vemb[vert] ‖ Semb[subvert]]                  task/cook.py:99-113
#include "common.cuh"

namespace lstur {

// tokens[n, :] = doc_tokens[doc_ids[n], :]   — int32, bit-exact. One warp per title row.
__global__ void token_gather_kernel(int N, int L, int n_docs, const int* __restrict__ doc_tokens,
                                    const int* __restrict__ doc_ids, int* __restrict__ tokens) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  int d = doc_ids[warp];
  d = (d < 0 || d >= n_docs) ? 0 : d;  // out-of-range ids read the pad doc
  const int* src = doc_tokens + (long long)d * L;
  int* dst = tokens + (long long)warp * L;
  for (int l = lane; l < L; l += 32) dst[l] = __ldg(src + l);
}

// Xp[n, pl+t, :] = word_emb[tok[n,t], :] * dropout with pl=(KS-1)/2 zero rows before and KS-1-pl after
// (TF 'SAME' padding); title stride Lp = L+KS-1 rows.
// One warp per padded row; float4 vectorised when E % 4 == 0.
__global__ void embed_gather_pad_kernel(int N, int L, int E, int V, int KS, const float* __restrict__ word_emb,
                                        const int* __restrict__ tok, float* __restrict__ Xp, uint32_t drop_thr,
                                        float inv_keep, uint32_t seed) {
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  const int Lp = L + KS - 1;
  if (row >= (long long)N * Lp) return;
  int n = (int)(row / Lp), t = (int)(row % Lp) - (KS - 1) / 2;
  float* dst = Xp + row * E;
  if (t < 0 || t >= L) {
    for (int e = lane; e < E; e += 32) dst[e] = 0.f;
    return;
  }
  int id = tok[(long long)n * L + t];
  id = (id < 0 || id >= V) ? 0 : id;
  const float* src = word_emb + (long long)id * E;
  const uint64_t base = ((uint64_t)n * L + t) * (uint64_t)E;
  if ((E & 3) == 0) {
    for (int e = lane * 4; e < E; e += 128) {
      float4 v = __ldg((const float4*)(src + e));
      if (drop_thr) {
        v.x = (rng_u32(seed, base + e + 0) >> 8) >= drop_thr ? v.x * inv_keep : 0.f;
        v.y = (rng_u32(seed, base + e + 1) >> 8) >= drop_thr ? v.y * inv_keep : 0.f;
        v.z = (rng_u32(seed, base + e + 2) >> 8) >= drop_thr ? v.z * inv_keep : 0.f;
        v.w = (rng_u32(seed, base + e + 3) >> 8) >= drop_thr ? v.w * inv_keep : 0.f;
      }
      *(float4*)(dst + e) = v;
    }
  } else {
    for (int e = lane; e < E; e += 32) {
      float v = __ldg(src + e);
      if (drop_thr) v = (rng_u32(seed, base + e) >> 8) >= drop_thr ? v * inv_keep : 0.f;
      dst[e] = v;
    }
  }
}

// For the B*W history titles: hm = any(tok != 0); H[row,:] *= hm; gm = any(H != 0).
__global__ void hist_mask_apply_kernel(int rows, int L, int D, const int* __restrict__ tok, float* __restrict__ H,
                                       long long ldh, float* __restrict__ hm_out, float* __restrict__ gm_out) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  int nz = 1;       // tok == null (cached document vectors): only the Masking() part, gm = any(H != 0)
  if (tok) {
    nz = 0;
    for (int l = lane; l < L; l += 32) nz |= (tok[(long long)warp * L + l] != 0);
    nz = warp_or(nz);
  }
  float* h = H + (long long)warp * ldh;
  int any = 0;
  for (int d = lane; d < D; d += 32) {
    float v = nz ? h[d] : 0.f;
    h[d] = v;
    any |= (v != 0.f);
  }
  any = warp_or(any);
  if (lane == 0) {
    if (hm_out) hm_out[warp] = (tok ? nz : any) ? 1.f : 0.f;
    gm_out[warp] = any ? 1.f : 0.f;
  }
}

// out[b, :] = table[ids[b], :] * (scale ? scale[b] : 1)
__global__ void row_gather_kernel(int B, int D, int n_rows, const float* __restrict__ table,
                                  const int* __restrict__ ids, const float* __restrict__ scale,
                                  float* __restrict__ out, long long ldo) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  int id = ids[warp];
  id = (id < 0 || id >= n_rows) ? 0 : id;
  float s = scale ? scale[warp] : 1.f;
  for (int d = lane; d < D; d += 32) out[(long long)warp * ldo + d] = __ldg(table + (long long)id * D + d) * s;
}


// One warp per title: ids -> vertical / subvertical rows -> the extra columns of the document vector.
__global__ void vert_concat_kernel(int n, int D, int col0, int dv, int ds, int n_docs, int n_vert, int n_sub,
                                   const int* __restrict__ doc_ids, const int* __restrict__ doc_vert,
                                   const int* __restrict__ doc_subvert, const float* __restrict__ vert_emb,
                                   const float* __restrict__ subvert_emb, float* __restrict__ docv,
                                   int* __restrict__ tv, int* __restrict__ ts) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  int d = warp;                       // doc_ids == NULL: doc_vert / doc_subvert are indexed by the title slot itself
  if (doc_ids) {
    d = doc_ids[warp];
    d = (d < 0 || d >= n_docs) ? 0 : d;
  }
  int v = dv ? doc_vert[d] : 0, sv = ds ? doc_subvert[d] : 0;
  v = (v < 0 || v >= n_vert) ? 0 : v;
  sv = (sv < 0 || sv >= n_sub) ? 0 : sv;
  float* row = docv + (long long)warp * D + col0;
  for (int j = lane; j < dv; j += 32) row[j] = vert_emb[(long long)v * dv + j];
  for (int j = lane; j < ds; j += 32) row[dv + j] = subvert_emb[(long long)sv * ds + j];
  if (lane == 0) {
    if (tv) tv[warp] = v;
    if (ts) ts[warp] = sv;
  }
}

// Stage 1 of the small-table Embedding backward: CTA (r, k) adds, in ascending title order, the gradient columns of
// the titles of chunk k whose id is r.  Stage 2 adds the chunk partials in ascending chunk order.
constexpr int STG_CHUNKS = 64;
__global__ void small_table_grad1_kernel(int n, int D, int col0, int dim, const int* __restrict__ ids,
                                         const float* __restrict__ dd, float* __restrict__ partial) {
  const int r = blockIdx.x, k = blockIdx.y, n_rows = gridDim.x;
  const int per = (n + STG_CHUNKS - 1) / STG_CHUNKS;
  const int beg = k * per, end = min(n, beg + per);
  float acc = 0.f;
  const int j = threadIdx.x;
  for (int i = beg; i < end; ++i)
    if (ids[i] == r && j < dim) acc += dd[(long long)i * D + col0 + j];
  if (j < dim) partial[((long long)k * n_rows + r) * dim + j] = acc;
}
__global__ void small_table_grad2_kernel(int n_rows, int dim, const float* __restrict__ partial, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * dim) return;
  float acc = 0.f;
  for (int k = 0; k < STG_CHUNKS; ++k) acc += partial[(long long)k * n_rows * dim + i];
  out[i] = acc;
}
__global__ void scale_rows_kernel(int B, int D, const float* __restrict__ scale, float* __restrict__ x, long long ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * D) return;
  const int b = (int)(i / D), d = (int)(i % D);
  x[(long long)b * ld + d] *= scale[b];
}


// Device-side sample assembly (train_gen / valid_gen + Window + Impression.negative_samples, task/paper.py:7-18,
// 387-441, 669-694; task/seq2vec.py:17-53).  Sample s = idx[b] is the click c = sample_click[s] of user u; its history is
// the W stream entries before hist_end (hist_end = sample_hist_end[s], or c when that table is NULL), left-padded with
// doc 0.  With click_time, a history slot j keeps its doc only while click_time[j] + expire >= click_time[c] (the Days
// Window's expiry, summed in 64 bits; times need not be monotonic along the stream).  The positive is the click itself,
// the negatives K draws WITH replacement from the negatives shown in the click's impression, counter-based on the global
// row row0 + b.  One thread per output element.
__global__ void assemble_samples_kernel(int B, int W, int K, const int* __restrict__ sample_click,
                                        const int* __restrict__ sample_hist_end, const int* __restrict__ idx,
                                        const int* __restrict__ click_user, const int* __restrict__ click_time,
                                        long long expire, const int* __restrict__ stream_off,
                                        const int* __restrict__ stream_docs, const int* __restrict__ neg_off,
                                        const int* __restrict__ neg_docs, uint32_t seed, long long row0,
                                        int* __restrict__ user_out, int* __restrict__ hist_out, int* __restrict__ cand_out) {
  const int T = W + 1 + K;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * T) return;
  const int b = (int)(i / T), e = (int)(i % T);
  const int s = idx[b];
  const int c = sample_click[s];
  const int u = click_user[c];
  const int off = stream_off[u];
  if (e < W) {
    const int j = (sample_hist_end ? sample_hist_end[s] : c) - W + e;
    int d = j >= off ? stream_docs[j] : 0;
    if (click_time && j >= off && (long long)click_time[j] + expire < (long long)click_time[c]) d = 0;
    hist_out[(long long)b * W + e] = d;
    if (e == 0) user_out[b] = u;
  } else if (e == W) {
    cand_out[(long long)b * (1 + K)] = stream_docs[c];
  } else {
    const int k = e - W - 1;
    const int n0 = neg_off[c], n = neg_off[c + 1] - n0;
    const uint32_t r = rng_u32(seed, (uint64_t)(row0 + b) * K + k);
    cand_out[(long long)b * (1 + K) + 1 + k] = n > 0 ? neg_docs[n0 + (int)(r % (uint32_t)n)] : 0;
  }
}

// ---- title compaction: the news encoder of an all-pad title (every token 0: the left padding of a short click history,
// task/seq2vec.py:23,46-49) is identically zero in value and gradient (pad mask, task/paper.py:150-155), so the
// tensor-core kernels run over the compacted list of live titles only.
__global__ void title_live_kernel(int N, int L, const int* __restrict__ tok, int* __restrict__ flags) {
  int warp = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (warp >= N) return;
  int nz = 0;
  for (int l = lane; l < L; l += 32) nz |= (tok[(long long)warp * L + l] != 0);
  nz = warp_or(nz);
  if (lane == 0) flags[warp] = nz ? 1 : 0;
}
// blocks of 1024 titles: rank of every live title inside its block + the block's live count
__global__ void __launch_bounds__(1024) title_rank_kernel(int N, const int* __restrict__ flags, int* __restrict__ local_rank,
                                                          int* __restrict__ block_tot) {
  __shared__ int wsum[32];
  const int n = blockIdx.x * 1024 + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int f = (n < N && flags[n]) ? 1 : 0;
  const unsigned bal = __ballot_sync(0xffffffffu, f);
  if (lane == 0) wsum[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {
    int v = wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    wsum[lane] = v;            // inclusive
  }
  __syncthreads();
  if (n < N) local_rank[n] = (warp ? wsum[warp - 1] : 0) + __popc(bal & ((1u << lane) - 1u));
  if (threadIdx.x == 0) block_tot[blockIdx.x] = wsum[31];
}
// one warp per title: global rank = live titles of the earlier blocks + rank inside the block; live titles are appended to
// live_idx (ascending) and their tokens copied
__global__ void title_compact_kernel(int N, int L, const int* __restrict__ tok, const int* __restrict__ flags,
                                     const int* __restrict__ local_rank, const int* __restrict__ block_tot, int n_blocks,
                                     int* __restrict__ live_idx, int* __restrict__ n_live, int* __restrict__ tok_c) {
  int warp = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (warp >= N) return;
  const int blk = warp >> 10;
  int before = 0;
  for (int b = lane; b < n_blocks; b += 32) before += (b < blk || warp == N - 1) ? block_tot[b] : 0;
  before = __reduce_add_sync(0xffffffffu, before);
  if (warp == N - 1) {         // the last title's warp summed every block: the live count
    if (lane == 0) *n_live = before;
    before = 0;
    for (int b = lane; b < blk; b += 32) before += block_tot[b];
    before = __reduce_add_sync(0xffffffffu, before);
  }
  if (!flags[warp]) return;
  const int ci = before + local_rank[warp];
  if (lane == 0) live_idx[ci] = warp;
  for (int l = lane; l < L; l += 32) tok_c[(long long)ci * L + l] = tok[(long long)warp * L + l];
}

// L == 1 (a list of non-zero entries of a mask, e.g. the unmasked (user, step) rows): one THREAD per entry
__global__ void mask_live_kernel(int N, const int* __restrict__ v, int* __restrict__ flags) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) flags[n] = v[n] != 0 ? 1 : 0;
}
__global__ void __launch_bounds__(1024) mask_compact_kernel(int N, const int* __restrict__ v, const int* __restrict__ flags,
                                                            const int* __restrict__ local_rank,
                                                            const int* __restrict__ block_tot, int n_blocks,
                                                            int* __restrict__ live_idx, int* __restrict__ n_live,
                                                            int* __restrict__ v_c) {
  __shared__ int s_before;
  const int blk = blockIdx.x, n = blk * 1024 + threadIdx.x;
  if (threadIdx.x < 32) {          // live entries of the earlier blocks (fixed order); the last block also publishes the total
    int before = 0, total = 0;
    for (int b = threadIdx.x; b < n_blocks; b += 32) {
      const int t = block_tot[b];
      total += t;
      if (b < blk) before += t;
    }
    before = __reduce_add_sync(0xffffffffu, before);
    total = __reduce_add_sync(0xffffffffu, total);
    if (threadIdx.x == 0) {
      s_before = before;
      if (blk == n_blocks - 1) *n_live = total;
    }
  }
  __syncthreads();
  if (n < N && flags[n]) {
    const int ci = s_before + local_rank[n];
    live_idx[ci] = n;
    v_c[ci] = v[n];
  }
}

// Rows of a sample table by position (Cook's interned .npz, task/cook.py:60-90): row b of the batch is sample
// s = pos[b] for b < m and pos[0] for the padding rows b >= m of a ragged last batch, whose label row is zero.  One thread
// per output element; a NULL table leaves its output alone.
__global__ void gather_samples_kernel(int B, int m, int W, int C, const int* __restrict__ pos, const int* __restrict__ user,
                                      const float* __restrict__ scale, const int* __restrict__ hist_doc,
                                      const int* __restrict__ cand_doc, const float* __restrict__ label,
                                      int* __restrict__ user_out, float* __restrict__ scale_out, int* __restrict__ hist_out,
                                      int* __restrict__ cand_out, float* __restrict__ label_out) {
  const int per = 2 + W + 2 * C;               // user, scale, W history slots, C candidates, C labels
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)B * per) return;
  const int b = (int)(e / per), j = (int)(e % per);
  const long long s = pos[b < m ? b : 0];
  if (j == 0) {
    if (user) user_out[b] = user[s];
  } else if (j == 1) {
    if (scale) scale_out[b] = scale[s];
  } else if (j < 2 + W) {
    if (hist_doc) hist_out[(long long)b * W + j - 2] = hist_doc[s * W + j - 2];
  } else if (j < 2 + W + C) {
    if (cand_doc) cand_out[(long long)b * C + j - 2 - W] = cand_doc[s * C + j - 2 - W];
  } else if (label) {
    const int c = j - 2 - W - C;
    label_out[(long long)b * C + c] = b < m ? label[s * C + c] : 0.f;
  }
}

}  // namespace lstur

using namespace lstur;

// tokens (N,L) -> n_live (1), live_idx (N; first n_live entries = ascending indices of the titles that have a non-zero
// token), tokens_c (N,L; first n_live rows = those titles' tokens); scratch = lstur_compact_titles_scratch_ints(N) ints.
extern "C" long long lstur_compact_titles_scratch_ints(int N) { return 2LL * N + (N + 1023) / 1024 + 8; }
extern "C" int lstur_compact_titles(int N, int L, const int* tokens, int* scratch, int* live_idx, int* n_live, int* tokens_c,
                                    cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L > 0 && n_live != nullptr, "lstur_compact_titles");
  if (N == 0) { cudaMemsetAsync(n_live, 0, sizeof(int), stream); return LSTUR_OK; }
  LSTUR_REQUIRE(tokens && scratch && live_idx && tokens_c, "lstur_compact_titles");
  const int nb = (N + 1023) / 1024;
  int *flags = scratch, *local_rank = scratch + N, *block_tot = scratch + 2 * (long long)N;
  if (L == 1) {      // list of the non-zero entries of a vector: thread-per-entry kernels
    mask_live_kernel<<<cdiv(N, 256), 256, 0, stream>>>(N, tokens, flags);
    LSTUR_CHECK_LAUNCH("lstur_compact_titles(flags)");
    title_rank_kernel<<<nb, 1024, 0, stream>>>(N, flags, local_rank, block_tot);
    LSTUR_CHECK_LAUNCH("lstur_compact_titles(rank)");
    mask_compact_kernel<<<nb, 1024, 0, stream>>>(N, tokens, flags, local_rank, block_tot, nb, live_idx, n_live, tokens_c);
    LSTUR_CHECK_LAUNCH("lstur_compact_titles(gather)");
    return LSTUR_OK;
  }
  title_live_kernel<<<cdiv((long long)N * 32, 256), 256, 0, stream>>>(N, L, tokens, flags);
  LSTUR_CHECK_LAUNCH("lstur_compact_titles(flags)");
  title_rank_kernel<<<nb, 1024, 0, stream>>>(N, flags, local_rank, block_tot);
  LSTUR_CHECK_LAUNCH("lstur_compact_titles(rank)");
  title_compact_kernel<<<cdiv((long long)N * 32, 256), 256, 0, stream>>>(N, L, tokens, flags, local_rank, block_tot, nb, live_idx,
                                                                        n_live, tokens_c);
  LSTUR_CHECK_LAUNCH("lstur_compact_titles(gather)");
  return LSTUR_OK;
}

extern "C" int lstur_token_gather(int N, int L, int n_docs, const int* doc_tokens, const int* doc_ids, int* tokens,
                                  cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L > 0 && n_docs > 0, "lstur_token_gather");
  if (N == 0) return LSTUR_OK;
  token_gather_kernel<<<cdiv((long long)N * 32, 256), 256, 0, stream>>>(N, L, n_docs, doc_tokens, doc_ids, tokens);
  LSTUR_CHECK_LAUNCH("lstur_token_gather");
  return LSTUR_OK;
}

extern "C" int lstur_embed_gather_pad(int N, int L, int E, int V, int KS, const float* word_emb, const int* tokens,
                                      float* Xp, float dropout, unsigned seed, cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L > 0 && E > 0 && KS >= 1 && dropout >= 0.f && dropout < 1.f, "lstur_embed_gather_pad");
  if (N == 0) return LSTUR_OK;
  long long rows = (long long)N * (L + KS - 1);
  embed_gather_pad_kernel<<<cdiv(rows * 32, 256), 256, 0, stream>>>(
      N, L, E, V, KS, word_emb, tokens, Xp, dropout > 0.f ? dropout_threshold(dropout) : 0u, 1.f / (1.f - dropout), seed);
  LSTUR_CHECK_LAUNCH("lstur_embed_gather_pad");
  return LSTUR_OK;
}

extern "C" int lstur_hist_mask_apply(int rows, int L, int D, const int* tokens, float* H, long long ldh, float* hm,
                                     float* gm, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && L > 0 && D > 0 && gm != nullptr, "lstur_hist_mask_apply");
  if (rows == 0) return LSTUR_OK;
  hist_mask_apply_kernel<<<cdiv((long long)rows * 32, 256), 256, 0, stream>>>(rows, L, D, tokens, H, ldh, hm, gm);
  LSTUR_CHECK_LAUNCH("lstur_hist_mask_apply");
  return LSTUR_OK;
}

extern "C" int lstur_row_gather(int B, int D, int n_rows, const float* table, const int* ids, const float* scale,
                                float* out, long long ldo, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && D > 0 && n_rows > 0, "lstur_row_gather");
  if (B == 0) return LSTUR_OK;
  row_gather_kernel<<<cdiv((long long)B * 32, 256), 256, 0, stream>>>(B, D, n_rows, table, ids, scale, out, ldo);
  LSTUR_CHECK_LAUNCH("lstur_row_gather");
  return LSTUR_OK;
}

extern "C" int lstur_vert_concat(int n, int D, int col0, int dv, int ds, int n_docs, int n_vert, int n_subvert, const int* doc_ids,
                                 const int* doc_vert, const int* doc_subvert, const float* vert_emb, const float* subvert_emb,
                                 float* doc_vec, int* title_vert, int* title_subvert, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && dv >= 0 && ds >= 0 && col0 >= 0 && col0 + dv + ds <= D && doc_vec, "lstur_vert_concat");
  LSTUR_REQUIRE((dv == 0 || (doc_vert && vert_emb && n_vert > 0)) && (ds == 0 || (doc_subvert && subvert_emb && n_subvert > 0)),
                "lstur_vert_concat");
  if (n == 0 || dv + ds == 0) return LSTUR_OK;
  vert_concat_kernel<<<cdiv((long long)n * 32, 256), 256, 0, stream>>>(n, D, col0, dv, ds, n_docs, n_vert, n_subvert, doc_ids,
                                                                       doc_vert, doc_subvert, vert_emb, subvert_emb, doc_vec,
                                                                       title_vert, title_subvert);
  LSTUR_CHECK_LAUNCH("lstur_vert_concat");
  return LSTUR_OK;
}

extern "C" size_t lstur_small_table_grad_workspace_bytes(int n_rows, int dim) {
  return (size_t)STG_CHUNKS * n_rows * dim * sizeof(float);
}

extern "C" int lstur_small_table_grad(int n, int D, int col0, int dim, int n_rows, const int* ids, const float* d_doc_vec,
                                      float* d_table, float* workspace, size_t workspace_bytes, cudaStream_t stream) {
  LSTUR_REQUIRE(n >= 0 && dim > 0 && dim <= 1024 && n_rows > 0 && col0 >= 0 && col0 + dim <= D && d_table, "lstur_small_table_grad");
  LSTUR_REQUIRE(workspace && workspace_bytes >= lstur_small_table_grad_workspace_bytes(n_rows, dim), "lstur_small_table_grad");
  LSTUR_REQUIRE(n == 0 || (ids && d_doc_vec), "lstur_small_table_grad");
  const int threads = (dim + 31) / 32 * 32;
  small_table_grad1_kernel<<<dim3(n_rows, STG_CHUNKS), threads, 0, stream>>>(n, D, col0, dim, ids, d_doc_vec, workspace);
  LSTUR_CHECK_LAUNCH("lstur_small_table_grad(stage 1)");
  small_table_grad2_kernel<<<cdiv((long long)n_rows * dim, 256), 256, 0, stream>>>(n_rows, dim, workspace, d_table);
  LSTUR_CHECK_LAUNCH("lstur_small_table_grad(stage 2)");
  return LSTUR_OK;
}

extern "C" int lstur_scale_rows(int B, int D, const float* scale, float* x, long long ld, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && D > 0 && scale && x && ld >= D, "lstur_scale_rows");
  if (B == 0) return LSTUR_OK;
  scale_rows_kernel<<<cdiv((long long)B * D, 256), 256, 0, stream>>>(B, D, scale, x, ld);
  LSTUR_CHECK_LAUNCH("lstur_scale_rows");
  return LSTUR_OK;
}

extern "C" int lstur_assemble_samples(int B, int W, int K, const int* sample_click, const int* sample_hist_end,
                                      const int* idx, const int* click_user, const int* click_time, long long expire_seconds,
                                      const int* stream_off, const int* stream_docs, const int* neg_off, const int* neg_docs,
                                      unsigned seed, long long row0, int* user_out, int* hist_doc_out, int* cand_doc_out,
                                      cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && K >= 0 && row0 >= 0, "lstur_assemble_samples");
  LSTUR_REQUIRE(B == 0 || (sample_click && idx && click_user && stream_off && stream_docs && neg_off && neg_docs && user_out &&
                           hist_doc_out && cand_doc_out), "lstur_assemble_samples");
  if (B == 0) return LSTUR_OK;
  const long long n = (long long)B * (W + 1 + K);
  assemble_samples_kernel<<<cdiv(n, 256), 256, 0, stream>>>(B, W, K, sample_click, sample_hist_end, idx, click_user,
                                                            click_time, expire_seconds, stream_off, stream_docs, neg_off,
                                                            neg_docs, seed, row0, user_out, hist_doc_out, cand_doc_out);
  LSTUR_CHECK_LAUNCH("lstur_assemble_samples");
  return LSTUR_OK;
}

extern "C" int lstur_assemble_batch(int B, int W, int K, const int* sample_click, const int* idx, const int* click_user,
                                    const int* stream_off, const int* stream_docs, const int* neg_off, const int* neg_docs,
                                    unsigned seed, int* user_out, int* hist_doc_out, int* cand_doc_out, cudaStream_t stream) {
  return lstur_assemble_samples(B, W, K, sample_click, nullptr, idx, click_user, nullptr, 0, stream_off, stream_docs, neg_off,
                                neg_docs, seed, 0, user_out, hist_doc_out, cand_doc_out, stream);
}

extern "C" int lstur_gather_samples(int B, int m, int W, int C, const int* pos, const int* user, const float* scale,
                                    const int* hist_doc, const int* cand_doc, const float* label, int* user_out,
                                    float* scale_out, int* hist_doc_out, int* cand_doc_out, float* label_out,
                                    cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W >= 0 && C >= 0 && (B == 0 || (m >= 1 && m <= B && pos)), "lstur_gather_samples");
  LSTUR_REQUIRE((!user || user_out) && (!scale || scale_out) && (!hist_doc || hist_doc_out) && (!cand_doc || cand_doc_out) &&
                (!label || label_out), "lstur_gather_samples");
  if (B == 0) return LSTUR_OK;
  gather_samples_kernel<<<cdiv((long long)B * (2 + W + 2 * C), 256), 256, 0, stream>>>(
      B, m, W, C, pos, user, scale, hist_doc, cand_doc, label, user_out, scale_out, hist_doc_out, cand_doc_out, label_out);
  LSTUR_CHECK_LAUNCH("lstur_gather_samples");
  return LSTUR_OK;
}
