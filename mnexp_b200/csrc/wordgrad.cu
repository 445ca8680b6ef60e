// Word-embedding gradient: deterministic segment-sorted scatter-add of the per-token input gradients of the title
// Conv1D into the rows of the word table.
//
// Reference: keras Embedding(..., trainable=config.textual_embedding_trainable) (task/paper.py:132-138, main.py:36); its
// backward is tf.IndexedSlices -> unsorted_segment_sum over the token ids (Keras / TF internal, SURVEY.md §9.7).
//
//   d word_emb[v, :] = sum over token positions p with tok[p] == v of  dX[p, :] * xdrop[p, :]
//
// No floating-point atomics: the positions are sorted by token with a stable LSD radix sort (so a token's positions stay
// in ascending order), and the sorted list is summed by a fixed tree of equal-sized chunks (see reduce_kernel): a chunk
// finishes every token whose positions it contains entirely and hands at most two partial rows to the next level.  A
// step is therefore bit-reproducible, and the heavy tokens of a Zipf vocabulary (one token can own > 10 % of all
// positions) are spread over many warps instead of serialising on one.
// Positions whose gradient is identically zero are dropped before the sort: a pad position that no conv output over a
// real token reads (dPre is exactly 0 under the pad mask, task/paper.py:150-155).  With the TF 'SAME' halo,
// pl = (KS-1)/2, output m reads positions m-pl .. m+KS-1-pl, so position t is live when a token in
// [t-(KS-1-pl), t+pl] of its title is non-zero: KS-1-pl positions back, pl forward (KS = 4: two back, one forward).
#include "radix.cuh"

namespace lstur {
namespace wg {

constexpr int R = 64;                              // rows (or piece slots) walked by one warp
constexpr int BATCH = 4;                           // rows whose loads a warp keeps in flight
constexpr int RED_THREADS = 256;                   // 8 warps = 8 work items per block

// ---- keys: token id of every live position, V for dead ones (sorted to the end and ignored) --------------------------
// back / fwd: reach of the conv window on each side (KS-1-pl and pl)
__global__ void keys_kernel(long long n_pos, int L, int V, int back, int fwd, const int* __restrict__ tok,
                            int* __restrict__ keys, int* __restrict__ pos, const int* __restrict__ n_titles_dev) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pos) return;
  const int t = (int)(p % L);
  const bool in_range = !n_titles_dev || p < (long long)__ldg(n_titles_dev) * L;   // compacted title list: rows beyond are unused
  int id = in_range ? tok[p] : 0;
  bool live = id != 0;
  if (in_range)
    for (int s = max(t - back, 0), e = min(t + fwd, L - 1); s <= e && !live; ++s) live = tok[p - t + s] != 0;
  id = (id < 0 || id >= V) ? 0 : id;          // out-of-range ids read row 0, like the forward gather
  keys[p] = live ? id : V;
  pos[p] = (int)p;
}

// ---- stable LSD radix sort, one 9-bit digit per pass --------------------------------------------------------------------
__global__ void __launch_bounds__(SORT_THREADS) radix_hist_kernel(const int* __restrict__ keys, long long n, int shift,
                                                                  int nblk, int* __restrict__ ghist) {
  __shared__ int h[RADIX];
  for (int i = threadIdx.x; i < RADIX; i += SORT_THREADS) h[i] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * SORT_CH;
#pragma unroll
  for (int k = 0; k < SORT_ITEMS; ++k) {
    const long long i = base + k * SORT_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & (RADIX - 1)], 1);     // integer counts: order-independent
  }
  __syncthreads();
  for (int b = threadIdx.x; b < RADIX; b += SORT_THREADS) ghist[(long long)b * nblk + blockIdx.x] = h[b];
}

// row b of ghist (the digit's counts per block) -> exclusive prefix over the blocks; bintot[b] = the digit's total
__global__ void __launch_bounds__(256) radix_rowscan_kernel(int* __restrict__ ghist, int nblk, int* __restrict__ bintot) {
  __shared__ int sm[8];
  int* row = ghist + (long long)blockIdx.x * nblk;
  int carry = 0;
  for (int i0 = 0; i0 < nblk; i0 += 256) {
    const int i = i0 + threadIdx.x;
    const int v = i < nblk ? row[i] : 0;
    const int inc = block_inclusive_scan_256(v, sm);
    if (i < nblk) row[i] = carry + inc - v;
    __shared__ int tot;
    if (threadIdx.x == 255) tot = inc;
    __syncthreads();
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) bintot[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(SORT_THREADS) radix_scatter_kernel(const int* __restrict__ keys_in, const int* __restrict__ pos_in,
                                                                     int* __restrict__ keys_out, int* __restrict__ pos_out,
                                                                     long long n, int shift, int nblk,
                                                                     const int* __restrict__ ghist, const int* __restrict__ bintot) {
  __shared__ int cnt[SORT_THREADS / 32][RADIX];
  __shared__ int binbase[RADIX];
  __shared__ int sm[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  {   // exclusive scan of the 512 digit totals: two per thread
    const int a = bintot[2 * tid], b = bintot[2 * tid + 1];
    const int inc = block_inclusive_scan_256(a + b, sm);
    binbase[2 * tid] = inc - a - b;
    binbase[2 * tid + 1] = inc - b;
  }
  for (int i = tid; i < (SORT_THREADS / 32) * RADIX; i += SORT_THREADS) (&cnt[0][0])[i] = 0;
  __syncthreads();
  // A warp owns 256 consecutive items, 32 per round: the rank of an item inside its (warp, digit) group is the number
  // of earlier items of the group — earlier rounds (cnt) plus lower lanes of this round (match_any) — so equal digits
  // keep their input order (stable).
  const long long base = (long long)blockIdx.x * SORT_CH + warp * (SORT_ITEMS * 32);
  int key[SORT_ITEMS], ps[SORT_ITEMS], rank[SORT_ITEMS];
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; ++r) {
    const long long i = base + r * 32 + lane;
    const bool valid = i < n;
    key[r] = valid ? keys_in[i] : 0;
    ps[r] = valid ? pos_in[i] : 0;
    const int d = (key[r] >> shift) & (RADIX - 1);
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? d : -1 - lane);
    const int lrank = __popc(peers & ((1u << lane) - 1u));
    const int old = valid ? cnt[warp][d] : 0;
    __syncwarp();
    if (valid && lrank == 0) cnt[warp][d] = old + __popc(peers);
    __syncwarp();
    rank[r] = old + lrank;
  }
  __syncthreads();
  for (int b = tid; b < RADIX; b += SORT_THREADS) {     // exclusive prefix of the digit's counts over the warps
    int run = 0;
#pragma unroll
    for (int w = 0; w < SORT_THREADS / 32; ++w) {
      const int t = cnt[w][b];
      cnt[w][b] = run;
      run += t;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; ++r) {
    const long long i = base + r * 32 + lane;
    if (i < n) {
      const int d = (key[r] >> shift) & (RADIX - 1);
      const long long dst = (long long)binbase[d] + ghist[(long long)d * nblk + blockIdx.x] + cnt[warp][d] + rank[r];
      keys_out[dst] = key[r];
      pos_out[dst] = ps[r];
    }
  }
}

int radix_sort_pairs(int** keys, int** pos, int** keys_tmp, int** pos_tmp, long long n, int bits, int* ghist, int* bintot,
                     cudaStream_t st, const char* name) {
  if (n <= 0) return LSTUR_OK;
  const int nblk = (int)sort_blocks(n);
  for (int shift = 0; shift < bits; shift += RB) {
    radix_hist_kernel<<<nblk, SORT_THREADS, 0, st>>>(*keys, n, shift, nblk, ghist);
    LSTUR_CHECK_LAUNCH(name);
    radix_rowscan_kernel<<<RADIX, 256, 0, st>>>(ghist, nblk, bintot);
    LSTUR_CHECK_LAUNCH(name);
    radix_scatter_kernel<<<nblk, SORT_THREADS, 0, st>>>(*keys, *pos, *keys_tmp, *pos_tmp, n, shift, nblk, ghist, bintot);
    LSTUR_CHECK_LAUNCH(name);
    int* t = *keys; *keys = *keys_tmp; *keys_tmp = t;
    t = *pos; *pos = *pos_tmp; *pos_tmp = t;
  }
  return LSTUR_OK;
}

int exclusive_scan_rows(int* rows, int n_rows, int len, int* totals, cudaStream_t st, const char* name) {
  if (n_rows <= 0) return LSTUR_OK;
  radix_rowscan_kernel<<<n_rows, 256, 0, st>>>(rows, len, totals);
  LSTUR_CHECK_LAUNCH(name);
  return LSTUR_OK;
}

// ---- segments of the sorted keys: seg_beg[v] / seg_end[v] (both zero-initialised; absent tokens keep 0, 0) ------------
__global__ void bounds_kernel(long long n, int V, const int* __restrict__ keys, int* __restrict__ seg_beg,
                              int* __restrict__ seg_end) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int k = keys[i];
  if (k >= V) return;
  if (i == 0 || keys[i - 1] != k) seg_beg[k] = (int)i;
  if (i + 1 == n || keys[i + 1] != k) seg_end[k] = (int)(i + 1);
}

// Row sources.  A lane owns the 4-column pieces lane, lane+32, ... (NP of them) of a row.
struct Src16 {          // level 1, tensor-core modes: 16-bit dX rows (n_pos, Ep) + keep bytes of the X-dropout
  const uint16_t* dx;
  const uint8_t* xmask;   // or null
  int Ep, fp16;
};
struct Src32 {          // level 1, fp32 mode: fp32 rows of the padded title buffer dXp (n_titles, Lp, E) + hash replay
  const float* dx;
  int L, Lp, pl, E;
  uint32_t drop_thr, seed;
};
struct SrcPart {        // levels 2 and 3: fp32 partial rows (rows, E)
  const float* rows;
  int E;
};

// A row is fetched (load_row: the loads of several rows are issued back to back, so a warp keeps up to BATCH rows in
// flight) and then accumulated (add_raw) in position order.
template <int NP> struct Raw16 { uint2 v[NP]; unsigned m[NP]; };
template <int NP> struct Raw32 { float4 v[NP]; unsigned m[NP]; };
template <int NP> struct RawPart { float4 v[NP]; };
template <typename SRC, int NP> struct RawOf;
template <int NP> struct RawOf<Src16, NP> { typedef Raw16<NP> type; };
template <int NP> struct RawOf<Src32, NP> { typedef Raw32<NP> type; };
template <int NP> struct RawOf<SrcPart, NP> { typedef RawPart<NP> type; };

template <int NP>
__device__ __forceinline__ void load_row(const Src16& s, long long pos, int lane, Raw16<NP>& r) {
  const uint16_t* row = s.dx + pos * s.Ep;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int piece = lane + 32 * j;
    r.v[j] = make_uint2(0u, 0u);
    r.m[j] = 0xffu;
    if (piece * 4 < s.Ep) {
      r.v[j] = __ldg(reinterpret_cast<const uint2*>(row + piece * 4));
      if (s.xmask) r.m[j] = __ldg(s.xmask + pos * (s.Ep >> 3) + (piece >> 1));
    }
  }
}
template <int NP>
__device__ __forceinline__ void add_raw(const Src16& s, const Raw16<NP>& r, int lane, float (&acc)[NP][4]) {
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int piece = lane + 32 * j;
    const uint2 u = r.v[j];
    const unsigned m = r.m[j];
    const int wj = (piece & 1) * 2;      // 32-bit word of the 16-byte piece; bit wj+h / 4+wj+h = low / high half of word wj+h
    float v[4];
    if (s.fp16) {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    } else {
      v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
      v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
    }
    acc[j][0] += ((m >> wj) & 1u) ? v[0] : 0.f;
    acc[j][1] += ((m >> (4 + wj)) & 1u) ? v[1] : 0.f;
    acc[j][2] += ((m >> (wj + 1)) & 1u) ? v[2] : 0.f;
    acc[j][3] += ((m >> (5 + wj)) & 1u) ? v[3] : 0.f;
  }
}
template <int NP>
__device__ __forceinline__ void load_row(const Src32& s, long long pos, int lane, Raw32<NP>& r) {
  const long long n = pos / s.L;
  const int t = (int)(pos % s.L);
  const float* row = s.dx + (n * s.Lp + t + s.pl) * s.E;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int e = (lane + 32 * j) * 4;
    r.v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    r.m[j] = 15u;
    if (e < s.E) {
      r.v[j] = __ldg(reinterpret_cast<const float4*>(row + e));
      if (s.drop_thr) {
        const uint64_t base = (uint64_t)pos * (uint64_t)s.E + e;
        r.m[j] = ((rng_u32(s.seed, base + 0) >> 8) >= s.drop_thr ? 1u : 0u) | ((rng_u32(s.seed, base + 1) >> 8) >= s.drop_thr ? 2u : 0u) |
                 ((rng_u32(s.seed, base + 2) >> 8) >= s.drop_thr ? 4u : 0u) | ((rng_u32(s.seed, base + 3) >> 8) >= s.drop_thr ? 8u : 0u);
      }
    }
  }
}
template <int NP>
__device__ __forceinline__ void add_raw(const Src32&, const Raw32<NP>& r, int, float (&acc)[NP][4]) {
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const float4 v = r.v[j];
    const unsigned m = r.m[j];
    acc[j][0] += (m & 1u) ? v.x : 0.f; acc[j][1] += (m & 2u) ? v.y : 0.f; acc[j][2] += (m & 4u) ? v.z : 0.f; acc[j][3] += (m & 8u) ? v.w : 0.f;
  }
}
template <int NP>
__device__ __forceinline__ void load_row(const SrcPart& s, long long rr, int lane, RawPart<NP>& r) {
  const float* row = s.rows + rr * s.E;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int e = (lane + 32 * j) * 4;
    r.v[j] = e < s.E ? __ldg(reinterpret_cast<const float4*>(row + e)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
template <int NP>
__device__ __forceinline__ void add_raw(const SrcPart&, const RawPart<NP>& r, int, float (&acc)[NP][4]) {
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    acc[j][0] += r.v[j].x; acc[j][1] += r.v[j].y; acc[j][2] += r.v[j].z; acc[j][3] += r.v[j].w;
  }
}

// ---- chunk tree.  Level 1: chunk c = the R consecutive sorted positions [c*R, (c+1)*R); level l > 1: chunk c = the
// pieces left by the FAN = R/2 level-(l-1) chunks [c*FAN, (c+1)*FAN) (two slots each), i.e. it spans S_l = R * FAN^(l-1)
// sorted positions.  One warp walks its chunk's rows in order and sums the runs of equal token id.  A run that covers the
// token's whole segment [seg_beg, seg_end) of the sorted list is final: it is scaled and written to the token's row of
// d_word_emb.  Otherwise the segment crosses the chunk's boundary (at most one run per side can): the partial sum goes to
// one of the chunk's two piece slots (token id + fp32 row; unused slots are tagged -1) and the next level continues.
// The top level has one chunk, which covers everything.  Summation order = position order at every level: no atomics,
// bit-reproducible, and every warp has the same amount of work however skewed the token frequencies are.
constexpr int FAN = R / 2;

template <typename SRC, int NP, bool LEVEL1>
__global__ void __launch_bounds__(RED_THREADS) reduce_kernel(SRC src, long long n_items, long long span, int V, int E,
                                                             const int* __restrict__ keys_in, const int* __restrict__ pos_sorted,
                                                             const int* __restrict__ seg_beg, const int* __restrict__ seg_end,
                                                             int* __restrict__ piece_keys, float* __restrict__ piece_rows,
                                                             float* __restrict__ d_word_emb, float scale) {
  const int lane = threadIdx.x & 31;
  const long long c = ((long long)blockIdx.x * RED_THREADS + threadIdx.x) >> 5;     // chunk
  const long long i0 = c * R, i1 = min(n_items, i0 + R);
  if (i0 >= n_items) return;
  const long long lo = c * span, hi = lo + span;       // sorted positions covered by this chunk
  float acc[NP][4];
  int cur = -1, n_out = 0;
  auto flush = [&]() {
    if (cur < 0) return;
    const bool whole = __ldg(seg_beg + cur) >= lo && __ldg(seg_end + cur) <= hi;
    float* dst;
    float sc = 1.f;
    if (whole) { dst = d_word_emb + (long long)cur * E; sc = scale; }
    else {
      dst = piece_rows + (2 * c + n_out) * E;
      if (lane == 0) piece_keys[2 * c + n_out] = cur;
      ++n_out;
    }
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const int e = (lane + 32 * j) * 4;
      if (e < E) *reinterpret_cast<float4*>(dst + e) = make_float4(acc[j][0] * sc, acc[j][1] * sc, acc[j][2] * sc, acc[j][3] * sc);
    }
  };
  for (long long b = i0; b < i1; b += 32) {
    const int cntb = (int)min((long long)32, i1 - b);
    int my_key = -1;
    long long my_row = b + lane;
    if (lane < cntb) {
      my_key = keys_in[b + lane];
      if (LEVEL1) { my_row = pos_sorted[b + lane]; if (my_key >= V) my_key = -1; }     // dead positions sort last
    }
    for (int j0 = 0; j0 < cntb; j0 += BATCH) {
      int ks[BATCH];
      typename RawOf<SRC, NP>::type raw[BATCH];
#pragma unroll
      for (int u = 0; u < BATCH; ++u) {         // issue the loads of BATCH rows
        ks[u] = __shfl_sync(0xffffffffu, my_key, (j0 + u) & 31);
        const long long r = __shfl_sync(0xffffffffu, my_row, (j0 + u) & 31);
        if (j0 + u >= cntb) ks[u] = -1;
        if (ks[u] >= 0) load_row<NP>(src, r, lane, raw[u]);
      }
#pragma unroll
      for (int u = 0; u < BATCH; ++u) {         // accumulate them in order
        if (ks[u] < 0) continue;                // empty slot / dead position
        if (ks[u] != cur) {
          flush();
          cur = ks[u];
#pragma unroll
          for (int q = 0; q < NP; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
        }
        add_raw<NP>(src, raw[u], lane, acc);
      }
    }
  }
  flush();
  if (piece_keys && lane == 0)
    for (int j = n_out; j < 2; ++j) piece_keys[2 * c + j] = -1;
}

struct Ws {          // carve-up of the caller's workspace
  int *keys_a, *keys_b, *pos_a, *pos_b, *ghist, *bintot, *seg_beg, *seg_end, *pk1, *pk2;
  float *pr1, *pr2;
  size_t bytes;
};
static long long n_chunks(long long items) { return (items + R - 1) / R; }
static Ws carve(void* base, long long n, int V, int E) {
  Ws w;
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off = (off + b + 255) & ~(size_t)255; return (char*)base + o; };
  const long long nblk = sort_blocks(n);
  const long long c1 = n_chunks(n > 0 ? n : 1), c2 = n_chunks(2 * c1);     // chunks of level 1 / level 2 (ping-pong buffers)
  w.keys_a = (int*)take(n * 4); w.keys_b = (int*)take(n * 4); w.pos_a = (int*)take(n * 4); w.pos_b = (int*)take(n * 4);
  w.ghist = (int*)take((size_t)RADIX * nblk * 4); w.bintot = (int*)take(RADIX * 4);
  w.seg_beg = (int*)take((size_t)V * 4 * 2); w.seg_end = w.seg_beg + V;       // contiguous: one memset
  w.pk1 = (int*)take((size_t)2 * c1 * 4); w.pk2 = (int*)take((size_t)2 * c2 * 4);
  w.pr1 = (float*)take((size_t)2 * c1 * E * 4); w.pr2 = (float*)take((size_t)2 * c2 * E * 4);
  w.bytes = off;
  return w;
}

template <typename SRC>
static int run(SRC src, long long n, int L, int KS, int V, int E, const int* tokens, const int* n_titles_dev, float scale,
               float* d_word_emb, void* workspace, size_t workspace_bytes, cudaStream_t st, const char* name) {
  LSTUR_REQUIRE(n >= 0 && n < (1LL << 31) && L >= 1 && V >= 1 && E >= 4 && E % 4 == 0 && E <= 512 && tokens && d_word_emb, name);
  Ws w = carve(workspace, n, V, E);
  LSTUR_REQUIRE(workspace != nullptr && workspace_bytes >= w.bytes, name);
  cudaMemsetAsync(d_word_emb, 0, (size_t)V * E * sizeof(float), st);
  if (n == 0) return LSTUR_OK;
  const int pl = (KS - 1) / 2;
  keys_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, L, V, KS - 1 - pl, pl, tokens, w.keys_a, w.pos_a, n_titles_dev);
  LSTUR_CHECK_LAUNCH(name);
  int bits = 1;
  while ((1LL << bits) <= V) ++bits;              // keys are 0 .. V inclusive
  int *ka = w.keys_a, *kb = w.keys_b, *pa = w.pos_a, *pb = w.pos_b;
  if (int rc = radix_sort_pairs(&ka, &pa, &kb, &pb, n, bits, w.ghist, w.bintot, st, name)) return rc;
  cudaMemsetAsync(w.seg_beg, 0, (size_t)V * 4 * 2, st);
  bounds_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, V, ka, w.seg_beg, w.seg_end);
  LSTUR_CHECK_LAUNCH(name);
  const int wpb = RED_THREADS / 32;
  const int np = (E / 4 + 31) / 32;               // 4-column pieces per lane
#define WG_LAUNCH(NP_)                                                                                                    \
  do {                                                                                                                    \
    long long items = n, span = R;                                                                                        \
    long long nc = n_chunks(items);                                                                                       \
    reduce_kernel<SRC, NP_, true><<<cdiv(nc, wpb), RED_THREADS, 0, st>>>(src, items, span, V, E, ka, pa, w.seg_beg, w.seg_end, \
                                                                         nc > 1 ? w.pk1 : nullptr, w.pr1, d_word_emb, scale); \
    LSTUR_CHECK_LAUNCH(name);                                                                                             \
    int* pk_in = w.pk1; float* pr_in = w.pr1; int* pk_out = w.pk2; float* pr_out = w.pr2;                                 \
    while (nc > 1) {                                                                                                      \
      items = 2 * nc; span *= FAN; nc = n_chunks(items);                                                                  \
      const SrcPart sp{pr_in, E};                                                                                         \
      reduce_kernel<SrcPart, NP_, false><<<cdiv(nc, wpb), RED_THREADS, 0, st>>>(sp, items, span, V, E, pk_in, nullptr, w.seg_beg, \
                                                                                w.seg_end, nc > 1 ? pk_out : nullptr, pr_out, \
                                                                                d_word_emb, scale);                       \
      LSTUR_CHECK_LAUNCH(name);                                                                                           \
      int* ti = pk_in; pk_in = pk_out; pk_out = ti;                                                                       \
      float* tf = pr_in; pr_in = pr_out; pr_out = tf;                                                                     \
    }                                                                                                                     \
  } while (0)
  if (np <= 1) WG_LAUNCH(1);
  else if (np == 2) WG_LAUNCH(2);
  else if (np == 3) WG_LAUNCH(3);
  else WG_LAUNCH(4);
#undef WG_LAUNCH
  return LSTUR_OK;
}

}  // namespace wg
}  // namespace lstur

using namespace lstur;

extern "C" int lstur_tc_padded_e(int E);

extern "C" size_t lstur_word_grad_workspace_bytes(long long n_pos, int V, int E) {
  if (n_pos < 0 || V < 1 || E < 1) return 0;
  return wg::carve(nullptr, n_pos, V, E).bytes;
}

// tensor-core modes: dx16 (n_titles, L, lstur_tc_padded_e(E)) from lstur_conv_dgrad_tc, keep bytes from the forward
extern "C" int lstur_word_grad_scatter_16(int n_titles, int L, int E, int V, const int* tokens, const void* dx16, int fp16,
                                          float scale, const void* xmask, float* d_word_emb, void* workspace,
                                          size_t workspace_bytes, const int* n_titles_dev, cudaStream_t stream) {
  LSTUR_REQUIRE(n_titles >= 0 && dx16 != nullptr, "lstur_word_grad_scatter_16");
  wg::Src16 s{(const uint16_t*)dx16, (const uint8_t*)xmask, lstur_tc_padded_e(E), fp16};
  return wg::run(s, (long long)n_titles * L, L, 3, V, E, tokens, n_titles_dev, scale, d_word_emb, workspace, workspace_bytes,
                 stream, "lstur_word_grad_scatter_16");     // the tensor-core conv has KS = 3
}

// fp32 mode: dXp (n_titles, L+KS-1, E) = gradient of the zero-haloed title buffer of lstur_embed_gather_pad; the X-dropout
// of that kernel (seed, dropout) is replayed
extern "C" int lstur_word_grad_scatter_f32(int n_titles, int L, int KS, int E, int V, const int* tokens, const float* dXp,
                                           float dropout, unsigned seed, float scale, float* d_word_emb, void* workspace,
                                           size_t workspace_bytes, cudaStream_t stream) {
  LSTUR_REQUIRE(n_titles >= 0 && dXp != nullptr && KS >= 1 && dropout >= 0.f && dropout < 1.f, "lstur_word_grad_scatter_f32");
  wg::Src32 s{dXp, L, L + KS - 1, (KS - 1) / 2, E, dropout > 0.f ? dropout_threshold(dropout) : 0u, seed};
  return wg::run(s, (long long)n_titles * L, L, KS, V, E, tokens, nullptr, scale / (1.f - dropout), d_word_emb, workspace,
                 workspace_bytes, stream, "lstur_word_grad_scatter_f32");
}
