// Row interning: n key rows (L tokens, vertical, subvertical) -> one id per row and a document table with one row per
// distinct key, so that the token rows of Cook's .npz files (task/cook.py:14-28: ch_title (N,W,L) / cd_title (N,5,L)
// with a vertical and a subvertical per slot) feed the doc-id protocol of lstur_forward and lstur_score_impressions.
//
// Exact by construction: the positions are sorted by the K = L + 2 columns with the stable LSD radix passes of the
// word-table gradient (last column first, as many 9-bit passes as the column's largest value needs), so rows with equal
// keys are adjacent and in position order; a run head is a row whose key differs from its sorted predecessor in some
// column.  Ids: 0 is the all-zero key (the pad document, present whether or not a row has it); the other keys are
// numbered 1, 2, ... in the order of their first row (an exclusive scan over the "first row of a non-zero key" flags in
// position order).  Nothing depends on a hash, on the launch configuration or on the order in which blocks run.
//
// lstur_group_rows (the user groups of Cook's device scoring) marks the rows whose (user, scale, history row) differs
// from the previous row's and compacts their positions with the same scan.
#include "radix.cuh"

namespace lstur {
namespace {

constexpr int SCAN_CH = wg::SORT_CH;          // items one block of the scan covers

// column k of row r: tokens[r, k] for k < L, then vert[r], subvert[r] (a NULL column reads 0)
__device__ __forceinline__ int key_col(int L, const int* __restrict__ tokens, const int* __restrict__ vert,
                                       const int* __restrict__ subvert, long long r, int k) {
  if (k < L) return tokens[r * L + k];
  const int* c = k == L ? vert : subvert;
  return c ? c[r] : 0;
}

// colbits[k] |= every value of column k (as unsigned bits): how many radix passes the column needs
__global__ void column_or_kernel(long long n, int L, const int* __restrict__ tokens, const int* __restrict__ vert,
                                 const int* __restrict__ subvert, unsigned* __restrict__ colbits) {
  const int K = L + 2;
  for (int k = blockIdx.y; k < K; k += gridDim.y) {
    unsigned v = 0u;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x)
      v |= (unsigned)key_col(L, tokens, vert, subvert, r, k);
    v = (unsigned)warp_or((int)v);
    if ((threadIdx.x & 31) == 0 && v) atomicOr(colbits + k, v);
  }
}

__global__ void iota_keys_kernel(long long n, int L, int k, const int* __restrict__ tokens, const int* __restrict__ vert,
                                 const int* __restrict__ subvert, const int* __restrict__ pos_in, int* __restrict__ keys,
                                 int* __restrict__ pos) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int p = pos_in ? pos_in[i] : (int)i;
  pos[i] = p;
  keys[i] = key_col(L, tokens, vert, subvert, p, k);
}

// sorted index i: head[i] = its key differs from row pos[i-1]'s; first[pos[i]] = head of a non-zero key
__global__ void heads_kernel(long long n, int L, const int* __restrict__ tokens, const int* __restrict__ vert,
                             const int* __restrict__ subvert, const int* __restrict__ pos, int* __restrict__ head,
                             int* __restrict__ first) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int p = pos[i];
  bool h = i == 0, nz = false;
  for (int k = 0; k < L + 2; ++k) {
    const int v = key_col(L, tokens, vert, subvert, p, k);
    nz |= v != 0;
    if (!h) h = v != key_col(L, tokens, vert, subvert, pos[i - 1], k);
  }
  head[i] = h;
  first[p] = h && nz;
}

// exclusive scan, phase 1: each block scans its SCAN_CH items and leaves their sum in bsum
__global__ void __launch_bounds__(wg::SORT_THREADS) scan_local_kernel(long long n, const int* __restrict__ in,
                                                                      int* __restrict__ out, int* __restrict__ bsum) {
  __shared__ int sm[8];
  const long long base = (long long)blockIdx.x * SCAN_CH + (long long)threadIdx.x * wg::SORT_ITEMS;
  int v[wg::SORT_ITEMS], s = 0;
#pragma unroll
  for (int j = 0; j < wg::SORT_ITEMS; ++j) {
    v[j] = base + j < n ? in[base + j] : 0;
    s += v[j];
  }
  const int inc = wg::block_inclusive_scan_256(s, sm);
  int run = inc - s;
#pragma unroll
  for (int j = 0; j < wg::SORT_ITEMS; ++j) {
    if (base + j < n) out[base + j] = run;
    run += v[j];
  }
  if (threadIdx.x == wg::SORT_THREADS - 1) bsum[blockIdx.x] = inc;
}

// phase 3: add each block's offset (phase 2 scanned bsum in place)
__global__ void scan_add_kernel(long long n, const int* __restrict__ bsum, int* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] += bsum[i / SCAN_CH];
}

// out = exclusive prefix sums of in (n items, in != out allowed to alias), *total (device) = their sum
int exclusive_scan(long long n, const int* in, int* out, int* bsum, int* total, cudaStream_t st, const char* name) {
  const int nblk = (int)wg::sort_blocks(n);
  scan_local_kernel<<<nblk, wg::SORT_THREADS, 0, st>>>(n, in, out, bsum);
  LSTUR_CHECK_LAUNCH(name);
  if (int rc = wg::exclusive_scan_rows(bsum, 1, nblk, total, st, name)) return rc;
  scan_add_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, bsum, out);
  LSTUR_CHECK_LAUNCH(name);
  return LSTUR_OK;
}

// run_of[i] = inclusive scan of head - 1 (computed as exclusive scan + head); a head writes its run's id and first row
__global__ void run_ids_kernel(long long n, const int* __restrict__ pos, const int* __restrict__ head,
                               const int* __restrict__ run_excl, const int* __restrict__ first,
                               const int* __restrict__ rank, int* __restrict__ run_id, int* __restrict__ first_row) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !head[i]) return;
  const int p = pos[i];
  const int id = first[p] ? rank[p] + 1 : 0;
  run_id[run_excl[i]] = id;
  if (id) first_row[id] = p;
}

__global__ void scatter_ids_kernel(long long n, const int* __restrict__ pos, const int* __restrict__ head,
                                   const int* __restrict__ run_excl, const int* __restrict__ run_id, int* __restrict__ ids) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ids[pos[i]] = run_id[run_excl[i] + head[i] - 1];
}

// table row u = row first_row[u] of the input (u = 0: zeros), one warp per row
__global__ void table_kernel(int n_unique, int L, const int* __restrict__ tokens, const int* __restrict__ vert,
                             const int* __restrict__ subvert, const int* __restrict__ first_row, int* __restrict__ doc_tokens,
                             int* __restrict__ doc_vert, int* __restrict__ doc_subvert) {
  const int u = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (u >= n_unique) return;
  const long long r = u ? first_row[u] : -1;
  for (int l = lane; l < L; l += 32) doc_tokens[(long long)u * L + l] = r >= 0 ? tokens[r * L + l] : 0;
  if (lane == 0) {
    if (doc_vert) doc_vert[u] = r >= 0 && vert ? vert[r] : 0;
    if (doc_subvert) doc_subvert[u] = r >= 0 && subvert ? subvert[r] : 0;
  }
}

// flag[i] = row i starts a group: i == 0, or its user, scale or history row differs from row i-1's
__global__ void group_flags_kernel(int n, int W, const int* __restrict__ user, const float* __restrict__ scale,
                                   const int* __restrict__ hist_doc, int* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool f = i == 0;
  if (!f) f = user[i] != user[i - 1] || (scale && __float_as_uint(scale[i]) != __float_as_uint(scale[i - 1]));
  for (int j = 0; j < W && !f; ++j) f = hist_doc[(long long)i * W + j] != hist_doc[(long long)(i - 1) * W + j];
  flag[i] = f;
}

__global__ void compact_kernel(int n, const int* __restrict__ flag, const int* __restrict__ excl, int* __restrict__ starts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && flag[i]) starts[excl[i]] = i;
}

struct InternWs {
  int *keys_a, *keys_b, *pos_a, *pos_b, *ghist, *bintot, *head, *first, *run_excl, *rank, *run_id, *bsum, *total;
  unsigned* colbits;
  size_t bytes;
};
InternWs carve(void* base, long long n, int L) {
  InternWs w;
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off = (off + b + 255) & ~(size_t)255; return (char*)base + o; };
  const long long m = n > 0 ? n : 1, nblk = wg::sort_blocks(m);
  w.keys_a = (int*)take(m * 4); w.keys_b = (int*)take(m * 4); w.pos_a = (int*)take(m * 4); w.pos_b = (int*)take(m * 4);
  w.ghist = (int*)take((size_t)wg::RADIX * nblk * 4); w.bintot = (int*)take(wg::RADIX * 4);
  w.head = (int*)take(m * 4); w.first = (int*)take(m * 4); w.run_excl = (int*)take(m * 4); w.rank = (int*)take(m * 4);
  w.run_id = (int*)take(m * 4); w.bsum = (int*)take(nblk * 4); w.total = (int*)take(2 * 4);
  w.colbits = (unsigned*)take((size_t)(L + 2) * 4);
  w.bytes = off;
  return w;
}

}  // namespace
}  // namespace lstur

using namespace lstur;

extern "C" size_t lstur_intern_workspace_bytes(long long n, int L) {
  if (n < 0 || L < 0) return 0;
  return carve(nullptr, n, L).bytes;
}

extern "C" int lstur_intern_rows(int n, int L, const int* tokens, const int* vert, const int* subvert, int* ids,
                                 int* first_row, int* n_unique, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const char* name = "lstur_intern_rows";
  LSTUR_REQUIRE(n >= 0 && L >= 1 && n_unique && (n == 0 || (tokens && ids && first_row)), name);
  InternWs w = carve(workspace, n, L);
  LSTUR_REQUIRE(workspace && workspace_bytes >= w.bytes, name);
  *n_unique = 1;                                   // the all-zero key always has id 0
  if (n == 0) return LSTUR_OK;
  const int K = L + 2;
  cudaMemsetAsync(w.colbits, 0, (size_t)K * 4, st);
  column_or_kernel<<<dim3(cdiv(n, 256) < 64 ? cdiv(n, 256) : 64, K < 32 ? K : 32), 256, 0, st>>>(n, L, tokens, vert,
                                                                                                 subvert, w.colbits);
  LSTUR_CHECK_LAUNCH(name);
  unsigned colbits[1024];
  LSTUR_REQUIRE(K <= 1024, name);
  cudaMemcpyAsync(colbits, w.colbits, (size_t)K * 4, cudaMemcpyDeviceToHost, st);
  if (cudaStreamSynchronize(st) != cudaSuccess) {
    set_error("%s: %s", name, cudaGetErrorString(cudaGetLastError()));
    return LSTUR_ERR_CUDA;
  }
  // LSD: the last column first; a column of zeros needs no pass
  int *pos = nullptr, *keys = w.keys_a, *keys_tmp = w.keys_b, *pos_tmp = w.pos_b;
  for (int k = K - 1; k >= 0; --k) {
    int bits = 0;
    while (bits < 32 && (colbits[k] >> bits) != 0u) ++bits;
    if (!bits) continue;
    int* dst = pos == w.pos_a ? w.pos_b : w.pos_a;
    iota_keys_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, L, k, tokens, vert, subvert, pos, keys, dst);
    LSTUR_CHECK_LAUNCH(name);
    pos = dst;
    pos_tmp = pos == w.pos_a ? w.pos_b : w.pos_a;
    keys_tmp = keys == w.keys_a ? w.keys_b : w.keys_a;
    if (int rc = wg::radix_sort_pairs(&keys, &pos, &keys_tmp, &pos_tmp, n, bits, w.ghist, w.bintot, st, name)) return rc;
  }
  if (!pos) {                                      // every key is zero: positions in order
    iota_keys_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, L, 0, tokens, vert, subvert, nullptr, keys, w.pos_a);
    LSTUR_CHECK_LAUNCH(name);
    pos = w.pos_a;
  }
  heads_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, L, tokens, vert, subvert, pos, w.head, w.first);
  LSTUR_CHECK_LAUNCH(name);
  if (int rc = exclusive_scan(n, w.head, w.run_excl, w.bsum, w.total, st, name)) return rc;
  if (int rc = exclusive_scan(n, w.first, w.rank, w.bsum, w.total + 1, st, name)) return rc;
  cudaMemsetAsync(first_row, 0xff, 4, st);         // id 0 has no source row unless a zero key occurs: the table zeroes it
  run_ids_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, pos, w.head, w.run_excl, w.first, w.rank, w.run_id, first_row);
  LSTUR_CHECK_LAUNCH(name);
  scatter_ids_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, pos, w.head, w.run_excl, w.run_id, ids);
  LSTUR_CHECK_LAUNCH(name);
  int nz = 0;
  cudaMemcpyAsync(&nz, w.total + 1, 4, cudaMemcpyDeviceToHost, st);
  if (cudaStreamSynchronize(st) != cudaSuccess) {
    set_error("%s: %s", name, cudaGetErrorString(cudaGetLastError()));
    return LSTUR_ERR_CUDA;
  }
  *n_unique = 1 + nz;
  return LSTUR_OK;
}

extern "C" int lstur_intern_table(int n_unique, int L, const int* tokens, const int* vert, const int* subvert,
                                  const int* first_row, int* doc_tokens, int* doc_vert, int* doc_subvert, cudaStream_t st) {
  LSTUR_REQUIRE(n_unique >= 1 && L >= 1 && doc_tokens && (n_unique == 1 || (tokens && first_row)), "lstur_intern_table");
  table_kernel<<<cdiv((long long)n_unique * 32, 256), 256, 0, st>>>(n_unique, L, tokens, vert, subvert, first_row, doc_tokens,
                                                                     doc_vert, doc_subvert);
  LSTUR_CHECK_LAUNCH("lstur_intern_table");
  return LSTUR_OK;
}

extern "C" int lstur_group_rows(int n, int W, const int* user, const float* scale, const int* hist_doc, int* starts,
                                int* n_groups, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const char* name = "lstur_group_rows";
  LSTUR_REQUIRE(n >= 0 && W >= 0 && n_groups && (n == 0 || (user && starts && (W == 0 || hist_doc))), name);
  InternWs w = carve(workspace, n, 0);
  LSTUR_REQUIRE(workspace && workspace_bytes >= w.bytes, name);
  *n_groups = 0;
  if (n == 0) return LSTUR_OK;
  group_flags_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, W, user, scale, hist_doc, w.head);
  LSTUR_CHECK_LAUNCH(name);
  if (int rc = exclusive_scan(n, w.head, w.run_excl, w.bsum, w.total, st, name)) return rc;
  compact_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, w.head, w.run_excl, starts);
  LSTUR_CHECK_LAUNCH(name);
  cudaMemcpyAsync(n_groups, w.total, 4, cudaMemcpyDeviceToHost, st);
  if (cudaStreamSynchronize(st) != cudaSuccess) {
    set_error("%s: %s", name, cudaGetErrorString(cudaGetLastError()));
    return LSTUR_ERR_CUDA;
  }
  return LSTUR_OK;
}
