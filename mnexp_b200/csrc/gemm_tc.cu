// Generic tensor-core GEMM (tcgen05.mma, fp16 operands, fp32 accumulate in TMEM) on fp32 global operands.
//
//   C[M,N] (+)= op(A)[M,K] . op(B)[K,N] (+ bias[N]) (relu)
//
// Replaces gemm_f32 in tensor-core precision for the plain dense contractions of the LSTUR path:
// Dense(F->U) (task/paper.py:159), the GRU input projection (keras GRU, task/paper.py:612) and all of their
// input / weight gradients.  Operands stay fp32 in HBM; producer warps convert to fp16 while staging 16-byte
// pieces into 128B-swizzled shared-memory tiles.  An operand whose K index is contiguous in memory (A
// non-transposed, B transposed) is staged K-major; one whose M/N index is contiguous (A transposed — the
// weight-gradient case — or B non-transposed) is staged MN-major, so no transposition ever happens in memory:
// only the UMMA descriptor's major-ness bits differ.  Split-K over CTA.z with a fixed-order reduction.
// Warp roles (416 threads): w0 MMA issuer + TMEM alloc, w1-8 producers, w9-12 epilogue.
#include <stdlib.h>

#include "tc_common.cuh"

namespace lstur {
namespace tc {

constexpr int G_KBLK = 64;
constexpr int G_STAGES = 4;
constexpr int G_A_BYTES = TILE_M * 128;    // 16 KB (either major-ness)
constexpr int G_B_BYTES = 256 * 128;       // up to N tile 256
constexpr int G_STAGE_BYTES = G_A_BYTES + G_B_BYTES;          // single-term fp16
constexpr int G_STAGE_BYTES_S3 = 2 * (G_A_BYTES + G_B_BYTES);  // hi + lo tiles for the 3-term split
constexpr int G_THREADS = 416;   // w0 MMA issuer + TMEM alloc, w1-8 producers, w9-12 epilogue (152 registers per thread)
constexpr int G_PRODUCERS = 256;

struct GemmParams {
  int M, N, K;
  const float* A; long long lda;
  const float* B; long long ldb;
  float* C; long long ldc;
  const float* bias;
  int flags, ntile, k_per_split, vec_ok;
  int tiles_m, tiles_n, splits;
  float* partial;
  // optional pre-packed B operand (gemm_pack_b_kernel): per (n tile, K block) one hi [+ one lo] 32 KB tile in the exact
  // shared-memory layout of a stage, fetched with bulk copies instead of being re-converted by every CTA for every tile
  const uint8_t* bimg;
  int nkb_total;
  // optional row list for the reduction index of a TN product (gemm_tc_async_kernel, A and B both stored [K, .]): only
  // the rows kidx[0 .. *kcount) of A and B are summed (ascending list of the rows that are not identically zero, e.g. the
  // unmasked (user, step) rows of the GRU tensors); the split-K ranges are cut from *kcount on the device
  const int* kidx;
  const int* kcount;
  // optional row list for the M index of an NN / NT product (gemm_tc_kernel, A stored [M, K]): only the rows
  // midx[0 .. *mcount) of A are multiplied and only those rows of C are written (ascending list, device count)
  const int* midx;
  const int* mcount;
};
constexpr int G_BIMG_TILE = 256 * 128;    // bytes reserved per image tile (= G_B_BYTES)

// 8 consecutive floats of row s_idx starting at column c0, zero-filled outside [0, s_lim) x [0, c_lim)
__device__ __forceinline__ void load_raw(const float* __restrict__ base, long long ld, int s_idx, int s_lim, int c0, int c_lim,
                                         bool vec_ok, float* v) {
  if (s_idx < s_lim && c0 + 8 <= c_lim && vec_ok) {
    const float4* p = reinterpret_cast<const float4*>(base + (long long)s_idx * ld + c0);
    float4 a = __ldg(p), b = __ldg(p + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      v[i] = (s_idx < s_lim && c0 + i < c_lim) ? __ldg(base + (long long)s_idx * ld + c0 + i) : 0.f;
  }
}
// 8 floats -> 8 fp16 (16 bytes) [+ the 8 fp16 residuals]
template <bool SPLIT>
__device__ __forceinline__ uint4 cvt_piece(const float* v, uint4& lo) {
  uint32_t o[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    o[i] = *reinterpret_cast<uint32_t*>(&h);
    if (SPLIT) {   // x = hi + lo with hi = fp16(x), lo = fp16(x - hi): ~22 mantissa bits across the pair
      float2 hf = __half22float2(h);
      __half2 r = __floats2half2_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
      l[i] = *reinterpret_cast<uint32_t*>(&r);
    }
  }
  if (SPLIT) lo = make_uint4(l[0], l[1], l[2], l[3]);
  return make_uint4(o[0], o[1], o[2], o[3]);
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Epilogue store of one 32-column accumulator chunk: lane = tile row holds r[0..31] (columns c0.. of the tile).  A
// row-per-lane float4 store touches 32 different lines per instruction (32 L1 wavefronts, half-filled sectors) — the
// epilogue, not the tensor core or the staging, bounded the large-M GEMMs.  Through a per-warp staging buffer (rows of
// 36 floats: conflict-free 16-byte accesses both ways) 8 lanes cover the 128 contiguous bytes of one row, so an
// instruction writes 4 full lines; bias / accumulate / relu are applied on the way out (one bias load per lane and
// chunk instead of one dependent scalar load per element, which had halved the speed of the GRU input projection).
constexpr int G_EPI_ROW = 36;                              // floats per staged row
constexpr int G_EPI_WARP_BYTES = 32 * G_EPI_ROW * 4;       // 4608
__device__ __forceinline__ void gemm_epi_store(float* stg, int lane, const uint32_t* r, bool have_acc, float* cbase,
                                               long long ldc, int row0, int M, int col0, int ncols, const float* bias,
                                               int flags, bool apply, bool vec_ok, const int* orow = nullptr) {
#pragma unroll
  for (int g = 0; g < 8; ++g)
    *reinterpret_cast<float4*>(stg + lane * G_EPI_ROW + 4 * g) =
        have_acc ? make_float4(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1]), __uint_as_float(r[4 * g + 2]),
                               __uint_as_float(r[4 * g + 3]))
                 : make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  const int piece = lane & 7, cc = 4 * piece;              // this lane's 4 columns of the chunk
  if (cc < ncols) {
    float b4[4] = {0.f, 0.f, 0.f, 0.f};
    if (apply && bias) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (cc + u < ncols) b4[u] = __ldg(bias + col0 + cc + u);
    }
    const bool full = cc + 4 <= ncols && vec_ok;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = (lane >> 3) + 4 * i;
      const int grow = orow ? orow[i] : (row0 + row < M ? row0 + row : -1);      // output row (listed rows: C row of list entry)
      if (grow < 0) continue;
      float4 v = *reinterpret_cast<const float4*>(stg + row * G_EPI_ROW + cc);
      float* dst = cbase + (long long)grow * ldc + col0 + cc;
      float x[4] = {v.x, v.y, v.z, v.w};
      if (apply) {
        if (flags & LSTUR_GEMM_ACCUM) {
          if (full) { const float4 o = *reinterpret_cast<const float4*>(dst); x[0] += o.x; x[1] += o.y; x[2] += o.z; x[3] += o.w; }
          else {
#pragma unroll
            for (int u = 0; u < 4; ++u) if (cc + u < ncols) x[u] += dst[u];
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          x[u] += b4[u];
          if (flags & LSTUR_GEMM_RELU) x[u] = fmaxf(x[u], 0.f);
        }
      }
      if (full) *reinterpret_cast<float4*>(dst) = make_float4(x[0], x[1], x[2], x[3]);
      else {
#pragma unroll
        for (int u = 0; u < 4; ++u) if (cc + u < ncols) dst[u] = x[u];
      }
    }
  }
  __syncwarp();
}

// TA: A is stored [K,M] (M contiguous) -> MN-major.  TB: B is stored [N,K] (K contiguous) -> K-major.
// SPLIT: 3-term fp16 split (Ahi.Bhi + Alo.Bhi + Ahi.Blo) for ~fp32 accuracy on the forward-path GEMMs.
// Persistent: a CTA walks the (m, n, k-split) tiles t = blockIdx.x, +gridDim.x, ... (n fastest, so CTAs that run
// together share an A tile in L2); the shared-memory stage ring runs across tile boundaries and two 256-column
// accumulators in tensor memory let the epilogue of one tile overlap the loads and MMAs of the next.
template <bool TA, bool TB, bool SPLIT>
__global__ void __launch_bounds__(G_THREADS, 1) gemm_tc_kernel(const GemmParams p) {
  constexpr int STAGES = SPLIT ? 2 : G_STAGES;
  constexpr int STAGE_BYTES = SPLIT ? G_STAGE_BYTES_S3 : G_STAGE_BYTES;
  constexpr int LO_OFF = G_A_BYTES + G_B_BYTES;     // lo tiles follow the hi tiles inside a stage
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t misc_base = smem_base + STAGES * STAGE_BYTES;
  uint8_t* misc_gen = smem_gen + (misc_base - smem_base);
  const uint32_t bar_full = misc_base, bar_empty = misc_base + 64, bar_t_full = misc_base + 128, bar_t_empty = misc_base + 144;
  uint32_t* tmem_ptr_smem = (uint32_t*)(misc_gen + 160);
  float* s_epi = (float*)(misc_gen + 256);      // [4 epilogue warps] staging rows (G_EPI_WARP_BYTES each)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // listed rows: the M extent is the device-side count of the list
  const int Meff = p.mcount ? min(__ldg(p.mcount), p.M) : p.M;
  const int tiles_m = p.mcount ? (Meff + TILE_M - 1) / TILE_M : p.tiles_m;
  const int n_tiles = tiles_m * p.tiles_n * p.splits;

  // tile index -> (m0, n0, split) and derived extents
  struct Tile { int m0, n0, nt, nmma, z, kbeg, kend, nkb; };
  auto tile_of = [&](int t) {
    Tile x;
    const int tn = t % p.tiles_n, tm = (t / p.tiles_n) % tiles_m;
    x.z = t / (p.tiles_n * tiles_m);
    x.m0 = tm * TILE_M;
    x.n0 = tn * p.ntile;
    x.nt = min(p.ntile, p.N - x.n0);                       // valid columns of this tile
    x.nmma = (x.nt + 15) & ~15;                            // UMMA N (multiple of 16)
    x.kbeg = x.z * p.k_per_split;
    x.kend = min(p.K, x.kbeg + p.k_per_split);
    x.nkb = x.kend > x.kbeg ? (x.kend - x.kbeg + G_KBLK - 1) / G_KBLK : 0;
    return x;
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, G_PRODUCERS / 32 + (p.bimg ? 1 : 0));   // + the bulk-copy issuer's arrive.expect_tx
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_t_full + 8 * a, 1);
      mbar_init(bar_t_empty + 8 * a, 4);     // the four epilogue warps
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    {   // the whole warp runs the loop, one elected lane issues (see elect_one)
      const bool leader = elect_one();
      int s = 0, acc = 0;
      uint32_t ph = 0, pht[2] = {0, 0};
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const Tile x = tile_of(t);
        const uint32_t idesc = make_idesc(TILE_M, x.nmma, true) | (TA ? (1u << 15) : 0u) | (!TB ? (1u << 16) : 0u);
        mbar_wait(bar_t_empty + 8 * acc, pht[acc] ^ 1, 24);      // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * 256;
        uint32_t accum = 0;
        for (int kb = 0; kb < x.nkb; ++kb) {
          mbar_wait(bar_full + 8 * s, ph, 21);
          tc_fence_after();
          const uint32_t a_addr = smem_base + s * STAGE_BYTES, b_addr = a_addr + G_A_BYTES;
          if (leader) {
#pragma unroll
            for (int kk = 0; kk < G_KBLK / 16; ++kk) {
              const uint64_t ad = TA ? make_desc_mn128(a_addr + kk * 2048, 8192) : make_desc_k128(a_addr + kk * 32);
              const uint64_t bd = TB ? make_desc_k128(b_addr + kk * 32) : make_desc_mn128(b_addr + kk * 2048, 8192);
              umma_bf16(tacc, ad, bd, idesc, accum);
              accum = 1;
              if (SPLIT) {
                const uint64_t al = TA ? make_desc_mn128(a_addr + LO_OFF + kk * 2048, 8192) : make_desc_k128(a_addr + LO_OFF + kk * 32);
                const uint64_t bl = TB ? make_desc_k128(b_addr + LO_OFF + kk * 32) : make_desc_mn128(b_addr + LO_OFF + kk * 2048, 8192);
                umma_bf16(tacc, al, bd, idesc, 1);
                umma_bf16(tacc, ad, bl, idesc, 1);
              }
            }
            umma_commit(bar_empty + 8 * s);
          }
          accum = 1;
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        if (leader) umma_commit(bar_t_full + 8 * acc);
        __syncwarp();
        pht[acc] ^= 1;
        acc ^= 1;
      }
    }
  } else if (warp >= 1 && warp < 9) {
    // ---- producers: fp32 global -> fp16 swizzled tiles
    const int pt = threadIdx.x - 32;         // 0..255
    int s = 0;
    uint32_t ph = 0;
    // A thread stages pieces i = pt + it*256: 4 of A (it < 4) and up to 8 of B.  The global loads of a whole batch of
    // pieces are issued before any of them is converted and stored (one memory round trip per batch instead of one per
    // piece), and the first batch of a K block is requested before waiting for its stage to drain.
    constexpr int BATCH = 6;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const Tile x = tile_of(t);
      const int m0 = x.m0, n0 = x.n0, nt = x.nt, kend = x.kend;
      const int bgroups = (x.nmma + 63) >> 6;
      const bool img = p.bimg != nullptr;
      const int nb_pieces = img ? 0 : (TB ? x.nmma * 8 : bgroups * 512);      // B pieces of this tile per K block
      const uint32_t b_tile_bytes = (uint32_t)(TB ? x.nmma * 128 : bgroups * 8192);
      // rows of A behind this thread's four pieces (the same for every K block of the tile); p.M = "no row"
      int arow[4];
#pragma unroll
      for (int idx = 0; idx < 4; ++idx) {
        const int r = m0 + ((pt + idx * G_PRODUCERS) >> 3);
        arow[idx] = r < Meff ? (p.midx ? __ldg(p.midx + r) : r) : p.M;
      }
      for (int kb = 0; kb < x.nkb; ++kb) {
        const int k0 = x.kbeg + kb * G_KBLK;
        const uint32_t a_addr = smem_base + s * STAGE_BYTES, b_addr = a_addr + G_A_BYTES;
        auto piece_load = [&](int idx, float* v) {
          if (idx < 4) {
            const int i = pt + idx * G_PRODUCERS, c = i & 7, r = i >> 3;
            if (!TA) load_raw(p.A, p.lda, arow[idx], p.M, k0 + 8 * c, kend, p.vec_ok, v);
            else load_raw(p.A, p.lda, k0 + (r & 63), kend, m0 + (r >> 6) * 64 + 8 * c, p.M, p.vec_ok, v);
          } else {
            const int i = pt + (idx - 4) * G_PRODUCERS, c = i & 7, r = i >> 3;
            if (i < nb_pieces) {
              if (TB) load_raw(p.B, p.ldb, n0 + r, n0 + nt, k0 + 8 * c, kend, p.vec_ok, v);
              else load_raw(p.B, p.ldb, k0 + (r & 63), kend, n0 + (r >> 6) * 64 + 8 * c, n0 + nt, p.vec_ok, v);
            }
          }
        };
        auto piece_store = [&](int idx, const float* v) {
          uint4 lo;
          if (idx < 4) {
            const int i = pt + idx * G_PRODUCERS, c = i & 7, r = i >> 3;
            const uint4 hi = cvt_piece<SPLIT>(v, lo);
            const uint32_t off = !TA ? (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4))
                                     : (uint32_t)((r >> 6) * 8192 + (r & 63) * 128 + ((c ^ (r & 7)) << 4));
            sts128(a_addr + off, hi);
            if (SPLIT) sts128(a_addr + LO_OFF + off, lo);
          } else {
            const int i = pt + (idx - 4) * G_PRODUCERS, c = i & 7, r = i >> 3;
            if (i < nb_pieces) {
              const uint4 hi = cvt_piece<SPLIT>(v, lo);
              const uint32_t off = TB ? (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4))
                                      : (uint32_t)((r >> 6) * 8192 + (r & 63) * 128 + ((c ^ (r & 7)) << 4));
              sts128(b_addr + off, hi);
              if (SPLIT) sts128(b_addr + LO_OFF + off, lo);
            }
          }
        };
        float v[BATCH][8];
#pragma unroll
        for (int j = 0; j < BATCH; ++j) piece_load(j, v[j]);
        if (lane == 0) mbar_wait(bar_empty + 8 * s, ph ^ 1, 22);
        __syncwarp();
        if (img && pt == 0) {     // this stage's B tile(s): bulk copies of the pre-packed image
          const uint8_t* src = p.bimg + ((size_t)(n0 / p.ntile) * p.nkb_total + (size_t)(k0 / G_KBLK)) * (SPLIT ? 2 : 1) * G_BIMG_TILE;
          mbar_expect_tx(bar_full + 8 * s, b_tile_bytes * (SPLIT ? 2u : 1u));
          bulk_g2s(b_addr, src, b_tile_bytes, bar_full + 8 * s);
          if (SPLIT) bulk_g2s(b_addr + LO_OFF, src + G_BIMG_TILE, b_tile_bytes, bar_full + 8 * s);
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) piece_store(j, v[j]);
        if (nb_pieces > (BATCH - 4) * G_PRODUCERS) {
#pragma unroll
          for (int j = 0; j < BATCH; ++j) piece_load(BATCH + j, v[j]);
#pragma unroll
          for (int j = 0; j < BATCH; ++j) piece_store(BATCH + j, v[j]);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * s);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 9) {
    // ---- epilogue (TMEM lane quarter = warp % 4)
    const int q = warp & 3;
    int acc = 0;
    uint32_t pht[2] = {0, 0};
    const bool split = p.splits > 1;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const Tile x = tile_of(t);
      mbar_wait(bar_t_full + 8 * acc, pht[acc], 23);
      pht[acc] ^= 1;
      tc_fence_after();
      float* cbase = split ? p.partial + (long long)x.z * p.M * p.N : p.C;
      const long long ldo = split ? (long long)p.N : p.ldc;
      const bool vec_st = (ldo % 4 == 0) && ((((uintptr_t)cbase) & 15) == 0) && ((x.n0 & 3) == 0);
      int orow[8];      // listed rows: the C rows of this lane's eight staged rows
      if (p.midx) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = x.m0 + q * 32 + (lane >> 3) + 4 * i;
          orow[i] = rr < Meff ? __ldg(p.midx + rr) : -1;
        }
      }
      for (int c0 = 0; c0 < x.nmma; c0 += 32) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
        if (x.nmma - c0 >= 32) { TMEM_LD_32(taddr, r); } else { TMEM_LD_16(taddr, r); }
        tmem_ld_wait();
        const int ncols = min(32, x.nt - c0);
        if (ncols > 0)
          gemm_epi_store(s_epi + (warp - 9) * (G_EPI_WARP_BYTES / 4), lane, r, x.nkb > 0, cbase, ldo, x.m0 + q * 32, Meff,
                         x.n0 + c0, ncols, p.bias, p.flags, !split, vec_st, p.midx ? orow : nullptr);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_t_empty + 8 * acc);     // accumulator free for the tile after next
      acc ^= 1;
    }
  }
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// B operand -> per (n tile, K block) fp16 tiles [hi][lo?] in the shared-memory layout of a stage (zero-filled outside
// the matrix).  grid = (K blocks, n tiles).
template <bool TB, bool SPLIT>
__global__ void gemm_pack_b_kernel(int N, int K, const float* __restrict__ B, long long ldb, int ntile, int vec_ok,
                                   uint8_t* __restrict__ img) {
  const int kb = blockIdx.x, tn = blockIdx.y, nkb_total = gridDim.x;
  const int n0 = tn * ntile, nt = min(ntile, N - n0), nmma = (nt + 15) & ~15, bgroups = (nmma + 63) >> 6;
  const int k0 = kb * G_KBLK;
  const int pieces = TB ? nmma * 8 : bgroups * 512;
  uint8_t* dst = img + ((size_t)tn * nkb_total + kb) * (SPLIT ? 2 : 1) * G_BIMG_TILE;
  for (int i = threadIdx.x; i < pieces; i += blockDim.x) {
    const int c = i & 7, r = i >> 3;
    float v[8];
    if (TB) load_raw(B, ldb, n0 + r, n0 + nt, k0 + 8 * c, K, vec_ok != 0, v);
    else load_raw(B, ldb, k0 + (r & 63), K, n0 + (r >> 6) * 64 + 8 * c, n0 + nt, vec_ok != 0, v);
    uint4 lo;
    const uint4 hi = cvt_piece<SPLIT>(v, lo);
    const uint32_t off = TB ? (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4))
                            : (uint32_t)((r >> 6) * 8192 + (r & 63) * 128 + ((c ^ (r & 7)) << 4));
    *reinterpret_cast<uint4*>(dst + off) = hi;
    if (SPLIT) *reinterpret_cast<uint4*>(dst + G_BIMG_TILE + off) = lo;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Asynchronously staged variant (used when every operand row is 16-byte addressable): the fp32 operand tiles of the
// next TWO K blocks are always in flight as cp.async copies into a raw shared-memory ring (2 x 64 KB), so the memory
// system sees a deep request queue instead of one register round trip per batch of pieces; the producer warps only
// convert raw fp32 -> swizzled fp16 tiles (shared to shared).  N tile <= 128, two 128-column accumulators.
constexpr int GA_NT = 128;                       // max N tile
constexpr int GA_RAW_A = TILE_M * G_KBLK * 4;    // 32 KB
constexpr int GA_RAW_B = GA_NT * G_KBLK * 4;     // 32 KB
constexpr int GA_RAW_STAGE = GA_RAW_A + GA_RAW_B;
constexpr int GA_F16_A = TILE_M * 128;           // 16 KB
constexpr int GA_F16_B = GA_NT * 128;            // 16 KB
constexpr int GA_F16_STAGE = GA_F16_A + GA_F16_B;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;     // src-size 0: the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void lds8(uint32_t addr, float* v) {
  float4 a, b;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(addr));
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(addr + 16));
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

template <bool TA, bool TB, bool SPLIT>
__global__ void __launch_bounds__(G_THREADS, 1) gemm_tc_async_kernel(const GemmParams p) {
  constexpr int FST = SPLIT ? 1 : 2;                                   // fp16 stages
  constexpr int F16_STAGE = SPLIT ? 2 * GA_F16_STAGE : GA_F16_STAGE;   // hi (+ lo) tiles
  constexpr int LO_OFF = GA_F16_STAGE;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t f16_base = smem_base, raw_base = smem_base + FST * F16_STAGE;
  const uint32_t misc_base = raw_base + 2 * GA_RAW_STAGE;
  uint8_t* misc_gen = smem_gen + (misc_base - smem_base);
  const uint32_t bar_full = misc_base, bar_empty = misc_base + 64, bar_t_full = misc_base + 128, bar_t_empty = misc_base + 144;
  uint32_t* tmem_ptr_smem = (uint32_t*)(misc_gen + 160);
  float* s_epi = (float*)(misc_gen + 256);      // [4 epilogue warps] staging rows (G_EPI_WARP_BYTES each)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.tiles_m * p.tiles_n * p.splits;

  // reduction extent: K, or the device-side count of listed rows; the split ranges follow it
  const int Keff = p.kcount ? min(__ldg(p.kcount), p.K) : p.K;
  const int kps = p.kcount ? max(G_KBLK, ((Keff + p.splits - 1) / p.splits + G_KBLK - 1) / G_KBLK * G_KBLK) : p.k_per_split;
  struct Tile { int m0, n0, nt, nmma, z, kbeg, kend, nkb; };
  auto tile_of = [&](int t) {
    Tile x;
    const int tn = t % p.tiles_n, tm = (t / p.tiles_n) % p.tiles_m;
    x.z = t / (p.tiles_n * p.tiles_m);
    x.m0 = tm * TILE_M;
    x.n0 = tn * p.ntile;
    x.nt = min(p.ntile, p.N - x.n0);
    x.nmma = (x.nt + 15) & ~15;
    x.kbeg = x.z * kps;
    x.kend = min(Keff, x.kbeg + kps);
    x.nkb = x.kend > x.kbeg ? (x.kend - x.kbeg + G_KBLK - 1) / G_KBLK : 0;
    return x;
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < FST; ++s) {
      mbar_init(bar_full + 8 * s, G_PRODUCERS / 32);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_t_full + 8 * a, 1);
      mbar_init(bar_t_empty + 8 * a, 4);
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(256)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    {   // the whole warp runs the loop, one elected lane issues (see elect_one)
      const bool leader = elect_one();
      int s = 0, acc = 0;
      uint32_t ph = 0, pht[2] = {0, 0};
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const Tile x = tile_of(t);
        const uint32_t idesc = make_idesc(TILE_M, x.nmma, true) | (TA ? (1u << 15) : 0u) | (!TB ? (1u << 16) : 0u);
        mbar_wait(bar_t_empty + 8 * acc, pht[acc] ^ 1, 24);
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * 128;
        uint32_t accum = 0;
        for (int kb = 0; kb < x.nkb; ++kb) {
          mbar_wait(bar_full + 8 * s, ph, 21);
          tc_fence_after();
          const uint32_t a_addr = f16_base + s * F16_STAGE, b_addr = a_addr + GA_F16_A;
          if (leader) {
#pragma unroll
            for (int kk = 0; kk < G_KBLK / 16; ++kk) {
              const uint64_t ad = TA ? make_desc_mn128(a_addr + kk * 2048, 8192) : make_desc_k128(a_addr + kk * 32);
              const uint64_t bd = TB ? make_desc_k128(b_addr + kk * 32) : make_desc_mn128(b_addr + kk * 2048, 8192);
              umma_bf16(tacc, ad, bd, idesc, accum);
              accum = 1;
              if (SPLIT) {
                const uint64_t al = TA ? make_desc_mn128(a_addr + LO_OFF + kk * 2048, 8192) : make_desc_k128(a_addr + LO_OFF + kk * 32);
                const uint64_t bl = TB ? make_desc_k128(b_addr + LO_OFF + kk * 32) : make_desc_mn128(b_addr + LO_OFF + kk * 2048, 8192);
                umma_bf16(tacc, al, bd, idesc, 1);
                umma_bf16(tacc, ad, bl, idesc, 1);
              }
            }
            umma_commit(bar_empty + 8 * s);
          }
          accum = 1;
          __syncwarp();
          if (++s == FST) { s = 0; ph ^= 1; }
        }
        if (leader) umma_commit(bar_t_full + 8 * acc);
        __syncwarp();
        pht[acc] ^= 1;
        acc ^= 1;
      }
    }
  } else if (warp >= 1 && warp < 9) {
    // ---- producers
    const int pt = threadIdx.x - 32;         // 0..255
    struct Iter { int t, kb; Tile x; };
    auto first = [&]() {
      Iter it;
      it.t = blockIdx.x; it.kb = 0;
      while (it.t < n_tiles && (it.x = tile_of(it.t)).nkb == 0) it.t += gridDim.x;
      return it;
    };
    auto advance = [&](Iter& it) {
      if (it.t >= n_tiles) return;
      if (++it.kb < it.x.nkb) return;
      it.kb = 0;
      it.t += gridDim.x;
      while (it.t < n_tiles && (it.x = tile_of(it.t)).nkb == 0) it.t += gridDim.x;
    };
    // listed reduction rows (GemmParams::kidx) of this thread's 8 chunk rows of a K block: fetched one K block ahead of
    // the copies that use them (a dependent index load in front of every cp.async made the kernel slower than the dense
    // sum over twice the rows)
    int krows[8];
    auto fetch_rows = [&](const Iter& it) {
      if (!p.kidx || it.t >= n_tiles) return;
      const int k0 = it.x.kbeg + it.kb * G_KBLK;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int kr = (pt >> 5) + 8 * i;
        krows[i] = (k0 + kr < it.x.kend) ? __ldg(p.kidx + k0 + kr) : 0;
      }
    };
    // request the raw fp32 tiles of K block `it` into raw stage rs (a group is committed even when nothing is left)
    auto issue = [&](const Iter& it, int rs) {
      if (it.t < n_tiles) {
        const Tile& x = it.x;
        const int k0 = x.kbeg + it.kb * G_KBLK;
        const uint32_t ra = raw_base + rs * GA_RAW_STAGE, rb = ra + GA_RAW_A;
#pragma unroll
        for (int i = 0; i < 8; ++i) {            // A: 2048 16-byte chunks
          const int ch = pt + i * G_PRODUCERS;
          if (!TA) {
            const int r = ch >> 4, c = ch & 15;
            const bool ok = (x.m0 + r < p.M) && (k0 + 4 * c < x.kend);
            cp_async16(ra + r * 256 + c * 16, p.A + (long long)(ok ? x.m0 + r : 0) * p.lda + (ok ? k0 + 4 * c : 0), ok);
          } else {
            const int kr = ch >> 5, c = ch & 31;
            const bool ok = (k0 + kr < x.kend) && (x.m0 + 4 * c < p.M);
            const int krow = !ok ? 0 : (p.kidx ? krows[i] : k0 + kr);
            cp_async16(ra + kr * 512 + c * 16, p.A + (long long)krow * p.lda + (ok ? x.m0 + 4 * c : 0), ok);
          }
        }
        if (TB) {
          for (int ch = pt; ch < x.nmma * 16; ch += G_PRODUCERS) {
            const int r = ch >> 4, c = ch & 15;
            const bool ok = (r < x.nt) && (k0 + 4 * c < x.kend);
            cp_async16(rb + r * 256 + c * 16, p.B + (long long)(ok ? x.n0 + r : 0) * p.ldb + (ok ? k0 + 4 * c : 0), ok);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int ch = pt + i * G_PRODUCERS, kr = ch >> 5, c = ch & 31;
            const bool ok = (k0 + kr < x.kend) && (4 * c < x.nt);
            const int krow = !ok ? 0 : (p.kidx ? krows[i] : k0 + kr);
            cp_async16(rb + kr * 512 + c * 16, p.B + (long long)krow * p.ldb + (ok ? x.n0 + 4 * c : 0), ok);
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    Iter cur = first(), pre = cur;
    fetch_rows(pre);
    issue(pre, 0); advance(pre); fetch_rows(pre);
    issue(pre, 1); advance(pre); fetch_rows(pre);
    int s = 0, rs = 0;
    uint32_t ph = 0;
    while (cur.t < n_tiles) {
      const Tile& x = cur.x;
      asm volatile("cp.async.wait_group 1;" ::: "memory");      // this thread's copies of the current K block have landed
      asm volatile("bar.sync 1, 256;" ::: "memory");            // ... and everyone else's
      if (lane == 0) mbar_wait(bar_empty + 8 * s, ph ^ 1, 22);
      __syncwarp();
      const uint32_t ra = raw_base + rs * GA_RAW_STAGE, rb = ra + GA_RAW_A;
      const uint32_t a_addr = f16_base + s * F16_STAGE, b_addr = a_addr + GA_F16_A;
      const int bgroups = (x.nmma + 63) >> 6;
      const int nb_pieces = TB ? x.nmma * 8 : bgroups * 512;
#pragma unroll
      for (int i = 0; i < 4; ++i) {            // A: 1024 pieces of 8 elements
        const int pi = pt + i * G_PRODUCERS, c = pi & 7, r = pi >> 3;
        float v[8];
        uint4 lo;
        uint32_t src, off;
        if (!TA) { src = ra + r * 256 + c * 32; off = (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }
        else { const int g = r >> 6, kr = r & 63; src = ra + kr * 512 + (g * 64 + 8 * c) * 4; off = (uint32_t)(g * 8192 + kr * 128 + ((c ^ (kr & 7)) << 4)); }
        lds8(src, v);
        const uint4 hi = cvt_piece<SPLIT>(v, lo);
        sts128(a_addr + off, hi);
        if (SPLIT) sts128(a_addr + LO_OFF + off, lo);
      }
      for (int pi = pt; pi < nb_pieces; pi += G_PRODUCERS) {
        const int c = pi & 7, r = pi >> 3;
        float v[8];
        uint4 lo;
        uint32_t src, off;
        if (TB) { src = rb + r * 256 + c * 32; off = (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }
        else { const int g = r >> 6, kr = r & 63; src = rb + kr * 512 + (g * 64 + 8 * c) * 4; off = (uint32_t)(g * 8192 + kr * 128 + ((c ^ (kr & 7)) << 4)); }
        lds8(src, v);
        const uint4 hi = cvt_piece<SPLIT>(v, lo);
        sts128(b_addr + off, hi);
        if (SPLIT) sts128(b_addr + LO_OFF + off, lo);
      }
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");            // the raw stage is fully consumed: refill it
      issue(pre, rs); advance(pre); fetch_rows(pre);
      if (lane == 0) mbar_arrive(bar_full + 8 * s);
      if (++s == FST) { s = 0; ph ^= 1; }
      rs ^= 1;
      advance(cur);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp >= 9) {
    // ---- epilogue (TMEM lane quarter = warp % 4)
    const int q = warp & 3;
    int acc = 0;
    uint32_t pht[2] = {0, 0};
    const bool split = p.splits > 1;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const Tile x = tile_of(t);
      mbar_wait(bar_t_full + 8 * acc, pht[acc], 23);
      pht[acc] ^= 1;
      tc_fence_after();
      float* cbase = split ? p.partial + (long long)x.z * p.M * p.N : p.C;
      const long long ldo = split ? (long long)p.N : p.ldc;
      const bool vec_st = (ldo % 4 == 0) && ((((uintptr_t)cbase) & 15) == 0) && ((x.n0 & 3) == 0);
      for (int c0 = 0; c0 < x.nmma; c0 += 32) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + acc * 128 + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
        if (x.nmma - c0 >= 32) { TMEM_LD_32(taddr, r); } else { TMEM_LD_16(taddr, r); }
        tmem_ld_wait();
        const int ncols = min(32, x.nt - c0);
        if (ncols > 0)
          gemm_epi_store(s_epi + (warp - 9) * (G_EPI_WARP_BYTES / 4), lane, r, x.nkb > 0, cbase, ldo, x.m0 + q * 32, p.M,
                         x.n0 + c0, ncols, p.bias, p.flags, !split, vec_st);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_t_empty + 8 * acc);
      acc ^= 1;
    }
  }
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
  }
}

__global__ void gemm_tc_splitk_reduce_kernel(int M, int N, int splits, const float* __restrict__ partial,
                                             float* __restrict__ C, long long ldc, const float* __restrict__ bias,
                                             int flags) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * N) return;
  int gm = (int)(i / N), gn = (int)(i % N);
  float v = 0.f;
  for (int s = 0; s < splits; ++s) v += partial[(long long)s * M * N + i];
  if (bias) v += bias[gn];
  if (flags & LSTUR_GEMM_ACCUM) v += C[(long long)gm * ldc + gn];
  if (flags & LSTUR_GEMM_RELU) v = fmaxf(v, 0.f);
  C[(long long)gm * ldc + gn] = v;
}

}  // namespace tc
}  // namespace lstur

using namespace lstur;

static void gemm_tc_tiling(int M, int N, int K, int* ntile, int* splits, int max_nt = 256) {
  int nparts = (N + max_nt - 1) / max_nt;
  int nt = ((N + nparts - 1) / nparts + 15) & ~15;
  if (nt > max_nt) nt = max_nt;
  long long tiles = (long long)((M + tc::TILE_M - 1) / tc::TILE_M) * ((N + nt - 1) / nt);
  int sp = 1;
  if (tiles < 148 && K >= 2048) {
    sp = (int)(148 / tiles);
    int maxs = K / 512;
    if (sp > maxs) sp = maxs;
    if (sp < 1) sp = 1;
  }
  *ntile = nt;
  *splits = sp;
}

extern "C" size_t lstur_gemm_tc_workspace_bytes(int M, int N, int K) {
  int nt, sp, sp2;
  gemm_tc_tiling(M, N, K, &nt, &sp);
  gemm_tc_tiling(M, N, K, &nt, &sp2, tc::GA_NT);
  if (sp2 > sp) sp = sp2;
  size_t b = sp > 1 ? (size_t)sp * M * N * sizeof(float) : 0;
  // pre-packed weight-operand image (hi + lo tiles per (n tile, K block)) for the large-M GEMMs
  gemm_tc_tiling(M, N, K, &nt, &sp);
  const size_t img = (size_t)((N + nt - 1) / nt) * ((K + tc::G_KBLK - 1) / tc::G_KBLK) * 2 * tc::G_BIMG_TILE;
  if (M >= 1024 && img > b) b = img;
  return b;
}

static int gemm_tc_impl(int transA, int transB, int M, int N, int K, const float* A, long long lda, const float* B,
                        long long ldb, float* C, long long ldc, const float* bias, int flags, void* workspace,
                        size_t workspace_bytes, const int* kidx, const int* kcount, cudaStream_t stream,
                        const int* midx = nullptr, const int* mcount = nullptr);

// Same contract as lstur_gemm_f32 (fp32 in / fp32 out); operands are rounded to fp16 inside the kernel.
extern "C" int lstur_gemm_tc(int transA, int transB, int M, int N, int K, const float* A, long long lda, const float* B,
                             long long ldb, float* C, long long ldc, const float* bias, int flags, void* workspace,
                             size_t workspace_bytes, cudaStream_t stream) {
  return gemm_tc_impl(transA, transB, M, N, K, A, lda, B, ldb, C, ldc, bias, flags, workspace, workspace_bytes, nullptr, nullptr,
                      stream);
}

// C[M,N] = sum over the listed rows k = k_rows[0 .. *k_count) of A[k, :M]^T B[k, :N]   (A, B stored [K, .]; k_rows ascending,
// k_count a device scalar <= K).  The weight gradients of the step reduce over (user, step) or title rows of which the
// masked ones are identically zero: summing the live rows only is the same sum (other than fp32 reassociation across the
// split-K ranges).  Falls back to the full range when the operands do not meet the 16-byte staging conditions.
extern "C" int lstur_gemm_tc_tn_rows(int M, int N, int K, const float* A, long long lda, const float* B, long long ldb, float* C,
                                     long long ldc, const int* k_rows, const int* k_count, void* workspace,
                                     size_t workspace_bytes, cudaStream_t stream) {
  return gemm_tc_impl(1, 0, M, N, K, A, lda, B, ldb, C, ldc, nullptr, 0, workspace, workspace_bytes, k_rows, k_count, stream);
}

// C[m, :] = (A[m, :K] . op(B)) (+ bias) (relu) for the listed rows m = m_rows[0 .. *m_count) only (A stored [M, K]; m_rows
// ascending device ints, m_count a device scalar <= M); the other rows of C are left untouched.  Used where half of the
// rows are padding whose result nobody reads (or whose result is a constant filled in separately).
extern "C" int lstur_gemm_tc_mrows(int transB, int M, int N, int K, const float* A, long long lda, const float* B, long long ldb,
                                   float* C, long long ldc, const float* bias, int flags, const int* m_rows, const int* m_count,
                                   void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return gemm_tc_impl(0, transB, M, N, K, A, lda, B, ldb, C, ldc, bias, flags, workspace, workspace_bytes, nullptr, nullptr, stream,
                      m_rows, m_count);
}

static int gemm_tc_impl(int transA, int transB, int M, int N, int K, const float* A, long long lda, const float* B,
                        long long ldb, float* C, long long ldc, const float* bias, int flags, void* workspace,
                        size_t workspace_bytes, const int* kidx, const int* kcount, cudaStream_t stream,
                        const int* midx, const int* mcount) {
  LSTUR_REQUIRE(M >= 0 && N >= 0 && K >= 0, "lstur_gemm_tc");
  if (M == 0 || N == 0) return LSTUR_OK;
  tc::GemmParams p;
  int splits;
  // cp.async staging needs every 16-byte chunk of an operand row to be aligned and entirely inside or outside the matrix
  const bool rows16 = (lda % 4 == 0) && (ldb % 4 == 0) && ((((uintptr_t)A) & 15) == 0) && ((((uintptr_t)B) & 15) == 0) &&
                      ((transA ? M : K) % 4 == 0) && ((transB ? K : N) % 4 == 0);
  // Measured at the LSTUR shapes (tools/perf_gemm.py): the cp.async ring wins for the long-K weight-gradient GEMMs
  // (A transposed, split-K: 192 -> 106 us), the register-staged kernel with its wider N tile for the short-K ones.
  const bool use_async = rows16 && K > 0 && transA;
  gemm_tc_tiling(M, N, K, &p.ntile, &splits, use_async ? tc::GA_NT : 256);
  size_t need = splits > 1 ? (size_t)splits * M * N * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace)) splits = 1;
  int kps = ((K + splits - 1) / splits + tc::G_KBLK - 1) / tc::G_KBLK * tc::G_KBLK;
  if (kps == 0) kps = tc::G_KBLK;
  splits = K > 0 ? (K + kps - 1) / kps : 1;
  p.M = M; p.N = N; p.K = K; p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc; p.bias = bias;
  p.flags = flags; p.k_per_split = kps; p.partial = (float*)workspace;
  p.bimg = nullptr; p.nkb_total = (K + tc::G_KBLK - 1) / tc::G_KBLK;
  p.kidx = use_async ? kidx : nullptr;            // the row list is honoured by the cp.async kernel only (else: all K rows)
  p.kcount = use_async ? kcount : nullptr;
  p.midx = nullptr; p.mcount = nullptr;
  p.vec_ok = (lda % 4 == 0) && (ldb % 4 == 0) && ((((uintptr_t)A) & 15) == 0) && ((((uintptr_t)B) & 15) == 0);
  const bool split3 = (flags & LSTUR_GEMM_PRECISE) != 0;
  size_t smem = 1024 + (split3 ? (size_t)2 * tc::G_STAGE_BYTES_S3 : (size_t)tc::G_STAGES * tc::G_STAGE_BYTES) + 256 +
                4 * tc::G_EPI_WARP_BYTES;
  static bool attr = false;
  if (!attr) {
    const int big = 1024 + 2 * tc::G_STAGE_BYTES_S3 + 256 + 4 * tc::G_EPI_WARP_BYTES;
    cudaError_t e = cudaSuccess;
#define SETATTR(TA_, TB_, S_) \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::gemm_tc_kernel<TA_, TB_, S_>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)
    SETATTR(false, false, false); SETATTR(true, false, false); SETATTR(false, true, false); SETATTR(true, true, false);
    SETATTR(false, false, true); SETATTR(true, false, true); SETATTR(false, true, true); SETATTR(true, true, true);
#undef SETATTR
    if (e != cudaSuccess) {
      set_error("lstur_gemm_tc: cannot opt in to %d B of shared memory: %s", big, cudaGetErrorString(e));
      return LSTUR_ERR_CUDA;
    }
    attr = true;
  }
  p.tiles_n = (N + p.ntile - 1) / p.ntile;
  p.tiles_m = (M + tc::TILE_M - 1) / tc::TILE_M;
  p.splits = splits;
  if (midx && mcount && !use_async && !transA && splits == 1) { p.midx = midx; p.mcount = mcount; }   // else: every row (a superset)
  // Large-M GEMMs against a small weight matrix (GRU input projection and its input gradient, scorer Dense layers):
  // pack B once per call into stage-layout fp16 tiles; the CTAs then fetch it with bulk copies.
  const size_t img_bytes = (size_t)p.tiles_n * p.nkb_total * (split3 ? 2 : 1) * tc::G_BIMG_TILE;
  if (!use_async && !transA && splits == 1 && M >= 1024 && K > 0 && workspace && img_bytes <= workspace_bytes) {
    dim3 pg((unsigned)p.nkb_total, (unsigned)p.tiles_n);
    uint8_t* img = (uint8_t*)workspace;
    if (transB) {
      if (split3) tc::gemm_pack_b_kernel<true, true><<<pg, 256, 0, stream>>>(N, K, B, ldb, p.ntile, p.vec_ok, img);
      else tc::gemm_pack_b_kernel<true, false><<<pg, 256, 0, stream>>>(N, K, B, ldb, p.ntile, p.vec_ok, img);
    } else {
      if (split3) tc::gemm_pack_b_kernel<false, true><<<pg, 256, 0, stream>>>(N, K, B, ldb, p.ntile, p.vec_ok, img);
      else tc::gemm_pack_b_kernel<false, false><<<pg, 256, 0, stream>>>(N, K, B, ldb, p.ntile, p.vec_ok, img);
    }
    LSTUR_CHECK_LAUNCH("lstur_gemm_tc(pack B)");
    p.bimg = img;
  }
  const long long n_tiles = (long long)p.tiles_m * p.tiles_n * splits;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  dim3 grid((unsigned)(n_tiles < sms ? n_tiles : sms));
  const size_t smem_async = 1024 + (size_t)2 * tc::GA_F16_STAGE + (size_t)2 * tc::GA_RAW_STAGE + 256 + 4 * tc::G_EPI_WARP_BYTES;
  static bool attr_async = false;
  if (use_async && !attr_async) {
    cudaError_t e = cudaSuccess;
#define SETATTR(TA_, TB_, S_) \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::gemm_tc_async_kernel<TA_, TB_, S_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_async)
    SETATTR(false, false, false); SETATTR(true, false, false); SETATTR(false, true, false); SETATTR(true, true, false);
    SETATTR(false, false, true); SETATTR(true, false, true); SETATTR(false, true, true); SETATTR(true, true, true);
#undef SETATTR
    if (e != cudaSuccess) {
      set_error("lstur_gemm_tc: cannot opt in to %zu B of shared memory: %s", smem_async, cudaGetErrorString(e));
      return LSTUR_ERR_CUDA;
    }
    attr_async = true;
  }
#define LAUNCH(TA_, TB_)                                                                                \
  do {                                                                                                  \
    if (use_async) {                                                                                    \
      if (split3) tc::gemm_tc_async_kernel<TA_, TB_, true><<<grid, tc::G_THREADS, smem_async, stream>>>(p);  \
      else tc::gemm_tc_async_kernel<TA_, TB_, false><<<grid, tc::G_THREADS, smem_async, stream>>>(p);        \
    } else {                                                                                            \
      if (split3) tc::gemm_tc_kernel<TA_, TB_, true><<<grid, tc::G_THREADS, smem, stream>>>(p);         \
      else tc::gemm_tc_kernel<TA_, TB_, false><<<grid, tc::G_THREADS, smem, stream>>>(p);               \
    }                                                                                                   \
  } while (0)
  if (!transA && !transB) LAUNCH(false, false);
  else if (transA && !transB) LAUNCH(true, false);
  else if (!transA && transB) LAUNCH(false, true);
  else LAUNCH(true, true);
#undef LAUNCH
  LSTUR_CHECK_LAUNCH("lstur_gemm_tc");
  if (splits > 1) {
    long long n = (long long)M * N;
    tc::gemm_tc_splitk_reduce_kernel<<<cdiv(n, 256), 256, 0, stream>>>(M, N, splits, p.partial, C, ldc, bias, flags);
    LSTUR_CHECK_LAUNCH("lstur_gemm_tc(splitk_reduce)");
  }
  return LSTUR_OK;
}
