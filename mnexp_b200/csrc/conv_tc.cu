// News encoder on the 5th-gen tensor cores: word-embedding gather fused into the Conv1D implicit GEMM
// (tcgen05.mma, fp32 accumulator in TMEM) with bias + ReLU + pad mask + Masking + Dropout +
// additive-attention pooling fused in the epilogue; the Conv1D weight gradient; the Conv1D input gradient.
//
// Reference ops replaced (task/paper.py:141-158, models.py:474-489; SURVEY.md §2b k1-k6):
//   Embedding(mask_zero=False) -> Dropout -> Conv1D(F,3,'same',relu) -> pad-token mask ->
//   Masking -> Dropout -> SimpleAttentionMaskSupport, and their backward.
//
// GEMM view of the forward: D[m, f] = sum_{j<3} sum_e X[m+j-1, e] * Wc[j, e, f], m = token position.
//   M tile  = 128 rows = title slots of SLOT rows: 4 x 32 (L <= 31) or 2 x 64 (L <= 63).  A slot holds the L tokens
//             of a title + >= 1 zero row, which is both the right halo of its title and the left halo of the next
//             one; the rows before / after the tile are zero pads.
//   N       = F (<= 512 TMEM columns), computed as two FEATURE PASSES over K (columns [0, 2*n0h) then the rest), each
//             with its own accumulator barriers so that the epilogue drains one pass while the tensor core runs the other.
//   K       = 3 taps x Ep (E padded to a multiple of 64), pipeline block = 32 columns = one 64-byte swizzle row.
// CTA pairs (cta_group::2, M = 256): each CTA owns one 128-row token tile and stages half of the weight rows.
// A operand: producer warps gather each embedding row ONCE per tile and 32-column chunk (16 B loads, 4 lanes per row),
//   apply the input dropout mask, and store ONE copy of it in the canonical K-major SWIZZLE_64B layout (16 B chunk index
//   XOR (row>>1)&3); the three taps are read through descriptors that start one row earlier / later.  The tile's chunks
//   stay resident (A ring, one slot per chunk) until both feature passes have read them.
// B operand: the conv weights are re-packed per call into 16-bit K-major SWIZZLE_64B images in consumption order, so
//   one cp.async.bulk per (pass, chunk, tap) lands an MMA-ready tile in the B ring.
// Warp roles (640 threads): w0 weight loader, w1 TMEM alloc + MMA issuer (leader CTA), w2 (peer CTA) weight-landed
//   forwarder, w4-11 A producers, w12-19 epilogue (TMEM lane quarter = warp%4, feature half = (warp-12)/4).
// The input gradient (word-table training, task/paper.py:136) runs the SAME main loop with the roles of the operands
// changed: "embedding rows" are the rows of the dPre image, the weights are Wc transposed with the taps reversed,
// N = Ep and the epilogue only scales and stores 16-bit rows (see news_conv_tc_kernel, MODE_DGRAD).
#include <limits.h>
#include <stdlib.h>

#include "tc_common.cuh"

namespace lstur {
namespace tc {

constexpr int MODE_FWD = 0, MODE_DGRAD = 1;
constexpr int EPAD = 64;                      // embedding rows are padded to a multiple of 64 columns
constexpr int KBLK = 32;                      // K elements per pipeline block: 64-byte rows, SWIZZLE_64B
constexpr int ROWB = KBLK * 2;                // bytes per shared-memory row
constexpr int A_TAP_BYTES = TILE_M * ROWB;    // 8 KB
constexpr int TAPS = 3;
// A operand of one 32-column chunk: ONE copy of the tile's 128 rows between two 512-byte zero pads; the three taps are
// read through descriptors whose start address is shifted by -1 / 0 / +1 rows (the 64-byte swizzle is a function of the
// absolute shared-memory address, so a start anywhere inside the 512-byte-aligned image reads consistently; the pads
// supply the zero rows -1 and 128).  (Round 1 stored three shifted copies, 24 KB per chunk.)
constexpr int A_PAD = 512;
constexpr int A_STAGE_BYTES = A_TAP_BYTES + 2 * A_PAD;   // 9 KB per chunk slot

// K-major SWIZZLE_64B descriptor: rows of 64 B, 8-row atoms of 512 B (16B chunk index XOR (row>>1)&3)
__device__ __forceinline__ uint64_t make_desc_k64(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
constexpr int THREADS = 640;                  // w0 loader, w1 MMA issuer, w4-11 A producers, w12-19 epilogue

// ------------------------------------------------------------------ operand packing kernels
// fp32 (V,E) -> 16-bit (V,Ep), zero-padded columns.  One thread per 16-byte output piece (8 columns).
__global__ void pack_emb_bf16_kernel(long long V, int E, int Ep, const float* __restrict__ src,
                                     uint16_t* __restrict__ dst, bool fp16) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ppr = Ep >> 3;                       // pieces per row (Ep % 64 == 0)
  if (i >= V * ppr) return;
  const long long v = i / ppr;
  const int e0 = (int)(i % ppr) * 8;
  float x[8];
  if ((E & 3) == 0 && e0 + 8 <= E) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(src + v * E + e0)), b = __ldg(reinterpret_cast<const float4*>(src + v * E + e0 + 4));
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = e0 + k < E ? __ldg(src + v * E + e0 + k) : 0.f;
  }
  uint32_t w[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) w[k] = (uint32_t)to16(x[2 * k], fp16) | ((uint32_t)to16(x[2 * k + 1], fp16) << 16);
  *reinterpret_cast<uint4*>(dst + v * Ep + e0) = make_uint4(w[0], w[1], w[2], w[3]);
}

// conv_w fp32 (3,E,F) -> per K block i = c*3 + j an [F rows][32 k] 16-bit image, K-major, 64B-swizzled.
__global__ void pack_conv_w_kernel(int E, int F, int EC, const float* __restrict__ Wc, uint16_t* __restrict__ img,
                                   bool fp16) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long per_blk = (long long)F * KBLK;
  if (i >= per_blk * EC * TAPS) return;
  int blk = (int)(i / per_blk);
  int rem = (int)(i % per_blk);
  int f = rem / KBLK, kk = rem % KBLK;
  int c = blk / TAPS, j = blk % TAPS;
  int e = c * KBLK + kk;
  float v = e < E ? Wc[((long long)j * E + e) * F + f] : 0.f;
  long long byte = (long long)f * ROWB + ((((kk >> 3) ^ ((f >> 1) & 3)) << 4) | ((kk & 7) << 1));
  img[blk * per_blk + byte / 2] = to16(v, fp16);
}

// Input-gradient weights: dX[m, e] = sum_j sum_f dPre[m+1-j, f] * Wc[j, e, f].  The kernel's tap tile j' holds the rows
// shifted by j'-1, so its weights are Wc[2-j'] transposed; K runs over the dPre IMAGE's column order: chunk
// c = half * cph + ch covers conv features f = half*Fh + ch*32 + kk (zero weights where ch*32 + kk >= Fh).
// Per K block i = c*3 + j' an [Eo rows][32 k] 16-bit image, K-major, 64B-swizzled (Eo = padded output width).
__global__ void pack_conv_w_dgrad_kernel(int E, int F, int Eo, int cph, const float* __restrict__ Wc,
                                         uint16_t* __restrict__ img, bool fp16) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_blk = (long long)Eo * KBLK;
  if (i >= per_blk * 2 * cph * TAPS) return;
  const int blk = (int)(i / per_blk), rem = (int)(i % per_blk);
  const int e = rem / KBLK, kk = rem % KBLK;
  const int c = blk / TAPS, jp = blk % TAPS;
  const int Fh = F >> 1, half = c / cph, ch = c % cph, fl = ch * KBLK + kk;
  float v = 0.f;
  if (e < E && fl < Fh) v = Wc[((long long)(TAPS - 1 - jp) * E + e) * F + half * Fh + fl];
  const long long byte = (long long)e * ROWB + ((((kk >> 3) ^ ((e >> 1) & 3)) << 4) | ((kk & 7) << 1));
  img[blk * per_blk + byte / 2] = to16(v, fp16);
}

struct FwdParams {
  int n_titles, L, F, EC, Ep, V;
  const int* tok;                 // (n_titles, L)
  const uint16_t* emb;            // (V, Ep) fp16 or bf16
  const uint16_t* wimg;           // EC*3 blocks of F*32 (EC = Ep/32)
  const float* conv_b;            // (F)
  const float* att_w;             // (F)
  const float* att_b;             // (1)
  uint16_t* c_out;                // (n_titles, L, F) attention input (fp16/bf16), saved for backward
  float* pooled;                  // (n_titles, F)
  float* att_a;                   // (n_titles, L) or null
  float* att_wt;                  // (n_titles, L) or null
  uint32_t drop_thr16;            // 0 = no dropout (quad stream threshold, 15 bits)
  uint32_t drop_addend;           // quad_addend(threshold)
  float inv_keep;
  uint32_t seed_x, seed_c;
  int nstages;                    // depth of the weight-stage ring (2 .. DEF_STAGES)
  long long* trace;               // optional: wait cycles of pair 0's MMA issuer (tools/perf_fwd.py)
  uint8_t* xmask;                 // optional (n_titles, L, Ep/8): keep bits of the X-dropout, one byte per 16-byte piece, so
                                  // the weight-gradient kernel need not replay the hash (bit j / 4+j: low / high half of word j)
  // MODE_DGRAD (conv input gradient): the A rows are rows of the dPre image written by attn_bwd_img_kernel
  // (per title [F half][64-column group][SLOT rows][128 B], SWIZZLE_128B), K chunk c = (half, 32-column chunk ch) of it;
  // F is the OUTPUT width (Ep of the word table), EC = 2 * cph chunks, c_out receives (n_titles, L, F) 16-bit rows
  const uint8_t* dimg;
  int ngh, cph;                   // 64-column groups / 32-column chunks per half of the conv features
  float out_scale;                // dX16 = out_scale * accumulator
  // compacted title list (lstur_compact_titles): n_dev = device count of titles to process (<= n_titles), title_idx =
  // original index of every processed title (pooled rows are written there); both optional
  const int* n_dev;
  const int* title_idx;
};

// Shared memory: an A ring with one slot per 32-column chunk of the tile (EC slots of 9 KB, filled once per tile, read by
// both feature passes) and a B ring of weight stages (this CTA's rows of one (pass, chunk): 3 taps x n0h x 64 B).
constexpr int MAX_CHUNKS = 16;                // A slots / barrier slots
constexpr int DEF_STAGES = 3;                 // B stages (<= 8 barrier slots); fewer where shared memory runs out
// rows per CTA of feature pass 0 (pass 1 takes the other Fh - n0h): half of Fh rounded up to a multiple of 8, at most 128
__host__ __device__ constexpr int conv_n0h(int Fh) { return ((Fh + 15) / 16) * 8 > 128 ? 128 : ((Fh + 15) / 16) * 8; }

struct EpiCtx {
  float sx;                       // scale applied to the accumulator (input-dropout and conv-dropout keep scales)
  const float* s_bias;            // conv bias x conv-dropout keep scale (ReLU is positively homogeneous)
  const float* s_ka;
  uint32_t thr, base_lo, inner0, inner1;   // conv-dropout stream of this thread's token row (thr = quad_addend)
};

// Epilogue pass 1 for NC accumulator columns of one token row -> features [f0, f0+NC): scale + bias + ReLU (+ pad-token
// mask) -> conv dropout -> 16-bit C stored to global, attention-logit partial sum z (from the ROUNDED values, so forward
// and backward see the same C).  The conv-dropout keep SCALE is folded into the accumulator scale and the bias (ReLU is
// positively homogeneous), so dropping is a bitwise AND on the packed pair.
// Per-warp staging buffer that turns row-per-lane register tiles into coalesced global accesses: a lane holds 64 B of
// ITS token row, but a warp-wide 16-byte access with one row per lane touches 32 different 128-byte lines (and half of
// every 32-byte sector).  Through the buffer, 4 lanes cover the 64 B of one row, so an instruction touches 8 lines and
// only full sectors — the epilogue of the previous version was bound by exactly these L1 line transactions.
constexpr int STG_ROW_U4 = 5;                       // 4 pieces + 1 pad (80-byte rows: conflict-free 16-byte accesses)
constexpr int STG_WARP_BYTES = 32 * STG_ROW_U4 * 16;

struct RowIO {
  uint4* stg;            // this warp's staging buffer
  uint16_t* title;       // c_out of the FIRST token row of this warp (token t0 of its title; rows are F apart), or null
                         // if the title is invalid
  int F, L, lane;        // L = token rows of the title that this warp covers (title length - t0, may be <= 0)
  // write `npieces` 16-byte pieces of every lane's row (features [f0, f0 + 8*npieces)) to global
  __device__ __forceinline__ void store(const uint32_t* packed, int f0, int npieces) const {
#pragma unroll
    for (int g = 0; g < 4; ++g)
      if (g < npieces) stg[lane * STG_ROW_U4 + g] = make_uint4(packed[4 * g], packed[4 * g + 1], packed[4 * g + 2], packed[4 * g + 3]);
    __syncwarp();
    if (title) {
      const int piece = lane & 3;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = (lane >> 2) + 8 * i;
        if (row < L && piece < npieces)
          *reinterpret_cast<uint4*>(title + (long long)row * F + f0 + piece * 8) = stg[row * STG_ROW_U4 + piece];
      }
    }
    __syncwarp();
  }
  // issue the coalesced global loads of features [f0, f0 + 8*npieces) of the warp's rows
  __device__ __forceinline__ void load_issue(int f0, int npieces, uint4* v) const {
    const int piece = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = (lane >> 2) + 8 * i;
      v[i] = make_uint4(0, 0, 0, 0);
      if (title && row < L && piece < npieces) v[i] = *reinterpret_cast<const uint4*>(title + (long long)row * F + f0 + piece * 8);
    }
  }
  // hand every lane the 4 pieces of ITS row
  __device__ __forceinline__ void load_finish(const uint4* v, uint4* mine) const {
    const int piece = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i) stg[((lane >> 2) + 8 * i) * STG_ROW_U4 + piece] = v[i];
    __syncwarp();
#pragma unroll
    for (int g = 0; g < 4; ++g) mine[g] = stg[lane * STG_ROW_U4 + g];
    __syncwarp();
  }
};

// Epilogue pass 1 for NC accumulator columns of one token row -> features [f0, f0+NC): scale + bias + ReLU (+ pad-token
// mask) -> conv dropout -> 16-bit C stored to global, attention-logit partial sum z (from the ROUNDED values, so forward
// and backward see the same C).  The conv-dropout keep SCALE is folded into the accumulator scale and the bias (ReLU is
// positively homogeneous), so dropping is a bitwise AND on the packed pair.
// (Measured alternative, round 2: the keep bits generated ahead of time by the two idle warps into shared memory and
// expanded here through a 16-entry nibble table — one LDS.64 per quad instead of one hash.  The kernel got 6 % SLOWER
// (0.85 -> 0.90 ms at C3): this pass is bound by the shared-memory / load-store pipe (staging-buffer stores + loads, operand
// traffic of the producers for the next tile), not by integer issue slots, so the hash stays.)
template <bool FP16, bool DROP, int NC>
__device__ __forceinline__ void epi_pass1_chunk(const EpiCtx& ec, const RowIO& io, uint32_t taddr, int f0, bool live, float& z,
                                                uint32_t& anybits) {
  uint32_t r[NC];
  if (NC == 32) { TMEM_LD_32(taddr, r); } else if (NC == 16) { TMEM_LD_16(taddr, r); } else { TMEM_LD_8(taddr, r); }
  tmem_ld_wait();
  uint32_t packed[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) packed[i] = 0u;
  if (live) {
#pragma unroll
    for (int g = 0; g < NC / 4; ++g) {
      const float4 b4 = *reinterpret_cast<const float4*>(ec.s_bias + f0 + 4 * g);
      const float v0 = fmaf(__uint_as_float(r[4 * g + 0]), ec.sx, b4.x);
      const float v1 = fmaf(__uint_as_float(r[4 * g + 1]), ec.sx, b4.y);
      const float v2 = fmaf(__uint_as_float(r[4 * g + 2]), ec.sx, b4.z);
      const float v3 = fmaf(__uint_as_float(r[4 * g + 3]), ec.sx, b4.w);
      uint32_t p0 = pack16x2_relu<FP16>(v0, v1), p1 = pack16x2_relu<FP16>(v2, v3);   // ReLU fused into the conversion
      anybits |= p0 | p1;      // Masking(): any(C != 0) before the dropout, on the values the model actually stores
      if (DROP) {   // the keep scale is already folded into sx / s_bias: dropping is a pure zeroing of the packed halves
        const uint32_t lo = ec.base_lo + (uint32_t)((f0 >> 2) + g);          // quad index of features f0+4g .. +3
        uint32_t u0, u1;
        quad_hash(lo ^ (lo < ec.base_lo ? ec.inner1 : ec.inner0), u0, u1);
        p0 &= quad_mask(u0, ec.thr);
        p1 &= quad_mask(u1, ec.thr);
      }
      packed[2 * g] = p0;
      packed[2 * g + 1] = p1;
      const float4 k4 = *reinterpret_cast<const float4*>(ec.s_ka + f0 + 4 * g);
      z = fmaf(lo16<FP16>(p0), k4.x, z);
      z = fmaf(hi16<FP16>(p0), k4.y, z);
      z = fmaf(lo16<FP16>(p1), k4.z, z);
      z = fmaf(hi16<FP16>(p1), k4.w, z);
    }
  }
  io.store(packed, f0, NC / 8);
}
// Input-gradient epilogue for NC accumulator columns of one token row: scale, round to 16 bits (saturating), store.
template <bool FP16, int NC>
__device__ __forceinline__ void epi_dgrad_chunk(float scale, const RowIO& io, uint32_t taddr, int f0) {
  uint32_t r[NC];
  if (NC == 32) { TMEM_LD_32(taddr, r); } else if (NC == 16) { TMEM_LD_16(taddr, r); } else { TMEM_LD_8(taddr, r); }
  tmem_ld_wait();
  uint32_t packed[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) packed[i] = 0u;
#pragma unroll
  for (int g = 0; g < NC / 2; ++g)
    packed[g] = pack16x2_sat<FP16>(__uint_as_float(r[2 * g]) * scale, __uint_as_float(r[2 * g + 1]) * scale);
  io.store(packed, f0, NC / 8);
}
template <bool FP16>
__device__ __forceinline__ void epi_dgrad_segment(float scale, const RowIO& io, uint32_t trow, int ca, int f0, int n) {
  int c = 0;
  for (; c + 32 <= n; c += 32) epi_dgrad_chunk<FP16, 32>(scale, io, trow + ca + c, f0 + c);
  if (c + 16 <= n) { epi_dgrad_chunk<FP16, 16>(scale, io, trow + ca + c, f0 + c); c += 16; }
  if (c + 8 <= n) epi_dgrad_chunk<FP16, 8>(scale, io, trow + ca + c, f0 + c);
}

// one accumulator segment [ca, ca+n) -> features [f0, f0+n), n a multiple of 8
template <bool FP16, bool DROP>
__device__ __forceinline__ void epi_pass1_segment(const EpiCtx& ec, const RowIO& io, uint32_t trow, int ca, int f0, int n,
                                                  bool live, float& z, uint32_t& anybits) {
  int c = 0;
  for (; c + 32 <= n; c += 32) epi_pass1_chunk<FP16, DROP, 32>(ec, io, trow + ca + c, f0 + c, live, z, anybits);
  if (c + 16 <= n) { epi_pass1_chunk<FP16, DROP, 16>(ec, io, trow + ca + c, f0 + c, live, z, anybits); c += 16; }
  if (c + 8 <= n) epi_pass1_chunk<FP16, DROP, 8>(ec, io, trow + ca + c, f0 + c, live, z, anybits);
}

// CTA pairs (cta_group::2): CTA `rank` of a pair owns the token tile 2*tp + rank (its own A rows, its own 128 x F
// accumulator in tensor memory) and stages only the weight rows f in [rank*F/2, (rank+1)*F/2); the pair's MMAs
// (M = 256, issued by rank 0) read both halves, which halves the weight bytes every SM has to pull through its shared
// memory — the limiter of the single-CTA version (see DESIGN.md).  Accumulator column c holds feature
//   f = half*Fh + (c % n0h)         for c <  2*n0h    (half = c / n0h,  feature pass 0,  n0h ~ Fh/2, see conv_n0h)
//   f = half*Fh + n0h + (c' % n1h)  for c' = c-2*n0h  (half = c'/ n1h,  feature pass 1,  n1h = Fh - n0h)
// so an epilogue thread of column half `half` sees one contiguous feature range [half*Fh, (half+1)*Fh).
// FEATURE PASSES: a tile is computed as two passes over K, pass 0 into accumulator columns [0, 2*n0h) and pass 1 into
// [2*n0h, F): each pass has its own full / empty barrier, so the epilogue drains pass 0 while the tensor core runs pass 1
// and drains pass 1 under the next tile's pass 0 — the accumulator (F = 400 of 512 columns) cannot be double-buffered as
// a whole, and with a single pass the 8.6 k-cycle drain serialised with the 12 k MMA cycles of a tile.  Both passes read
// the SAME gathered rows: the tile's EC chunks stay in shared memory (one 9 KB slot each — affordable only since the taps
// are row-shifted views of one copy) until the second pass has consumed them; only the weight rows are streamed per pass.
// (Measured alternative: re-gathering the rows for the second pass — the producers' gather + dropout hash became the
// limiter, 1.04 ms instead of 0.78 ms at C3.)
template <bool FP16, bool DROP, int SLOT, int MODE>
__global__ void __launch_bounds__(THREADS, 1) news_conv_tc_kernel(const FwdParams p) {
  constexpr int TPT = TILE_M / SLOT;               // titles per 128-row tile
  constexpr bool DG = MODE == MODE_DGRAD;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int F = p.F, EC = p.EC, Fh = F >> 1;
  const int n0h = conv_n0h(Fh), n1h = Fh - n0h;
  const int NP = n1h > 0 ? 2 : 1;                                   // feature passes per tile
  // shared memory: [A ring: EC slots, one per 32-column chunk of the tile, each read by BOTH feature passes]
  //                [B ring: NB stages of this CTA's weight rows of one (pass, chunk): 3 taps x n0h rows x 64 B] [misc]
  const uint32_t b_tap_bytes = (uint32_t)n0h * ROWB;                // room for this CTA's weight rows of one tap of a pass
  const uint32_t b_stage_bytes = TAPS * b_tap_bytes;                // multiple of 512 (n0h % 8 == 0)
  const int NB = p.nstages;
  const uint32_t a_base = smem_base, b_base = a_base + (uint32_t)EC * A_STAGE_BYTES;
  const uint32_t misc_base = b_base + (uint32_t)NB * b_stage_bytes;
  uint8_t* misc_gen = smem_gen + (misc_base - smem_base);
  // barriers (8 B each): a_full[16] a_empty[16] b_full[8] b_empty[8] tmem_full[2] tmem_empty[2]
  const uint32_t bar_a_full = misc_base, bar_a_empty = misc_base + 128, bar_b_full = misc_base + 256, bar_b_empty = misc_base + 320;
  const uint32_t bar_t_full = misc_base + 384, bar_t_empty = misc_base + 400;
  uint32_t* tmem_ptr_smem = (uint32_t*)(misc_gen + 416);
  float* s_w = (float*)(misc_gen + 512);          // [128 rows] attention weights of the tile (SLOT == 64: pass 2 reads both warps' rows)
  float* s_z = (float*)(misc_gen + 1024);         // [2 parity][2 halves][128 rows]
  int* s_any = (int*)(misc_gen + 1024 + 2048);    // [2][2][128]
  float* s_bias = (float*)(misc_gen + 1024 + 4096);  // [F]  (x conv-dropout keep scale)
  float* s_ka = s_bias + F;                           // [F]
  uint4* s_stg = (uint4*)(misc_gen + 1024 + 4096 + (((size_t)2 * F * sizeof(float) + 15) & ~(size_t)15));   // [8 warps] staging

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  // number of titles: optionally a device scalar (the compacted count of live titles, lstur_compact_titles)
  const int n_titles = p.n_dev ? min(__ldg(p.n_dev), p.n_titles) : p.n_titles;
  const int n_tiles = (n_titles + TPT - 1) / TPT;
  const int n_tp = (n_tiles + 1) / 2;                  // tile pairs
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const float ik = DROP ? p.inv_keep : 1.f;

  if (threadIdx.x == 0) {
    for (int c = 0; c < EC; ++c) {
      // leader: the 8 producer warps of BOTH CTAs (the peer's arrive remotely).  The slot is free again once the MMAs of
      // every feature pass that read it have completed (one multicast commit per pass).
      mbar_init(bar_a_full + 8 * c, 16);
      mbar_init(bar_a_empty + 8 * c, NP);
    }
    for (int s = 0; s < NB; ++s) {
      // leader: its loader's expect_tx arrival + the peer's "my rows have landed" (remote arrive); peer: its loader only
      mbar_init(bar_b_full + 8 * s, crank == 0 ? 2 : 1);
      mbar_init(bar_b_empty + 8 * s, 1);   // multicast tcgen05.commit of the leader
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_t_full + 8 * a, 1);    // multicast tcgen05.commit of the leader
      mbar_init(bar_t_empty + 8 * a, 16);  // (leader) one arrival per epilogue warp of BOTH CTAs
    }
    fence_barrier_init();
  }
  if (!DG) {
    for (int f = threadIdx.x; f < F; f += THREADS) {
      s_bias[f] = p.conv_b[f] * ik;
      s_ka[f] = p.att_w[f];
    }
  }
  {   // zero rows before and after the A tile of every slot (never written afterwards)
    for (int i = threadIdx.x; i < EC * 2 * (A_PAD / 16); i += THREADS) {
      const int c = i / (2 * (A_PAD / 16)), r = i % (2 * (A_PAD / 16));
      const uint32_t off = r < A_PAD / 16 ? (uint32_t)r * 16 : (uint32_t)(A_PAD + A_TAP_BYTES) + (uint32_t)(r - A_PAD / 16) * 16;
      *reinterpret_cast<uint4*>(smem_gen + (size_t)c * A_STAGE_BYTES + off) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== weight loader (bulk copies of this CTA's rows of the pre-swizzled K blocks) ===========
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tp = pair; tp < n_tp; tp += n_pairs) {
        for (int fp = 0; fp < NP; ++fp) {
          const uint32_t rows_bytes = (uint32_t)(fp ? n1h : n0h) * ROWB;
          const size_t row0 = (size_t)crank * Fh + (fp ? n0h : 0);
          for (int c = 0; c < EC; ++c) {
            mbar_wait(bar_b_empty + 8 * s, ph ^ 1, 1);
            mbar_expect_tx(bar_b_full + 8 * s, TAPS * rows_bytes);
#pragma unroll
            for (int j = 0; j < TAPS; ++j)
              bulk_g2s(b_base + s * b_stage_bytes + j * b_tap_bytes,
                       (const uint8_t*)p.wimg + ((size_t)(c * TAPS + j) * F + row0) * ROWB, rows_bytes, bar_b_full + 8 * s);
            if (++s == NB) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 2) {
    // ===================== peer CTA: tell the leader that this CTA's weight rows of a stage have landed ============
    if (crank != 0 && lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tp = pair; tp < n_tp; tp += n_pairs)
        for (int k = 0; k < NP * EC; ++k) {
          mbar_wait(bar_b_full + 8 * s, ph, 7);
          mbar_arrive_remote(map_to_cta(bar_b_full + 8 * s, 0));
          if (++s == NB) { s = 0; ph ^= 1; }
        }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer of the pair =====================
    if (crank == 0) {      // the whole warp runs the loop, one elected lane issues (see elect_one)
      const bool leader = elect_one();
      const uint32_t idesc0 = make_idesc(2 * TILE_M, 2 * n0h, FP16), idesc1 = make_idesc(2 * TILE_M, n1h > 0 ? 2 * n1h : 16, FP16);
      int s = 0;
      uint32_t ph = 0, pht = 0, pha = 0;
      const bool tracing = p.trace != nullptr && blockIdx.x == 0;
      long long tw_acc = 0, tw_full = 0, t_start = tracing ? clock64() : 0;
      for (int tp = pair; tp < n_tp; tp += n_pairs) {
       for (int fp = 0; fp < NP; ++fp) {
        long long t0 = tracing ? clock64() : 0;
        mbar_wait(bar_t_empty + 8 * fp, pht ^ 1, 2);     // the epilogue has drained this pass's columns of the previous tile
        if (tracing) tw_acc += clock64() - t0;
        tc_fence_after();
        const uint32_t tacc = tmem_base + (fp ? 2 * n0h : 0);
        const uint32_t idesc = fp ? idesc1 : idesc0;
        uint32_t accum = 0;
        for (int c = 0; c < EC; ++c) {
          t0 = tracing ? clock64() : 0;
          if (fp == 0) mbar_wait(bar_a_full + 8 * c, pha, 3);     // the tile's rows of chunk c (they stay for pass 1)
          mbar_wait(bar_b_full + 8 * s, ph, 4);
          if (tracing) tw_full += clock64() - t0;
          tc_fence_after();
          if (leader) {
            const uint32_t a_slot = a_base + c * A_STAGE_BYTES, b_stage = b_base + s * b_stage_bytes;
#pragma unroll
            for (int j = 0; j < TAPS; ++j) {
              // tap j multiplies X[m + j - 1]: the single copy of the rows, read from row j - 1 on
              const uint32_t a_addr = a_slot + A_PAD + (uint32_t)((j - 1) * ROWB);
              const uint32_t b_addr = b_stage + j * b_tap_bytes;
#pragma unroll
              for (int kk = 0; kk < KBLK / 16; ++kk) {
                umma_f16_2cta(tacc, make_desc_k64(a_addr + kk * 32), make_desc_k64(b_addr + kk * 32), idesc, accum);
                accum = 1;
              }
            }
            umma_commit_2cta(bar_b_empty + 8 * s, 3);
            umma_commit_2cta(bar_a_empty + 8 * c, 3);
          }
          accum = 1;
          __syncwarp();
          if (++s == NB) { s = 0; ph ^= 1; }
        }
        if (leader) umma_commit_2cta(bar_t_full + 8 * fp, 3);
        __syncwarp();
       }
        pht ^= 1;
        pha ^= 1;
      }
      if (tracing && lane == 0) { p.trace[0] = tw_acc; p.trace[1] = tw_full; p.trace[2] = clock64() - t_start; }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== A producers: row gather -> the tile's chunk slots =====================
    // lane -> (row within a group of 8, 16-byte piece of the 64-byte row); loads for chunk c+1 (and the row ids of
    // the next tile) are issued before chunk c is hashed and stored, so L2 latency is off the critical path.
    // Eight warps share the tile's title slots (two warps per 32-row slot, four per 64-row slot), each thread two
    // rows per chunk (a producer warp's instruction stream is latency-bound, so the work is spread over more warps
    // rather than over more rows per thread).  A chunk is produced ONCE per tile and read by both feature passes.
    const int pw = (warp - 4) % TPT;         // title slot of the tile
    const int rh = (warp - 4) / TPT;         // which pair of the slot's 8-row groups
    const int rsub = lane >> 2, piece = lane & 3;
    uint32_t ph = 0;
    constexpr int kNoToken = INT_MIN;
    // MODE_FWD: id = token id (clamped when its embedding row is requested).  MODE_DGRAD: id = n * SLOT + t, the slot
    // row of the dPre image.
    auto load_ids = [&](int tp, int* ids) {
      const int n = (2 * tp + (int)crank) * TPT + pw;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int t = 8 * (2 * rh + i) + rsub;
        const bool ok = tp < n_tp && n < n_titles && t < p.L;
        // raw id: not inspected here (no stall on the load); clamped when the rows are requested
        if (DG) ids[i] = ok ? n * SLOT + t : kNoToken;
        else ids[i] = ok ? __ldg(p.tok + (long long)n * p.L + t) : kNoToken;
      }
    };
    auto load_rows = [&](const int* ids, int c, uint4* v) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        v[i] = make_uint4(0, 0, 0, 0);
        if (ids[i] != kNoToken) {
          if (DG) {
            const int n = ids[i] / SLOT, t = ids[i] % SLOT, half = c / p.cph, ch = c % p.cph;
            const uint8_t* src = p.dimg + ((long long)n * 2 * p.ngh + half * p.ngh + (ch >> 1)) * (SLOT * 128) + t * 128 +
                                 ((((ch & 1) * 4 + piece) ^ (t & 7)) << 4);
            v[i] = __ldg((const uint4*)src);
          } else {
            const int id = (ids[i] < 0 || ids[i] >= p.V) ? 0 : ids[i];
            v[i] = __ldg((const uint4*)(p.emb + (long long)id * p.Ep + c * KBLK + piece * 8));
          }
        }
      }
    };
    int ids[2], ids_next[2];
    uint4 v[2], v_next[2];
    uint32_t row_lo[2], row_in0[2], row_in1[2];
    load_ids(pair, ids);
    load_rows(ids, 0, v_next);
    for (int tp = pair; tp < n_tp; tp += n_pairs) {
      const int n = (2 * tp + (int)crank) * TPT + pw;
      for (int c = 0; c < EC; ++c) {
#pragma unroll
        for (int i = 0; i < 2; ++i) v[i] = v_next[i];
        if (c + 1 < EC) {
          load_rows(ids, c + 1, v_next);
          if (c + 2 == EC) load_ids(tp + n_pairs, ids_next);
        } else {
          if (EC == 1) load_ids(tp + n_pairs, ids_next);
          load_rows(ids_next, 0, v_next);
        }
        if (DROP) {
          if (c == 0) {   // per tile: pair index of column 0 of each of this thread's rows, inner hash of its high word
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const uint64_t rowquad = (((uint64_t)n * p.L + (8 * (2 * rh + i) + rsub)) * (uint64_t)p.Ep) >> 2;
              const uint32_t hi = (uint32_t)(rowquad >> 32);
              row_lo[i] = (uint32_t)rowquad;
              row_in0[i] = quad_key(hi, p.seed_x);
              row_in1[i] = row_lo[i] > 0xfffff000u ? quad_key(hi + 1u, p.seed_x) : row_in0[i];
            }
          }
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            if (ids[i] == kNoToken) continue;
            const uint32_t lo0 = row_lo[i] + (uint32_t)((c * KBLK + piece * 8) >> 2);
            uint32_t* w = reinterpret_cast<uint32_t*>(&v[i]);
            uint32_t keep = 0;
#pragma unroll
            for (int q = 0; q < 2; ++q) {     // two quads per 16-byte piece
              const uint32_t lo = lo0 + q;
              uint32_t u0, u1;
              quad_hash(lo ^ (lo < row_lo[i] ? row_in1[i] : row_in0[i]), u0, u1);
              const uint32_t m0 = quad_mask(u0, p.drop_addend), m1 = quad_mask(u1, p.drop_addend);
              w[2 * q] &= m0;
              w[2 * q + 1] &= m1;
              keep |= (m0 & (0x00010001u << (2 * q))) | (m1 & (0x00010001u << (2 * q + 1)));
            }
            // bits 0-3 (low halves of words 0-3) and 16-19 (high halves) -> one byte
            if (p.xmask)
              p.xmask[((long long)n * p.L + (8 * (2 * rh + i) + rsub)) * (p.Ep >> 3) + c * (KBLK / 8) + piece] =
                  (uint8_t)((keep | (keep >> 12)) & 0xffu);
          }
        }
        if (lane == 0) mbar_wait(bar_a_empty + 8 * c, ph ^ 1, 5);   // one poller per warp: both passes of the previous tile read it
        __syncwarp();
        const uint32_t slot_addr = a_base + c * A_STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int r = pw * SLOT + 8 * (2 * rh + i) + rsub;
          const uint32_t addr = slot_addr + A_PAD + r * ROWB + ((piece ^ ((r >> 1) & 3)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v[i].x), "r"(v[i].y), "r"(v[i].z), "r"(v[i].w)
                       : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (crank == 0) mbar_arrive(bar_a_full + 8 * c);
          else mbar_arrive_remote(map_to_cta(bar_a_full + 8 * c, 0));
        }
        if (c + 1 == EC) {
#pragma unroll
          for (int i = 0; i < 2; ++i) ids[i] = ids_next[i];
        }
      }
      ph ^= 1;
    }
  } else if (warp >= 12) {
    // ===================== epilogue =====================
    // Thread (q, lane) owns row 32q+lane of this CTA's tile = token t = (32q+lane) % SLOT of title slot (32q+lane) / SLOT;
    // the two feature halves of a row are handled by warps ew and ew+4 and combined through shared memory.
    const int ew = warp - 12, q = ew & 3, half = ew >> 2;
    const int f_beg = half * Fh, f_end = f_beg + Fh;
    const int slot = (q * 32) / SLOT, t0 = (q * 32) % SLOT;      // this warp's title slot, its first token
    uint32_t pht = 0;
    RowIO io;
    io.stg = s_stg + (size_t)ew * (STG_WARP_BYTES / 16);
    io.F = F; io.L = p.L - t0; io.lane = lane;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    if (DG) {
      // ---- input gradient: scale, round, store the 16-bit rows
      for (int tp = pair; tp < n_tp; tp += n_pairs) {
        const int n = (2 * tp + (int)crank) * TPT + slot;
        io.title = n < n_titles ? p.c_out + ((long long)n * p.L + t0) * F : nullptr;
        for (int fp = 0; fp < NP; ++fp) {
          mbar_wait(bar_t_full + 8 * fp, pht, 6);
          tc_fence_after();
          if (fp == 0) epi_dgrad_segment<FP16>(p.out_scale, io, trow, half * n0h, f_beg, n0h);
          else epi_dgrad_segment<FP16>(p.out_scale, io, trow, 2 * n0h + half * n1h, f_beg + n0h, n1h);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (crank == 0) mbar_arrive(bar_t_empty + 8 * fp);
            else mbar_arrive_remote(map_to_cta(bar_t_empty + 8 * fp, 0));
          }
        }
        pht ^= 1;
      }
    } else {
    // ---- forward: bias/ReLU/masks/dropout/attention pooling
    const float att_bias = p.att_b[0];
    EpiCtx ec;
    ec.sx = DROP ? p.inv_keep * p.inv_keep : 1.f;   // input-dropout and conv-dropout keep scales
    ec.s_bias = s_bias;
    ec.s_ka = s_ka;
    ec.thr = p.drop_addend;
    int par = 0;
    for (int tp = pair; tp < n_tp; tp += n_pairs) {
      const int n = (2 * tp + (int)crank) * TPT + slot, t = t0 + lane;
      const bool valid = n < n_titles && t < p.L;
      const long long m = (long long)n * p.L + t;
      const int tk = valid ? p.tok[m] : 0;
      io.title = n < n_titles ? p.c_out + ((long long)n * p.L + t0) * F : nullptr;
      if (DROP) {
        const uint64_t base = ((uint64_t)(valid ? m : 0) * (uint64_t)F) >> 2;     // F % 4 == 0: quad index of (m, f) = base + f/4
        ec.base_lo = (uint32_t)base;
        const uint32_t hi = (uint32_t)(base >> 32);
        ec.inner0 = quad_key(hi, p.seed_c);
        ec.inner1 = quad_key(hi + 1u, p.seed_c);
      }
      float z = 0.f;
      uint32_t vmax = 0u;      // OR of the packed pre-dropout values of this row half
      // ---- pass 1: drain this row's accumulator columns, one feature pass at a time (the tensor core meanwhile runs
      // the other pass / the next tile's first pass)
      for (int fp = 0; fp < NP; ++fp) {
        mbar_wait(bar_t_full + 8 * fp, pht, 6);
        tc_fence_after();
        epi_pass1_segment<FP16, DROP>(ec, io, trow, fp ? 2 * n0h + half * n1h : half * n0h, fp ? f_beg + n0h : f_beg, fp ? n1h : n0h,
                                      tk != 0, z, vmax);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (crank == 0) mbar_arrive(bar_t_empty + 8 * fp);
          else mbar_arrive_remote(map_to_cta(bar_t_empty + 8 * fp, 0));
        }
      }
      pht ^= 1;
      const int row = q * 32 + lane;
      s_z[(par * 2 + half) * 128 + row] = z;
      s_any[(par * 2 + half) * 128 + row] = vmax != 0u ? 1 : 0;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const float zt = s_z[(par * 2) * 128 + row] + s_z[(par * 2 + 1) * 128 + row];
      const int anyt = s_any[(par * 2) * 128 + row] | s_any[(par * 2 + 1) * 128 + row];
      const float a = tanhf(zt + att_bias);
      const float e = (valid && anyt) ? expf(a) : 0.f;
      float esum = e;
      if (SLOT == 64) {
        // the title's other 32 tokens belong to the neighbour warp (row ^ 32): the same exp() of their logits, so both
        // warps of a title arrive at the identical softmax denominator
        const int row2 = row ^ 32, t2 = (t0 ^ 32) + lane;
        const float zt2 = s_z[(par * 2) * 128 + row2] + s_z[(par * 2 + 1) * 128 + row2];
        const int any2 = s_any[(par * 2) * 128 + row2] | s_any[(par * 2 + 1) * 128 + row2];
        const float e2 = (n < n_titles && t2 < p.L && any2) ? expf(tanhf(zt2 + att_bias)) : 0.f;
        esum = t0 == 0 ? e + e2 : e2 + e;       // same operand order in both warps
      }
      par ^= 1;
      const float S = warp_sum(esum);
      const float w = e / (S + 1e-7f);
      if (half == 0 && valid) {
        if (p.att_a) p.att_a[m] = a;
        if (p.att_wt) p.att_wt[m] = w;
      }
      // ---- pass 2: pooled[n, f] = sum_t w_t * C[t, f].  The stored rows are re-read (this CTA's writes, L2) in the
      // coalesced mapping — lane (r8 = lane/4, piece = lane%4) holds piece `piece` of rows r8, r8+8, r8+16, r8+24 —
      // weighted with those rows' attention weights, and the 8 lanes that share a piece finish with a 3-stage
      // reduce-scatter (7 shuffles per 32 features): no shared-memory staging on this pass.
      // SLOT == 64: the two warps of a title split the 32-feature chunks between them (even / odd) and each sums all 64
      // rows (the neighbour's rows and weights become visible through a second barrier), so no cross-warp reduction.
      // pooled rows go to the title's ORIGINAL index when the kernel runs over a compacted title list
      const int n_out = (p.title_idx && n < n_titles) ? __ldg(p.title_idx + n) : n;
      constexpr int NRH = SLOT / 32;                 // 32-row halves of a title
      float wr[NRH][4];
      if (SLOT == 64) {
        if (half == 0) s_w[row] = w;
        asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
        for (int h = 0; h < NRH; ++h)
#pragma unroll
          for (int i = 0; i < 4; ++i) wr[h][i] = s_w[slot * SLOT + h * 32 + (lane >> 2) + 8 * i];
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) wr[0][i] = __shfl_sync(0xffffffffu, w, (lane >> 2) + 8 * i);
      }
      RowIO io2 = io;                                // pass-2 view: all rows of the title from token 0
      if (SLOT == 64) {
        io2.title = n < n_titles ? p.c_out + (long long)n * p.L * F : nullptr;
        io2.L = p.L;
      }
      const int c_first = f_beg + (SLOT == 64 ? (q & 1) * 32 : 0), c_step = SLOT == 64 ? 64 : 32;
      uint4 nxt[4];
      if (c_first < f_end) io2.load_issue(c_first, min(4, (f_end - c_first) >> 3), nxt);
      const int jfeat = ((lane >> 2) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 4) & 1);   // feature of the piece this lane ends with
      for (int c0 = c_first; c0 < f_end; c0 += c_step) {
        const int np = min(4, (f_end - c0) >> 3);
        float x[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = 0.f;
#pragma unroll
        for (int h = 0; h < NRH; ++h) {
          uint4 cur[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) cur[g] = nxt[g];
          // prefetch: the title's next 32 rows of this chunk, or the first rows of the next chunk
          if (h + 1 < NRH) {
            RowIO io3 = io2;
            io3.title = io2.title ? io2.title + (long long)32 * (h + 1) * F : nullptr;
            io3.L = io2.L - 32 * (h + 1);
            io3.load_issue(c0, np, nxt);
          } else if (c0 + c_step < f_end) {
            io2.load_issue(c0 + c_step, min(4, (f_end - c0 - c_step) >> 3), nxt);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float wi = wr[h][i];
            x[0] = fmaf(wi, lo16<FP16>(cur[i].x), x[0]); x[1] = fmaf(wi, hi16<FP16>(cur[i].x), x[1]);
            x[2] = fmaf(wi, lo16<FP16>(cur[i].y), x[2]); x[3] = fmaf(wi, hi16<FP16>(cur[i].y), x[3]);
            x[4] = fmaf(wi, lo16<FP16>(cur[i].z), x[4]); x[5] = fmaf(wi, hi16<FP16>(cur[i].z), x[5]);
            x[6] = fmaf(wi, lo16<FP16>(cur[i].w), x[6]); x[7] = fmaf(wi, hi16<FP16>(cur[i].w), x[7]);
          }
        }
#pragma unroll
        for (int st = 0; st < 3; ++st) {
          const int off = 4 << st, half_n = 4 >> st;
          const bool up = (lane & off) != 0;
#pragma unroll
          for (int k = 0; k < half_n; ++k) {
            const float send = up ? x[k] : x[k + half_n];
            const float keep = up ? x[k + half_n] : x[k];
            x[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
          }
        }
        if (n < n_titles && (lane & 3) < np) p.pooled[(long long)n_out * F + c0 + (lane & 3) * 8 + jfeat] = x[0];
      }
    }
    }
  }
  __syncthreads();
  cluster_sync_all();     // no CTA leaves while the pair's MMAs / remote arrives may still target it
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}


// =====================================================================================================
// Conv1D weight gradient on tcgen05:  dW[(j,e), f] = sum_m X[m+j-1, e] * dPre[m, f]
//   (backward of keras Conv1D, task/paper.py:146; X = dropout(Embedding(tok)), dPre from attn bwd)
// GEMM view: M = 3*Ep rows (j,e) in 128-row slices, N = F, K = token slot rows.
// Both operands are "MN-major" (the reduction index = token is the slow index of the row-major data):
//   A[K=token][M=e] : gathered embedding rows — the same 128B-swizzled row image as in the forward, but
//                     described to the tensor core as MN-major (64-element groups, LBO between groups).
//   B[K=token][N=f] : dPre, written by the attention-backward kernel directly as pre-swizzled K-block
//                     images, fetched with one bulk copy each.
// CTA pairs (cta_group::2, M = 256): two adjacent slices share one dPre stream.  Each CTA stages its own A
// slice and only ITS HALF of dPre's columns (f in [rank*F/2, (rank+1)*F/2)), so the shared-memory traffic per
// SM (TMA writes + tensor-core operand reads, the limiter of the single-CTA version: 36 KB written + 34 KB read per
// 400-cycle K block) halves for B; the pair's MMA reads both halves.  Accumulator column c maps to
//   f = half*Fh + (c % n0h)            for c <  2*n0h   (half = c / n0h,  first MMA,  n0h = min(Fh,128))
//   f = half*Fh + n0h + (c' % n1h)     for c' = c-2*n0h (half = c'/ n1h,  second MMA, n1h = Fh - n0h).
// The peer CTA's producer warps arrive directly on the leader's stage-full barrier (remote mbarrier arrive; one of them
// first waits for the peer's own bulk copy); stage-empty and accumulator-full events come back to both CTAs through
// the multicast commit.
// The token range is split over CTA.y; partial sums go to global and are reduced in a fixed order.
// tokens (K rows) per title slot: template parameter KT = 32 (L <= 31) or 64 (L <= 63)
constexpr int WG_ES = 40;                           // embedding columns per (tap, e) slice: a slice's 128 M rows are the
                                                    // three taps of the SAME 40 columns (3 x 40 = 120 rows used), so a token's
                                                    // 16-byte pieces are gathered once and stored at the three tap shifts
constexpr int WG_STAGE_ROWS = 64;                   // K rows per pipeline stage: two 32-row titles or one 64-row title
                                                    // (amortises the per-stage handshake, ~500 cycles of issue-thread +
                                                    // commit latency, over 800 MMA cycles)
constexpr int WG_STAGES = 4;
constexpr int WG_THREADS = 640;   // 4 control warps + 16 producer warps (8 per title of a stage; warps 8-11 also run the epilogue)

struct WgradParams {
  int n_titles, L, F, EC, Ep, V;
  int n_kblocks, kb_per_split, n_slices, ngh;    // ngh = 64-column groups per F half; kb_per_split % WG_TPS == 0
  const int* tok;
  const uint16_t* emb;        // (V, Ep)
  const uint16_t* dpre_img;   // n_kblocks * 2 * ngh * 4 KB
  float* partial;             // [splits][n_slices*128][F]
  uint32_t drop_thr16, drop_addend, seed_x;   // quad-stream threshold (0 = no dropout) and its mask addend
  float scale;
  long long* trace;           // optional: accumulated wait cycles of CTA (0,0)'s roles (tools/perf_conv.py)
  const uint8_t* xmask;       // optional keep bits written by the forward (FwdParams::xmask); null: replay the hash
  const int* n_dev;           // optional device count of titles (K blocks) to process (<= n_kblocks): compacted title list
};

template <bool FP16, int KT>
__global__ void __launch_bounds__(WG_THREADS, 1) conv_wgrad_tc_kernel(const WgradParams p) {
  constexpr int WG_KTOK = KT;
  constexpr int WG_GROUP_BYTES = WG_KTOK * 128;       // one 64-element group of one title: 4 / 8 KB
  constexpr int WG_A_TILE_BYTES = 2 * WG_GROUP_BYTES; // A of one title: two 64-column chunks
  constexpr int WG_TPS = WG_STAGE_ROWS / KT;          // titles per pipeline stage
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int F = p.F, Fh = F >> 1;
  const int n0h = Fh > 128 ? 128 : Fh, n1h = Fh - n0h;
  const uint32_t b_tile_bytes = (uint32_t)p.ngh * WG_GROUP_BYTES;          // this CTA's half of one title's dPre
  const uint32_t a_stage_bytes = WG_TPS * WG_A_TILE_BYTES, b_stage_bytes = WG_TPS * b_tile_bytes;
  const uint32_t a_base = smem_base;
  const uint32_t b_base = a_base + WG_STAGES * a_stage_bytes;
  const uint32_t misc_base = b_base + WG_STAGES * b_stage_bytes;
  uint8_t* misc_gen = smem_gen + (misc_base - smem_base);
  const uint32_t bar_full = misc_base, bar_empty = misc_base + 64, bar_t_full = misc_base + 128;
  uint32_t* tmem_ptr_smem = (uint32_t*)(misc_gen + 144);
  uint4* mask_lut = reinterpret_cast<uint4*>(misc_gen + 256);    // keep byte -> four 16x2 AND masks (4 KB)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slice = blockIdx.x, split = blockIdx.y;
  const uint32_t crank = cluster_ctarank();     // 0 = leader (issues the pair's MMAs)
  int n_kblocks = p.n_kblocks, kb_per_split = p.kb_per_split;
  if (p.n_dev) {             // live titles only: the same even split of the (device-side) count over the token splits
    n_kblocks = min(__ldg(p.n_dev), p.n_kblocks);
    kb_per_split = ((n_kblocks + (int)gridDim.y - 1) / (int)gridDim.y + WG_TPS - 1) / WG_TPS * WG_TPS;
  }
  const int kb_beg = split * kb_per_split;
  const int kb_end = min(n_kblocks, kb_beg + kb_per_split);
  const int n_stage_blocks = kb_end > kb_beg ? (kb_end - kb_beg + WG_TPS - 1) / WG_TPS : 0;
  const bool tracing = p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < WG_STAGES; ++s) {
      // leader: its 16 producer warps + its B loader's expect_tx arrival + the 16 producer warps of the peer (remote
      // arrives; the peer's warp 4 first waits for the peer's own bulk copies).  peer: only its B loader's expect_tx.
      mbar_init(bar_full + 8 * s, crank == 0 ? 33 : 1);
      mbar_init(bar_empty + 8 * s, 1);   // multicast tcgen05.commit of the leader
    }
    mbar_init(bar_t_full, 1);
    fence_barrier_init();
  }
  for (uint32_t i = threadIdx.x; i < WG_STAGES * a_stage_bytes / 16; i += WG_THREADS)   // M rows never written stay zero
    reinterpret_cast<uint4*>(smem_gen)[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  if (p.xmask && threadIdx.x < 256) {
    const uint32_t b = threadIdx.x;
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = ((b >> j) & 1u ? 0x0000ffffu : 0u) | ((b >> (4 + j)) & 1u ? 0xffff0000u : 0u);
    mask_lut[b] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // both CTAs' barriers and tensor memory exist before any remote arrive / pair MMA
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {   // B loader: this CTA's half of the dPre columns of the WG_TPS titles of every stage
      int s = 0;
      uint32_t ph = 0;
      long long twl = 0;
      for (int sb = 0; sb < n_stage_blocks; ++sb) {
        long long t0 = tracing ? clock64() : 0;
        mbar_wait(bar_empty + 8 * s, ph ^ 1, 11);
        if (tracing) { twl += clock64() - t0; p.trace[5] = twl; }
        mbar_expect_tx(bar_full + 8 * s, b_stage_bytes);
#pragma unroll
        for (int t = 0; t < WG_TPS; ++t) {
          // a title past the end re-reads the last valid block: finite values, multiplied by the zero A rows
          const int kb = max(0, min(kb_beg + sb * WG_TPS + t, n_kblocks - 1));
          const uint8_t* src = (const uint8_t*)p.dpre_img + ((size_t)kb * 2 + crank) * b_tile_bytes;
          bulk_g2s(b_base + s * b_stage_bytes + t * b_tile_bytes, src, b_tile_bytes, bar_full + 8 * s);
        }
        if (++s == WG_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (crank == 0) {   // MMA issuer of the pair: the whole warp runs the loop, one elected lane issues
      const bool leader = elect_one();
      const uint32_t idesc0 = make_idesc_mn(2 * TILE_M, 2 * n0h, FP16), idesc1 = make_idesc_mn(2 * TILE_M, n1h > 0 ? 2 * n1h : 16, FP16);
      const uint32_t b1_off = (uint32_t)(n0h / 64) * WG_GROUP_BYTES;
      int s = 0;
      uint32_t ph = 0, accum = 0;
      long long tw = 0, t_start = tracing ? clock64() : 0;
      for (int sb = 0; sb < n_stage_blocks; ++sb) {
        long long t0 = tracing ? clock64() : 0;
        mbar_wait(bar_full + 8 * s, ph, 12);
        if (tracing) tw += clock64() - t0;
        tc_fence_after();
        if (leader) {
#pragma unroll
          for (int t = 0; t < WG_TPS; ++t) {
            const uint32_t a_addr = a_base + s * a_stage_bytes + t * WG_A_TILE_BYTES;
            const uint32_t b_addr = b_base + s * b_stage_bytes + t * b_tile_bytes;
#pragma unroll
            for (int kk = 0; kk < WG_KTOK / 16; ++kk) {
              const uint64_t ad = make_desc_mn128(a_addr + kk * 2048, WG_GROUP_BYTES);
              umma_f16_2cta(tmem_base, ad, make_desc_mn128(b_addr + kk * 2048, WG_GROUP_BYTES), idesc0, accum);
              if (n1h > 0)
                umma_f16_2cta(tmem_base + 2 * n0h, ad, make_desc_mn128(b_addr + b1_off + kk * 2048, WG_GROUP_BYTES), idesc1, accum);
              accum = 1;
            }
          }
          umma_commit_2cta(bar_empty + 8 * s, 3);
        }
        __syncwarp();
        if (++s == WG_STAGES) { s = 0; ph ^= 1; }
      }
      if (leader) umma_commit_2cta(bar_t_full, 3);
      __syncwarp();
      if (tracing && lane == 0) { p.trace[0] = tw; p.trace[1] = clock64() - t_start; p.trace[2] = n_stage_blocks; }
    }
  }
  if (warp >= 4) {
    // A producers (16 warps: 8 per title of a stage; warps 8-11 run the epilogue afterwards).  A producer warp's
    // instruction stream is latency-bound (few independent instructions between the gather, the dropout mask and the
    // shared-memory store), so the stage's work is spread over twice the warps rather than 4 pieces per thread: per
    // stage a thread handles (row r, 16-byte piece q) of both 64-column chunks (u0,u1) of this CTA's (tap, e) slice
    // for ONE of the stage's titles.  Dropout: keep bytes left by the forward, or a replay of its stream.
    const int pt = threadIdx.x - 128;          // 0..511
    const int tsel = pt / (KT * 8);            // title of the stage
    const int r = (pt % (KT * 8)) >> 3, q = pt & 7; // token row, 16-byte piece of the slice's 40 columns (q < 5)
    const int e0 = slice * WG_ES + q * 8;      // first embedding column of the piece
    const bool piece_ok = q < WG_ES / 8 && e0 < p.Ep;
    // The token id is NOT inspected when it is loaded (that would stall the warp for the load's full latency every
    // stage); validity is kept in the row index and the id is clamped when its embedding row is requested.
    constexpr int kNoTitle = INT_MIN;
    const bool use_mask = p.xmask != nullptr && p.drop_thr16 != 0;
    auto load_id = [&](int kb) { return (piece_ok && kb < kb_end && r < p.L) ? __ldg(p.tok + (long long)kb * p.L + r) : kNoTitle; };
    auto load_row = [&](int id) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (id != kNoTitle) {
        id = (id < 0 || id >= p.V) ? 0 : id;
        v = __ldg((const uint4*)(p.emb + (long long)id * p.Ep + e0));
      }
      return v;
    };
    // keep byte of the piece of title kb (row r): requested with the row, applied when the stage is stored
    auto load_mask = [&](int kb) {
      uint32_t m = 0xffu;
      if (use_mask && piece_ok && kb < kb_end && r < p.L) m = __ldg(p.xmask + ((long long)kb * p.L + r) * (p.Ep >> 3) + (e0 >> 3));
      return m;
    };
    int s = 0;
    uint32_t ph = 0;
    long long twait = 0, t_start = tracing ? clock64() : 0;
    // Gather pipeline: the row of stage sb+2 and the token id of stage sb+3 are requested while stage sb is masked
    // and stored (the gather's L2/HBM latency under load is about one stage period).
    uint4 vq[3];              // vq[sb % 3]: this thread's piece of its title of stage sb
    uint32_t mq[3];           // its keep byte
    int idn;                  // token id of the title of stage sb+2 while stage sb is stored
    vq[0] = load_row(load_id(kb_beg + tsel)); mq[0] = load_mask(kb_beg + tsel);
    vq[1] = load_row(load_id(kb_beg + WG_TPS + tsel)); mq[1] = load_mask(kb_beg + WG_TPS + tsel);
    idn = load_id(kb_beg + 2 * WG_TPS + tsel);
    auto drop_piece = [&](int kb, uint4& v) {      // replay of the forward's dropout stream (no keep bytes given)
      const uint64_t rowquad = (((uint64_t)kb * p.L + r) * (uint64_t)p.Ep) >> 2;   // Ep % 4 == 0
      const uint32_t base_lo = (uint32_t)rowquad, hi = (uint32_t)(rowquad >> 32);
      const uint32_t inner0 = quad_key(hi, p.seed_x);
      const uint32_t inner1 = base_lo > 0xfffff000u ? quad_key(hi + 1u, p.seed_x) : inner0;   // carry into the high word
      const uint32_t lo0 = base_lo + (uint32_t)(e0 >> 2);
      uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
      for (int x = 0; x < 2; ++x) {     // two quads per 16-byte piece
        const uint32_t lo = lo0 + x;
        uint32_t u0, u1;
        quad_hash(lo ^ (lo < base_lo ? inner1 : inner0), u0, u1);
        w[2 * x] &= quad_mask(u0, p.drop_addend);
        w[2 * x + 1] &= quad_mask(u1, p.drop_addend);
      }
    };
    long long tseg[4] = {0, 0, 0, 0};
    auto stage_step = [&](int sb, uint4& cur, uint4& nxt, uint32_t mcur, uint32_t& mnxt) {
      const int kb0 = kb_beg + sb * WG_TPS;
      long long tA = tracing ? clock64() : 0;
      nxt = load_row(idn);                                // stage sb+2
      mnxt = load_mask(kb0 + 2 * WG_TPS + tsel);
      idn = load_id(kb0 + 3 * WG_TPS + tsel);             // stage sb+3
      if (use_mask) {
        const uint4 lm = mask_lut[mcur];
        cur.x &= lm.x; cur.y &= lm.y; cur.z &= lm.z; cur.w &= lm.w;
      } else if (p.drop_thr16 && piece_ok) {
        drop_piece(kb0 + tsel, cur);
      }
      long long t0 = tracing ? clock64() : 0;
      if (tracing) tseg[0] += t0 - tA;
      if (lane == 0) mbar_wait(bar_empty + 8 * s, ph ^ 1, 13);   // one poller per warp
      __syncwarp();
      if (tracing) twait += clock64() - t0;
      long long tB = tracing ? clock64() : 0;
      if (piece_ok) {
        const uint32_t tile = a_base + s * a_stage_bytes + tsel * WG_A_TILE_BYTES;
#pragma unroll
        for (int j = 0; j < TAPS; ++j) {     // M row of (tap j, column e0 + i) = j * 40 + (e0 - slice * 40) + i
          const int m0 = j * WG_ES + q * 8;
          const int rr = (r + 1 - j) & (WG_KTOK - 1);
          const uint32_t addr = tile + (m0 >> 6) * WG_GROUP_BYTES + rr * 128 + ((((m0 & 63) >> 3) ^ (rr & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(cur.x), "r"(cur.y), "r"(cur.z), "r"(cur.w) : "memory");
        }
      }
      long long tC = tracing ? clock64() : 0;
      if (tracing) tseg[1] += tC - tB;
      fence_proxy_async();
      if (tracing) tseg[2] += clock64() - tC;
      long long tD = tracing ? clock64() : 0;
      __syncwarp();
      if (lane == 0) {
        if (crank == 0) {
          mbar_arrive(bar_full + 8 * s);
        } else {
          if (warp == 4) mbar_wait(bar_full + 8 * s, ph, 16);   // this CTA's halves of dPre have landed
          mbar_arrive_remote(map_to_cta(bar_full + 8 * s, 0));
        }
      }
      if (tracing) tseg[3] += clock64() - tD;
      if (++s == WG_STAGES) { s = 0; ph ^= 1; }
    };
    for (int sb = 0; sb < n_stage_blocks; sb += 3) {
      stage_step(sb, vq[0], vq[2], mq[0], mq[2]);
      if (sb + 1 < n_stage_blocks) stage_step(sb + 1, vq[1], vq[0], mq[1], mq[0]);
      if (sb + 2 < n_stage_blocks) stage_step(sb + 2, vq[2], vq[1], mq[2], mq[1]);
    }
    if (tracing && pt == 0) {
      p.trace[3] = twait; p.trace[4] = clock64() - t_start;
      p.trace[6] = tseg[0]; p.trace[7] = tseg[1]; p.trace[8] = tseg[2]; p.trace[9] = tseg[3];
    }
  }
  if (warp >= 8 && warp < 12) {
    // epilogue (once): TMEM -> scaled fp32 partial sums in global memory; accumulator columns are mapped back to f
    const int q = warp & 3;
    mbar_wait(bar_t_full, 0, 14);
    tc_fence_after();
    const int row = q * 32 + lane;
    float* dst = p.partial + ((size_t)split * p.n_slices * TILE_M + (size_t)slice * TILE_M + row) * F;
    const bool any = n_stage_blocks > 0;
    for (int seg = 0; seg < 4; ++seg) {
      const int nseg = seg < 2 ? n0h : n1h;
      const int c_beg = seg < 2 ? seg * n0h : 2 * n0h + (seg - 2) * n1h;
      const int f_beg = (seg & 1) * Fh + (seg < 2 ? 0 : n0h);
      for (int c = 0; c < nseg; c += 8) {
        uint32_t rv[8];
        TMEM_LD_8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c_beg + c), rv);
        tmem_ld_wait();
        float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi4 = lo;
        if (any) {
          lo = make_float4(__uint_as_float(rv[0]) * p.scale, __uint_as_float(rv[1]) * p.scale, __uint_as_float(rv[2]) * p.scale,
                           __uint_as_float(rv[3]) * p.scale);
          hi4 = make_float4(__uint_as_float(rv[4]) * p.scale, __uint_as_float(rv[5]) * p.scale, __uint_as_float(rv[6]) * p.scale,
                            __uint_as_float(rv[7]) * p.scale);
        }
        *reinterpret_cast<float4*>(dst + f_beg + c) = lo;
        *reinterpret_cast<float4*>(dst + f_beg + c + 4) = hi4;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  cluster_sync_all();     // no CTA leaves while the pair's MMAs / remote arrives may still target it
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// d_conv_w[j][e][f] = sum_split partial[split][(e / 40) * 128 + j * 40 + e % 40][f]   (fixed order, deterministic)
__global__ void wgrad_reduce_kernel(int E, int Ep, int F, int splits, int rows_total, const float* __restrict__ partial,
                                    float* __restrict__ dW) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)TAPS * E * F) return;
  int f = (int)(i % F);
  int je = (int)(i / F);
  int j = je / E, e = je % E;
  long long row = (long long)(e / WG_ES) * TILE_M + j * WG_ES + e % WG_ES;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += partial[((long long)s * rows_total + row) * F + f];
  dW[i] = acc;
}

}  // namespace tc
}  // namespace lstur

// ======================================================================== host side
using namespace lstur;

// Padded embedding width (multiple of the 64-element K block).
extern "C" int lstur_tc_padded_e(int E) { return (E + tc::EPAD - 1) / tc::EPAD * tc::EPAD; }
// Elements (bf16) of the packed conv-weight image.
extern "C" long long lstur_tc_wimg_elems(int E, int F) {
  return (long long)(lstur_tc_padded_e(E) / tc::KBLK) * tc::TAPS * F * tc::KBLK;
}

// keras Embedding weights (task/paper.py:132-138) -> bf16 (V, Ep) table used by the tensor-core gather.
extern "C" int lstur_pack_word_emb_16(long long V, int E, const float* word_emb, void* emb_bf16, int fp16,
                                      cudaStream_t stream) {
  LSTUR_REQUIRE(V > 0 && E > 0, "lstur_pack_word_emb_16");
  int Ep = lstur_tc_padded_e(E);
  long long n = V * (Ep / 8);
  tc::pack_emb_bf16_kernel<<<cdiv(n, 256), 256, 0, stream>>>(V, E, Ep, word_emb, (uint16_t*)emb_bf16, fp16 != 0);
  LSTUR_CHECK_LAUNCH("lstur_pack_word_emb_16");
  return LSTUR_OK;
}

// Conv1D kernel (3,E,F) (task/paper.py:146) -> swizzled bf16 K-block images.
extern "C" int lstur_pack_conv_w_tc(int E, int F, const float* conv_w, void* wimg, int fp16, cudaStream_t stream) {
  LSTUR_REQUIRE(E > 0 && F > 0, "lstur_pack_conv_w_tc");
  long long n = lstur_tc_wimg_elems(E, F);
  tc::pack_conv_w_kernel<<<cdiv(n, 256), 256, 0, stream>>>(E, F, lstur_tc_padded_e(E) / tc::KBLK, conv_w,
                                                           (uint16_t*)wimg, fp16 != 0);
  LSTUR_CHECK_LAUNCH("lstur_pack_conv_w_tc");
  return LSTUR_OK;
}

size_t tc_conv_smem_bytes(int EC, int F, int nstages);
extern "C" int lstur_tc_supported(int L, int E, int F, int KS) {
  if (!(KS == 3 && L >= 1 && L <= 63 && E >= 1 && F >= 16 && F % 16 == 0 && F <= tc::TMEM_COLS)) return 0;
  // the tile's K chunks stay resident in shared memory next to >= 2 weight stages
  const int EC = lstur_tc_padded_e(E) / tc::KBLK;
  return EC <= tc::MAX_CHUNKS && tc_conv_smem_bytes(EC, F, 2) <= 232448;
}
// rows of a title slot: the L tokens + at least one zero row (the conv halo), 32 or 64
extern "C" int lstur_tc_slot(int L) { return L <= 31 ? 32 : 64; }

static void* g_tc_trace_ptr = nullptr;
// Debug/profiling hook: device buffer of 8*16 int64 receiving clock64() stamps of CTA 0's warp roles (NULL = off).
extern "C" int lstur_tc_set_trace(void* dev_buf) { g_tc_trace_ptr = dev_buf; return LSTUR_OK; }

// Fused news-encoder forward (k1-k6): tokens (n_titles,L) -> C (bf16, saved), pooled (n_titles,F), att a / w.
// bytes of the X-dropout keep-bit buffer the forward can leave for the weight-gradient kernel (one byte per 16-byte piece)
extern "C" size_t lstur_tc_xmask_bytes(int n_titles, int L, int E) {
  return (size_t)n_titles * L * (lstur_tc_padded_e(E) / 8);
}

// Launch news_conv_tc_kernel<FP16, DROP, SLOT, MODE> on CTA pairs: persistent, one pair per two 128-row token tiles.
template <bool FP16, bool DROP, int SLOT, int MODE>
static cudaError_t tc_launch_one(const tc::FwdParams& p, size_t smem, int pairs, cudaStream_t stream) {
  static size_t attr_smem = 0;
  auto kern = tc::news_conv_tc_kernel<FP16, DROP, SLOT, MODE>;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_smem = smem;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(tc::THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, p);
}

// dynamic shared memory of news_conv_tc_kernel: alignment slack + A ring + B ring + barriers / epilogue scratch
constexpr size_t TC_SMEM_LIMIT = 232448;      // 227 KB opt-in maximum per CTA on sm_100
size_t tc_conv_smem_bytes(int EC, int F, int nstages) {
  return 1024 + (size_t)EC * tc::A_STAGE_BYTES + (size_t)nstages * tc::TAPS * tc::conv_n0h(F / 2) * tc::ROWB + 1024 + 4096 +
         (((size_t)2 * F * sizeof(float) + 15) & ~(size_t)15) + (size_t)8 * tc::STG_WARP_BYTES;
}

static int tc_launch_conv(const tc::FwdParams& p, int L, bool fp16, bool drop, int mode, int max_ctas, cudaStream_t stream,
                          const char* name) {
  const int F = p.F, slot = lstur_tc_slot(L);
  int nst = tc::DEF_STAGES;
  while (nst > 2 && tc_conv_smem_bytes(p.EC, F, nst) > TC_SMEM_LIMIT) --nst;
  if (p.EC > tc::MAX_CHUNKS || tc_conv_smem_bytes(p.EC, F, nst) > TC_SMEM_LIMIT) {
    set_error("%s: K = %d chunks x N = %d does not fit the shared-memory plan of the tensor-core conv kernel", name, p.EC, F);
    return LSTUR_ERR_UNSUPPORTED;
  }
  const_cast<tc::FwdParams&>(p).nstages = nst;
  size_t smem = tc_conv_smem_bytes(p.EC, F, nst);
  int n_tiles = (p.n_titles + (tc::TILE_M / slot) - 1) / (tc::TILE_M / slot);
  int n_tp = (n_tiles + 1) / 2;             // CTA pairs take two token tiles at a time
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  int pairs = n_tp < sms / 2 ? n_tp : sms / 2;
  if (max_ctas > 0 && pairs > max_ctas / 2) pairs = max_ctas / 2 > 0 ? max_ctas / 2 : 1;
  cudaError_t e;
#define TC_DISPATCH_SLOT(FP16_, DROP_, MODE_)                                                        \
  (slot == 32 ? tc_launch_one<FP16_, DROP_, 32, MODE_>(p, smem, pairs, stream)                      \
              : tc_launch_one<FP16_, DROP_, 64, MODE_>(p, smem, pairs, stream))
  if (mode == tc::MODE_DGRAD) e = fp16 ? TC_DISPATCH_SLOT(true, false, tc::MODE_DGRAD) : TC_DISPATCH_SLOT(false, false, tc::MODE_DGRAD);
  else if (fp16 && drop) e = TC_DISPATCH_SLOT(true, true, tc::MODE_FWD);
  else if (fp16) e = TC_DISPATCH_SLOT(true, false, tc::MODE_FWD);
  else if (drop) e = TC_DISPATCH_SLOT(false, true, tc::MODE_FWD);
  else e = TC_DISPATCH_SLOT(false, false, tc::MODE_FWD);
#undef TC_DISPATCH_SLOT
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", name, cudaGetErrorString(e));
    return LSTUR_ERR_CUDA;
  }
  LSTUR_CHECK_LAUNCH(name);
  return LSTUR_OK;
}

extern "C" int lstur_news_conv_tc_fwd(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_bf16,
                                      const void* wimg, const float* conv_b, const float* att_w, const float* att_b,
                                      void* c_out_bf16, float* pooled, float* att_a, float* att_wt, float dropout,
                                      unsigned seed, int fp16, int max_ctas, cudaStream_t stream) {
  return lstur_news_conv_tc_fwd_m(n_titles, L, E, F, V, tokens, emb_bf16, wimg, conv_b, att_w, att_b, c_out_bf16, pooled,
                                  att_a, att_wt, dropout, seed, fp16, max_ctas, nullptr, nullptr, nullptr, stream);
}

extern "C" int lstur_news_conv_tc_fwd_m(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_bf16,
                                        const void* wimg, const float* conv_b, const float* att_w, const float* att_b,
                                        void* c_out_bf16, float* pooled, float* att_a, float* att_wt, float dropout,
                                        unsigned seed, int fp16, int max_ctas, void* xmask_out, const int* n_titles_dev,
                                        const int* title_idx, cudaStream_t stream) {
  LSTUR_REQUIRE(n_titles >= 0 && lstur_tc_supported(L, E, F, 3), "lstur_news_conv_tc_fwd");
  LSTUR_REQUIRE(dropout >= 0.f && dropout < 1.f && c_out_bf16 && pooled, "lstur_news_conv_tc_fwd");
  if (n_titles == 0) return LSTUR_OK;
  tc::FwdParams p{};
  p.n_titles = n_titles; p.L = L; p.F = F; p.Ep = lstur_tc_padded_e(E); p.EC = p.Ep / tc::KBLK; p.V = V;
  p.tok = tokens; p.emb = (const uint16_t*)emb_bf16; p.wimg = (const uint16_t*)wimg;
  p.conv_b = conv_b; p.att_w = att_w; p.att_b = att_b;
  p.c_out = (uint16_t*)c_out_bf16; p.pooled = pooled; p.att_a = att_a; p.att_wt = att_wt;
  p.drop_thr16 = dropout > 0.f ? quad_thr15(dropout) : 0u;
  p.drop_addend = quad_addend(p.drop_thr16);
  p.inv_keep = 1.f / (1.f - dropout);
  p.seed_x = seed * 2u; p.seed_c = seed * 2u + 1u;
  p.xmask = (uint8_t*)xmask_out;
  p.n_dev = n_titles_dev; p.title_idx = title_idx;
  p.trace = (long long*)g_tc_trace_ptr;
  return tc_launch_conv(p, L, fp16 != 0, p.drop_thr16 != 0, tc::MODE_FWD, max_ctas, stream, "lstur_news_conv_tc_fwd");
}

// ---- conv input gradient (word-table training: keras Embedding(trainable=True), task/paper.py:132-138) ----------
extern "C" int lstur_tc_wgrad_groups(int F);
// 32-column K chunks per half of the conv features in the dPre image
static int dgrad_cph(int F) { return (F / 2 + tc::KBLK - 1) / tc::KBLK; }
extern "C" long long lstur_tc_wimg_dgrad_elems(int E, int F) {
  return (long long)2 * dgrad_cph(F) * tc::TAPS * lstur_tc_padded_e(E) * tc::KBLK;
}
extern "C" int lstur_pack_conv_w_dgrad_tc(int E, int F, const float* conv_w, void* wimg_d, int fp16, cudaStream_t stream) {
  LSTUR_REQUIRE(E > 0 && F > 0 && F % 16 == 0 && conv_w && wimg_d, "lstur_pack_conv_w_dgrad_tc");
  long long n = lstur_tc_wimg_dgrad_elems(E, F);
  tc::pack_conv_w_dgrad_kernel<<<cdiv(n, 256), 256, 0, stream>>>(E, F, lstur_tc_padded_e(E), dgrad_cph(F), conv_w,
                                                                 (uint16_t*)wimg_d, fp16 != 0);
  LSTUR_CHECK_LAUNCH("lstur_pack_conv_w_dgrad_tc");
  return LSTUR_OK;
}
// dx16 (n_titles, L, Ep) 16-bit rows = out_scale * dX, dX[m, e] = sum_j sum_f dPre[m+1-j, f] Wc[j, e, f] (columns
// e >= E are zero); dpre_img is the image written by lstur_attn_pool_bwd_img (whose own scale multiplies through).
extern "C" int lstur_conv_dgrad_tc(int n_titles, int L, int E, int F, const void* dpre_img, const void* wimg_d, void* dx16,
                                   float out_scale, int fp16, int max_ctas, const int* n_titles_dev, cudaStream_t stream) {
  LSTUR_REQUIRE(n_titles >= 0 && lstur_tc_supported(L, E, F, 3) && dpre_img && wimg_d && dx16, "lstur_conv_dgrad_tc");
  const int Eo = lstur_tc_padded_e(E);
  LSTUR_REQUIRE(Eo <= tc::TMEM_COLS && (Eo <= 256 || Eo - 256 >= 16), "lstur_conv_dgrad_tc(E too wide for one accumulator)");
  if (n_titles == 0) return LSTUR_OK;
  tc::FwdParams p{};
  p.n_titles = n_titles; p.L = L; p.F = Eo; p.Ep = Eo; p.V = 0;
  p.cph = dgrad_cph(F); p.ngh = lstur_tc_wgrad_groups(F); p.EC = 2 * p.cph;
  p.dimg = (const uint8_t*)dpre_img; p.wimg = (const uint16_t*)wimg_d; p.c_out = (uint16_t*)dx16;
  p.out_scale = out_scale;
  p.n_dev = n_titles_dev;
  p.inv_keep = 1.f;
  p.trace = nullptr;
  return tc_launch_conv(p, L, fp16 != 0, false, tc::MODE_DGRAD, max_ctas, stream, "lstur_conv_dgrad_tc");
}

// ---- wgrad host side ------------------------------------------------------------------------------
extern "C" int lstur_tc_wgrad_kblocks(int n_titles) { return n_titles; }   // one 32-row slot = one K block
// 64-column groups per half of the F columns (each CTA of a pair stages one half)
extern "C" int lstur_tc_wgrad_groups(int F) { return (F / 2 + 63) / 64; }
// bytes of the dPre image consumed by lstur_conv_wgrad_tc: per title [half][group][32 rows][128 B]
extern "C" size_t lstur_tc_dpre_img_bytes(int n_titles, int L, int F) {
  return (size_t)lstur_tc_wgrad_kblocks(n_titles) * 2 * lstur_tc_wgrad_groups(F) * lstur_tc_slot(L) * 128;
}
static int wgrad_slices(int E) {
  int n = (lstur_tc_padded_e(E) + tc::WG_ES - 1) / tc::WG_ES;     // 40 embedding columns x 3 taps per 128-row slice
  return (n + 1) & ~1;   // CTA pairs
}
extern "C" int lstur_tc_wgrad_splits(int n_titles, int E) {
  int n_slices = wgrad_slices(E);
  int kb = lstur_tc_wgrad_kblocks(n_titles);
  int sms = 148;
  int splits = sms / n_slices;
  if (splits < 1) splits = 1;
  if (splits > kb) splits = kb;
  return splits;
}
extern "C" size_t lstur_tc_wgrad_partial_bytes(int n_titles, int E, int F) {
  return (size_t)lstur_tc_wgrad_splits(n_titles, E) * wgrad_slices(E) * tc::TILE_M * F * sizeof(float);
}

// d_conv_w (3,E,F) = sum over tokens of X[m+j-1,e] * dPre[m,f]; X re-gathered from emb_16 with the forward's dropout
// stream (seed), dPre given as the K-block image written by lstur_attn_pool_bwd_img.
extern "C" int lstur_conv_wgrad_tc(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                                   const void* dpre_img, float* d_conv_w, float dropout, unsigned seed, int fp16,
                                   void* partial_ws, size_t partial_bytes, cudaStream_t stream) {
  return lstur_conv_wgrad_tc_m(n_titles, L, E, F, V, tokens, emb_16, dpre_img, d_conv_w, dropout, seed, fp16, partial_ws,
                               partial_bytes, nullptr, 1.f, nullptr, stream);
}

extern "C" int lstur_conv_wgrad_tc_m(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                                     const void* dpre_img, float* d_conv_w, float dropout, unsigned seed, int fp16,
                                     void* partial_ws, size_t partial_bytes, const void* xmask, float dpre_scale,
                                     const int* n_titles_dev, cudaStream_t stream) {
  LSTUR_REQUIRE(n_titles >= 0 && lstur_tc_supported(L, E, F, 3) && dpre_scale > 0.f, "lstur_conv_wgrad_tc");
  if (n_titles == 0) {
    cudaMemsetAsync(d_conv_w, 0, (size_t)3 * E * F * sizeof(float), stream);
    return LSTUR_OK;
  }
  tc::WgradParams p;
  p.n_titles = n_titles; p.L = L; p.F = F; p.Ep = lstur_tc_padded_e(E); p.EC = p.Ep / tc::EPAD; p.V = V;
  p.n_kblocks = lstur_tc_wgrad_kblocks(n_titles);
  p.n_slices = wgrad_slices(E);
  int splits = lstur_tc_wgrad_splits(n_titles, E);
  p.kb_per_split = (p.n_kblocks + splits - 1) / splits;
  const int kt = lstur_tc_slot(L), tps = tc::WG_STAGE_ROWS / kt;
  p.kb_per_split = (p.kb_per_split + tps - 1) / tps * tps;   // whole pipeline stages per split
  p.ngh = lstur_tc_wgrad_groups(F);
  p.tok = tokens; p.emb = (const uint16_t*)emb_16; p.dpre_img = (const uint16_t*)dpre_img;
  p.partial = (float*)partial_ws;
  LSTUR_REQUIRE(partial_ws != nullptr && partial_bytes >= lstur_tc_wgrad_partial_bytes(n_titles, E, F), "lstur_conv_wgrad_tc");
  p.drop_thr16 = dropout > 0.f ? quad_thr15(dropout) : 0u;
  p.drop_addend = quad_addend(p.drop_thr16);
  p.seed_x = seed * 2u;
  p.scale = 1.f / ((1.f - dropout) * dpre_scale);
  p.trace = (long long*)g_tc_trace_ptr;
  p.xmask = (const uint8_t*)xmask;
  p.n_dev = n_titles_dev;
  // a stage holds WG_STAGE_ROWS K rows whatever the slot height: A = 2 groups, B = ngh groups of 128-byte rows
  size_t smem = 1024 + (size_t)tc::WG_STAGES * tc::WG_STAGE_ROWS * 128 * (2 + (size_t)p.ngh) + 256 + 4096;
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(tc::conv_wgrad_tc_kernel<true, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::conv_wgrad_tc_kernel<false, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::conv_wgrad_tc_kernel<true, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::conv_wgrad_tc_kernel<false, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("lstur_conv_wgrad_tc: cannot opt in to %zu B of shared memory: %s", smem, cudaGetErrorString(e));
      return LSTUR_ERR_CUDA;
    }
    attr_smem = smem;
  }
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.n_slices, splits);
    cfg.blockDim = dim3(tc::WG_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;   // CTA pair = two adjacent slices of the same token split
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    if (kt == 32) e = fp16 ? cudaLaunchKernelEx(&cfg, tc::conv_wgrad_tc_kernel<true, 32>, p)
                           : cudaLaunchKernelEx(&cfg, tc::conv_wgrad_tc_kernel<false, 32>, p);
    else e = fp16 ? cudaLaunchKernelEx(&cfg, tc::conv_wgrad_tc_kernel<true, 64>, p)
                  : cudaLaunchKernelEx(&cfg, tc::conv_wgrad_tc_kernel<false, 64>, p);
    if (e != cudaSuccess) {
      set_error("lstur_conv_wgrad_tc: launch failed: %s", cudaGetErrorString(e));
      return LSTUR_ERR_CUDA;
    }
  }
  LSTUR_CHECK_LAUNCH("lstur_conv_wgrad_tc");
  long long n = (long long)3 * E * F;
  tc::wgrad_reduce_kernel<<<cdiv(n, 256), 256, 0, stream>>>(E, p.Ep, F, splits, p.n_slices * tc::TILE_M, p.partial, d_conv_w);
  LSTUR_CHECK_LAUNCH("lstur_conv_wgrad_tc(reduce)");
  return LSTUR_OK;
}
