// Pad-token mask + Masking + Dropout + additive-attention pooling, forward and backward.
//
// Reference: task/paper.py:150-158 (Lambda pad mask, Masking, Dropout) and
// models.SimpleAttentionMaskSupport.call models.py:474-489 (SURVEY.md §9.2-9.3):
//   C <- C*[tok!=0];  m = any_f(C != 0);  C <- dropout(C*m)
//   a = tanh(C.ka + ba);  e = exp(a)*m;  w = e/(sum_t e + 1e-7);  p = sum_t w_t C_t
// These are the un-fused (verification) kernels; the tensor-core conv kernel
// carries the same arithmetic in its epilogue.
#include <cuda_fp16.h>

#include "common.cuh"

namespace lstur {

constexpr int ATT_THREADS = 128;
constexpr int ATT_MAX_L = 256;

// One CTA per title.  C (in/out): conv+bias+relu on entry, attention input on exit.
__global__ void __launch_bounds__(ATT_THREADS)
attn_pool_fwd_kernel(int N, int L, int F, float* __restrict__ C, long long title_stride,
                     const int* __restrict__ tok, const float* __restrict__ ka, const float* __restrict__ ba,
                     float* __restrict__ p, long long ldp, float* __restrict__ a_out, float* __restrict__ w_out,
                     uint32_t drop_thr, float inv_keep, uint32_t seed) {
  __shared__ float sa[ATT_MAX_L], se[ATT_MAX_L];
  const int n = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* Cn = C + (long long)n * title_stride;
  const float bias = ba[0];
  for (int t = warp; t < L; t += ATT_THREADS / 32) {
    const int tk = tok[(long long)n * L + t];
    float dot = 0.f;
    int any = 0;
    const uint64_t base = ((uint64_t)n * L + t) * (uint64_t)F;
    for (int f = lane; f < F; f += 32) {
      float v = tk != 0 ? Cn[(long long)t * F + f] : 0.f;
      any |= (v != 0.f);
      if (drop_thr) v = (rng_u32(seed, base + f) >> 8) >= drop_thr ? v * inv_keep : 0.f;
      Cn[(long long)t * F + f] = v;
      dot = fmaf(v, ka[f], dot);
    }
    any = warp_or(any);
    dot = warp_sum(dot);
    if (lane == 0) {
      float a = tanhf(dot + bias);
      sa[t] = a;
      se[t] = any ? expf(a) : 0.f;
    }
  }
  __syncthreads();
  float S = 0.f;
  for (int t = 0; t < L; ++t) S += se[t];
  const float invS = 1.f / (S + 1e-7f);
  for (int t = tid; t < L; t += ATT_THREADS) {
    if (a_out) a_out[(long long)n * L + t] = sa[t];
    if (w_out) w_out[(long long)n * L + t] = se[t] * invS;
  }
  for (int f = tid; f < F; f += ATT_THREADS) {
    float acc = 0.f;
    for (int t = 0; t < L; ++t) acc = fmaf(se[t] * invS, Cn[(long long)t * F + f], acc);
    p[(long long)n * ldp + f] = acc;
  }
}

// Backward of the block above.  Grid-strided over titles; each CTA keeps
// per-thread partial sums of d(ka), d(conv bias) and d(ba) and writes them to
// partials[cta][2F+1] (reduced afterwards in a fixed order -> deterministic).
//   dPre = d(loss)/d(conv pre-activation) incl. ReLU/pad/Masking/Dropout gates, as fp32 rows (title stride
//   dpre_title_stride, rows L..Lrows-1 zeroed).
template <int FPT>
__global__ void __launch_bounds__(ATT_THREADS)
attn_pool_bwd_kernel(int N, int L, int Lrows, int F, const float* __restrict__ Cd, long long title_stride,
                     const float* __restrict__ a_in, const float* __restrict__ w_in, const float* __restrict__ dp,
                     long long lddp, const float* __restrict__ ka, float* __restrict__ dPre,
                     long long dpre_title_stride, float inv_keep, float* __restrict__ partials) {
  __shared__ float sdw[ATT_MAX_L], sdz[ATT_MAX_L], sw[ATT_MAX_L];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float dka[FPT], dbc[FPT], dba = 0.f;
#pragma unroll
  for (int i = 0; i < FPT; ++i) dka[i] = dbc[i] = 0.f;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    const float* Cn = Cd + (long long)n * title_stride;
    const float* dpn = dp + (long long)n * lddp;
    float* dPn = dPre + (long long)n * dpre_title_stride;
    for (int t = warp; t < L; t += ATT_THREADS / 32) {
      float dot = 0.f;
      for (int f = lane; f < F; f += 32) dot = fmaf(Cn[(long long)t * F + f], dpn[f], dot);
      dot = warp_sum(dot);
      if (lane == 0) {
        sdw[t] = dot;
        sw[t] = w_in[(long long)n * L + t];
      }
    }
    __syncthreads();
    float q = 0.f;
    for (int t = 0; t < L; ++t) q = fmaf(sdw[t], sw[t], q);
    for (int t = tid; t < L; t += ATT_THREADS) {
      float a = a_in[(long long)n * L + t];
      sdz[t] = (sdw[t] - q) * sw[t] * (1.f - a * a);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < FPT; ++i) {
      int f = tid + i * ATT_THREADS;
      if (f < F) {
        const float dpf = dpn[f], kaf = ka[f];
        for (int t = 0; t < L; ++t) {
          float c = Cn[(long long)t * F + f];
          float g = fmaf(sw[t], dpf, sdz[t] * kaf);
          float dpre = c > 0.f ? g * inv_keep : 0.f;
          dPn[(long long)t * F + f] = dpre;
          dka[i] = fmaf(sdz[t], c, dka[i]);
          dbc[i] += dpre;
        }
        for (int t = L; t < Lrows; ++t) dPn[(long long)t * F + f] = 0.f;
      }
    }
    if (tid == 0)
      for (int t = 0; t < L; ++t) dba += sdz[t];
    __syncthreads();
  }
  float* out = partials + (long long)blockIdx.x * (2 * F + 1);
#pragma unroll
  for (int i = 0; i < FPT; ++i) {
    int f = tid + i * ATT_THREADS;
    if (f < F) {
      out[f] = dka[i];
      out[F + f] = dbc[i];
    }
  }
  if (tid == 0) out[2 * F] = dba;
}

// out[c] (+)= sum_r in[r*ld + c], two fixed-order stages (deterministic).
__global__ void colsum_stage1_kernel(long long rows, int cols, const float* __restrict__ in, long long ld,
                                     int rows_per_chunk, float* __restrict__ partial) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  long long r0 = (long long)blockIdx.y * rows_per_chunk, r1 = min(rows, r0 + rows_per_chunk);
  // four independent partial sums (rows r0 + 4k + i), combined in a fixed order: the single dependent add chain made this
  // pass latency-bound (28 us for the 45 MB of d doc_vec)
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
    s0 += in[r * ld + c];
    s1 += in[(r + 1) * ld + c];
    s2 += in[(r + 2) * ld + c];
    s3 += in[(r + 3) * ld + c];
  }
  for (; r < r1; ++r) s0 += in[r * ld + c];
  partial[(long long)blockIdx.y * cols + c] = (s0 + s1) + (s2 + s3);
}
// 256 threads = 32 columns x 8 chunk strides, stride sums combined in ascending order (fixed order, deterministic)
__global__ void colsum_stage2_kernel(int chunks, int cols, const float* __restrict__ partial, float* __restrict__ out,
                                     int accumulate) {
  __shared__ float sm[8][32];
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < cols)
    for (int k = part; k < chunks; k += 8) s += partial[(long long)k * cols + c];
  sm[part][lane] = s;
  __syncthreads();
  if (part != 0 || c >= cols) return;
  float t = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) t += sm[q][lane];
  out[c] = accumulate ? out[c] + t : t;
}

// Tensor-core-mode backward (v2): the title's 16-bit C tile is staged once in shared memory with 16-byte loads,
// every thread owns one 8-column chunk (fixed columns -> private d att_w / d conv_b accumulators) and writes dPre
// as 16-byte pieces straight into the MN-major swizzled K-block image consumed by conv_wgrad_tc_kernel.
// HBM traffic = read C once + write dPre once.
template <typename CT>
__device__ __forceinline__ void unpack8(const uint4& u, float* v);
template <>
__device__ __forceinline__ void unpack8<__half>(const uint4& u, float* v) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
template <>
__device__ __forceinline__ void unpack8<__nv_bfloat16>(const uint4& u, float* v) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
template <typename CT>
__device__ __forceinline__ uint4 pack8(const float* v);
template <>
__device__ __forceinline__ uint4 pack8<__half>(const float* v) {
  uint4 u;
  __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {     // saturating conversion in one instruction per pair
    uint32_t w;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
    reinterpret_cast<uint32_t*>(&u)[i] = w;
  }
  (void)h;
  return u;
}
template <>
__device__ __forceinline__ uint4 pack8<__nv_bfloat16>(const float* v) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  return u;
}

constexpr int IMG_THREADS = 256;     // 64 chunk columns x 4 row groups
// SLOT = rows of a title slot of the image (32 for L <= 31, 64 for L <= 63).  The image holds one block per title slot n,
// [half h = f / (F/2)][64-column group][SLOT rows][128 B]; with fl = f - h*F/2 the 16-bit element lives at byte
//   n*2*ngh*SLOT*128 + (h*ngh + fl/64)*SLOT*128 + t*128 + ((((fl%64)/8) ^ (t%8)) << 4) + (fl%8)*2
// (MN-major SWIZZLE_128B, one half per CTA of the weight gradient's CTA pair; ngh = ceil(F/2/64)).
// img_scale: power-of-two loss scale of the 16-bit dPre values (gradients of a mean over a large global batch would
// otherwise sit in fp16's subnormal range); the consumers (conv weight / input gradient) divide it out, and the d conv_b
// partial sums are unscaled on the way out.
template <typename CT, int SLOT>
__global__ void __launch_bounds__(IMG_THREADS)
attn_bwd_img_kernel(int N, int L, int F, const CT* __restrict__ Cd, const float* __restrict__ a_in,
                    const float* __restrict__ w_in, const float* __restrict__ dp, long long lddp,
                    const float* __restrict__ ka, uint8_t* __restrict__ img, float inv_keep, float img_scale,
                    float* __restrict__ partials, const int* __restrict__ n_dev,
                    const int* __restrict__ title_idx) {
  if (n_dev) N = min(N, __ldg(n_dev));          // compacted title list: live titles only (lstur_compact_titles)
  extern __shared__ __align__(16) uint8_t att_smem[];
  const int nchunk = F >> 3;                       // 16-byte chunks per row
  // Two title buffers: the (contiguous, L*F*2-byte) saved C of the NEXT title is fetched with one bulk copy while the
  // current one is processed; its d_pooled row and attention weights are prefetched into registers.
  const size_t buf_bytes = (size_t)SLOT * nchunk * 16;
  float* sdp = reinterpret_cast<float*>(att_smem + 2 * buf_bytes);   // [F]
  float* ska = sdp + F;                                           // [F]
  float* sred = reinterpret_cast<float*>(att_smem);                  // [3][64][16] reduction scratch, after the title loop
  __shared__ float sdw[SLOT], sdz[SLOT], sw[SLOT];
  __shared__ __align__(8) unsigned long long s_bar[2];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c = tid & 63, tg = tid >> 6;           // chunk owned by this thread, row group (0..3)
  const bool c_ok = c < nchunk;
  const int Fh = F >> 1, ngh = (Fh + 63) >> 6;     // image: [half][group][SLOT rows][128 B] per title
  constexpr int GROUP_BYTES = SLOT * 128;
  const long long blk_bytes = (long long)2 * ngh * GROUP_BYTES;
  // 16-byte pieces between the last feature of a half and the end of its last 32-column K chunk: the input-gradient
  // kernel reads whole chunks, so they are zeroed (by the otherwise idle chunk threads c >= nchunk)
  const int pad_pieces = ((((Fh + 31) >> 5) << 5) - Fh) >> 3;
  const uint32_t title_bytes = (uint32_t)L * F * sizeof(CT);
  const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_bar[0]);
  const uint32_t buf0 = (uint32_t)__cvta_generic_to_shared(att_smem);
  auto fetch_title = [&](int n, int b) {   // one thread
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * b), "r"(title_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     buf0 + (uint32_t)(b * buf_bytes)),
                 "l"(Cd + (long long)n * L * F), "r"(title_bytes), "r"(bar0 + 8 * b)
                 : "memory");
  };
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int f = tid; f < F; f += IMG_THREADS) ska[f] = ka[f];
  __syncthreads();
  float dka[8], dbc[8], dba = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) dka[i] = dbc[i] = 0.f;
  constexpr int DPR = 2;                            // d_pooled values per thread (F <= DPR * IMG_THREADS)
  float ndp[DPR], nw = 0.f, na = 0.f;
  auto prefetch_small = [&](int n) {
    const int no = (title_idx && n < N) ? __ldg(title_idx + n) : n;   // d_pooled rows live at the original title index
#pragma unroll
    for (int i = 0; i < DPR; ++i) {
      const int f = tid + i * IMG_THREADS;
      ndp[i] = (n < N && f < F) ? dp[(long long)no * lddp + f] : 0.f;
    }
    nw = (n < N && tid < L) ? w_in[(long long)n * L + tid] : 0.f;
    na = (n < N && tid < L) ? a_in[(long long)n * L + tid] : 0.f;
  };
  if (blockIdx.x < N) {
    if (tid == 0) fetch_title(blockIdx.x, 0);
    prefetch_small(blockIdx.x);
  }
  uint32_t phase[2] = {0, 0};
  int it = 0;
  for (int n = blockIdx.x; n < N; n += gridDim.x, ++it) {
    const int b = it & 1;
    const uint4* sC = reinterpret_cast<const uint4*>(att_smem + b * buf_bytes);  // [L][nchunk]
    __syncthreads();   // previous title fully consumed: its buffer, sdp and sw may be overwritten
    const int n_next = n + gridDim.x;
    if (tid == 0 && n_next < N) fetch_title(n_next, b ^ 1);
#pragma unroll
    for (int i = 0; i < DPR; ++i) {
      const int f = tid + i * IMG_THREADS;
      if (f < F) sdp[f] = ndp[i];
    }
    if (tid < L) sw[tid] = nw;
    const float a_cur = na;
    prefetch_small(n_next);
    {   // wait for this title's bulk copy
      uint32_t done = 0;
      while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar0 + 8 * b), "r"(phase[b])
            : "memory");
      }
      phase[b] ^= 1;
    }
    __syncthreads();
    {   // d w_t = c_t . d_pooled: a lane keeps its (at most two) chunks of d_pooled in registers for all rows
      float dpa[2][8];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int cc = lane + 32 * k;
        const float4 lo = cc < nchunk ? *reinterpret_cast<const float4*>(sdp + cc * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 hi = cc < nchunk ? *reinterpret_cast<const float4*>(sdp + cc * 8 + 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        dpa[k][0] = lo.x; dpa[k][1] = lo.y; dpa[k][2] = lo.z; dpa[k][3] = lo.w;
        dpa[k][4] = hi.x; dpa[k][5] = hi.y; dpa[k][6] = hi.z; dpa[k][7] = hi.w;
      }
#pragma unroll
      for (int tt = 0; tt < SLOT / 8; ++tt) {
        const int t = warp + tt * (IMG_THREADS / 32);
        if (t >= L) break;
        float dot = 0.f;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int cc = lane + 32 * k;
          if (cc < nchunk) {
            float v[8];
            unpack8<CT>(sC[t * nchunk + cc], v);
#pragma unroll
            for (int i = 0; i < 8; ++i) dot = fmaf(v[i], dpa[k][i], dot);
          }
        }
        dot = warp_sum(dot);
        if (lane == 0) sdw[t] = dot;
      }
    }
    __syncthreads();
    if (SLOT == 32) {
      if (tid < 32) {
        const float dwt = tid < L ? sdw[tid] : 0.f, wt = tid < L ? sw[tid] : 0.f;
        const float q = warp_sum(dwt * wt);
        const float dz = tid < L ? (dwt - q) * wt * (1.f - a_cur * a_cur) : 0.f;
        if (tid < L) sdz[tid] = dz;
        const float dzs = warp_sum(dz);
        if (tid == 0) dba += dzs;
      }
    } else {
      __shared__ float sq[2], sdzs[2];
      float dwt = 0.f, wt = 0.f;
      if (tid < SLOT) {
        dwt = tid < L ? sdw[tid] : 0.f; wt = tid < L ? sw[tid] : 0.f;
        const float qh = warp_sum(dwt * wt);
        if (lane == 0) sq[warp] = qh;
      }
      __syncthreads();
      if (tid < SLOT) {
        const float q = sq[0] + sq[1];
        const float dz = tid < L ? (dwt - q) * wt * (1.f - a_cur * a_cur) : 0.f;
        if (tid < L) sdz[tid] = dz;
        const float dzs = warp_sum(dz);
        if (lane == 0) sdzs[warp] = dzs;
      }
      __syncthreads();
      if (tid == 0) dba += sdzs[0] + sdzs[1];
    }
    __syncthreads();
    if (c_ok) {
      // d_pooled and the attention vector of this chunk, times the dropout keep scale.  (Packed fma.rn.f32x2 arithmetic
      // was measured here: 3 % slower — the pack/unpack moves cost more issue slots than the pairing saves.)
      float dpf[8], kaf[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) { dpf[i] = sdp[c * 8 + i] * (inv_keep * img_scale); kaf[i] = ska[c * 8 + i] * (inv_keep * img_scale); }
      const int hf = (c * 8 >= Fh) ? 1 : 0, fl = c * 8 - hf * Fh;
      const int g = hf * ngh + (fl >> 6), piece = (fl & 63) >> 3;
      uint8_t* dst0 = img + (long long)n * blk_bytes + (long long)g * GROUP_BYTES;
#pragma unroll
      for (int k = 0; k < SLOT / 4; ++k) {
        const int t = tg + 4 * k;
        float o[8];
        if (t < L) {
          float v[8];
          unpack8<CT>(sC[t * nchunk + c], v);
          const float wt = sw[t], dzt = sdz[t];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float gi = fmaf(wt, dpf[i], dzt * kaf[i]);
            o[i] = v[i] > 0.f ? gi : 0.f;
            dka[i] = fmaf(dzt, v[i], dka[i]);
            dbc[i] += o[i];
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = 0.f;
        }
        *reinterpret_cast<uint4*>(dst0 + t * 128 + ((piece ^ (t & 7)) << 4)) = pack8<CT>(o);
      }
    } else if (c - nchunk < 2 * pad_pieces) {
      const int k = c - nchunk, hf = k / pad_pieces, fl = Fh + (k % pad_pieces) * 8;
      const int g = hf * ngh + (fl >> 6), piece = (fl & 63) >> 3;
      uint8_t* dst0 = img + (long long)n * blk_bytes + (long long)g * GROUP_BYTES;
#pragma unroll
      for (int kk = 0; kk < SLOT / 4; ++kk) {
        const int t = tg + 4 * kk;
        *reinterpret_cast<uint4*>(dst0 + t * 128 + ((piece ^ (t & 7)) << 4)) = make_uint4(0, 0, 0, 0);
      }
    }
  }
  // combine the four row groups in a fixed order, then one partial row per CTA
  __syncthreads();
  if (tg > 0 && c_ok) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { sred[((tg - 1) * 64 + c) * 16 + i] = dka[i]; sred[((tg - 1) * 64 + c) * 16 + 8 + i] = dbc[i]; }
  }
  __syncthreads();
  float* out = partials + (long long)blockIdx.x * (2 * F + 1);
  if (tg == 0 && c_ok) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = dka[i], bsum = dbc[i];
#pragma unroll
      for (int g = 0; g < 3; ++g) { a += sred[(g * 64 + c) * 16 + i]; bsum += sred[(g * 64 + c) * 16 + 8 + i]; }
      out[c * 8 + i] = a;
      out[F + c * 8 + i] = bsum;
    }
  }
  if (tid == 0) out[2 * F] = dba;
}

// partials[grid][2F+1] -> d_att_w[F], d_conv_b[F], d_att_b[1] in a fixed order: 256 threads = 32 columns x 8 row
// strides; the eight stride sums of a column are combined in ascending order.
__global__ void attn_bwd_reduce_kernel(int grid, int F, const float* __restrict__ partials, float* __restrict__ d_att_w,
                                       float* __restrict__ d_conv_b, float* __restrict__ d_att_b, int accumulate,
                                       float cb_scale) {
  __shared__ float sm[8][32];
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c <= 2 * F)
    for (int g = part; g < grid; g += 8) s += partials[(long long)g * (2 * F + 1) + c];
  sm[part][lane] = s;
  __syncthreads();
  if (part != 0 || c > 2 * F) return;
  float t = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) t += sm[q][lane];
  float* dst = c < F ? d_att_w + c : (c < 2 * F ? d_conv_b + (c - F) : d_att_b);
  if (c >= F && c < 2 * F) t *= cb_scale;     // d conv_b was summed from loss-scaled dPre values
  *dst = accumulate ? *dst + t : t;
}

}  // namespace lstur

using namespace lstur;

extern "C" int lstur_attn_pool_fwd(int N, int L, int F, float* C, long long title_stride, const int* tokens,
                                   const float* att_w, const float* att_b, float* pooled, long long ldp, float* a_out,
                                   float* w_out, float dropout, unsigned seed, cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L > 0 && L <= ATT_MAX_L && F > 0 && dropout >= 0.f && dropout < 1.f, "lstur_attn_pool_fwd");
  if (N == 0) return LSTUR_OK;
  attn_pool_fwd_kernel<<<N, ATT_THREADS, 0, stream>>>(N, L, F, C, title_stride, tokens, att_w, att_b, pooled, ldp, a_out,
                                                      w_out, dropout > 0.f ? dropout_threshold(dropout) : 0u,
                                                      1.f / (1.f - dropout), seed);
  LSTUR_CHECK_LAUNCH("lstur_attn_pool_fwd");
  return LSTUR_OK;
}

// CTAs of the attention-backward kernels: one per title, at most 4 per SM of a 148-SM B200 (shared memory: two 25.6 KB
// title buffers + 3.2 KB per CTA at F=400; the final reduction scratch aliases the title buffers), and at least one
extern "C" int lstur_attn_bwd_grid(int N) {
  constexpr int max_ctas = 148 * 4;
  return N < max_ctas ? (N > 0 ? N : 1) : max_ctas;
}

extern "C" int lstur_colsum(long long rows, int cols, const float* in, long long ld, float* out, int accumulate,
                            float* workspace, size_t workspace_bytes, cudaStream_t stream) {
  LSTUR_REQUIRE(rows >= 0 && cols > 0, "lstur_colsum");
  int chunks = (int)((rows + 255) / 256);
  if (chunks > 1024) chunks = 1024;
  if (chunks < 1) chunks = 1;
  LSTUR_REQUIRE(workspace != nullptr && workspace_bytes >= (size_t)chunks * cols * sizeof(float), "lstur_colsum");
  int rpc = (int)((rows + chunks - 1) / chunks);
  if (rpc < 1) rpc = 1;
  dim3 g1(cdiv(cols, 128), chunks);
  colsum_stage1_kernel<<<g1, 128, 0, stream>>>(rows, cols, in, ld, rpc, workspace);
  LSTUR_CHECK_LAUNCH("lstur_colsum(stage1)");
  colsum_stage2_kernel<<<cdiv(cols, 32), 256, 0, stream>>>(chunks, cols, workspace, out, accumulate);
  LSTUR_CHECK_LAUNCH("lstur_colsum(stage2)");
  return LSTUR_OK;
}

// partials must hold lstur_attn_bwd_grid(N) * (2F+1) floats; after the call
// d_att_w[F], d_conv_b[F], d_att_b[1] are written (or accumulated).
extern "C" int lstur_attn_pool_bwd(int N, int L, int Lrows, int F, const float* Cd, long long title_stride,
                                   const float* a_in, const float* w_in, const float* d_pooled, long long lddp,
                                   const float* att_w, float* dPre, long long dpre_title_stride, float dropout,
                                   float* d_att_w, float* d_conv_b, float* d_att_b, int accumulate, float* partials,
                                   size_t partial_bytes, cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L > 0 && L <= ATT_MAX_L && Lrows >= L && F > 0 && F <= 8 * ATT_THREADS, "lstur_attn_pool_bwd");
  int grid = lstur_attn_bwd_grid(N);
  size_t need = (size_t)grid * (2 * F + 1) * sizeof(float);
  LSTUR_REQUIRE(partials != nullptr && partial_bytes >= need, "lstur_attn_pool_bwd");
  if (N == 0) {
    if (!accumulate) {
      cudaMemsetAsync(d_att_w, 0, F * sizeof(float), stream);
      cudaMemsetAsync(d_conv_b, 0, F * sizeof(float), stream);
      cudaMemsetAsync(d_att_b, 0, sizeof(float), stream);
    }
    return LSTUR_OK;
  }
  float inv_keep = 1.f / (1.f - dropout);
  int fpt = cdiv(F, ATT_THREADS);
#define LAUNCH(FPT_)                                                                                                  \
  attn_pool_bwd_kernel<FPT_><<<grid, ATT_THREADS, 0, stream>>>(N, L, Lrows, F, Cd, title_stride, a_in, w_in, d_pooled, lddp, \
                                                               att_w, dPre, dpre_title_stride, inv_keep, partials)
  if (fpt <= 1) LAUNCH(1);
  else if (fpt <= 2) LAUNCH(2);
  else if (fpt <= 4) LAUNCH(4);
  else LAUNCH(8);
#undef LAUNCH
  LSTUR_CHECK_LAUNCH("lstur_attn_pool_bwd");
  attn_bwd_reduce_kernel<<<cdiv(2 * F + 1, 32), 256, 0, stream>>>(grid, F, partials, d_att_w, d_conv_b, d_att_b,
                                                                     accumulate, 1.f);
  LSTUR_CHECK_LAUNCH("lstur_attn_pool_bwd(reduce)");
  return LSTUR_OK;
}

// Tensor-core backward: same arithmetic, dPre emitted as 16-bit K-block images for lstur_conv_wgrad_tc /
// lstur_conv_dgrad_tc (lstur_tc_dpre_img_bytes(N,L,F) bytes; title slots of lstur_tc_slot(L) rows, pad rows zero).
// The image holds img_scale * dPre (img_scale > 0, a power of two keeps it exact); the consumers divide it out.
extern "C" int lstur_attn_pool_bwd_img(int fp16, int N, int L, int F, const void* Cd_16, const float* a_in,
                                       const float* w_in, const float* d_pooled, long long lddp, const float* att_w,
                                       void* dpre_img, float dropout, float img_scale, float* d_att_w, float* d_conv_b,
                                       float* d_att_b, int accumulate, float* partials, size_t partial_bytes,
                                       const int* n_titles_dev, const int* title_idx, cudaStream_t stream) {
  LSTUR_REQUIRE(N >= 0 && L >= 1 && L <= 63 && F % 16 == 0 && F <= 512 && dpre_img != nullptr && img_scale > 0.f,
                "lstur_attn_pool_bwd_img");
  int grid = lstur_attn_bwd_grid(N);
  LSTUR_REQUIRE(partials != nullptr && partial_bytes >= (size_t)grid * (2 * F + 1) * sizeof(float), "lstur_attn_pool_bwd_img");
  if (N == 0) {
    if (!accumulate) {
      cudaMemsetAsync(d_att_w, 0, F * sizeof(float), stream);
      cudaMemsetAsync(d_conv_b, 0, F * sizeof(float), stream);
      cudaMemsetAsync(d_att_b, 0, sizeof(float), stream);
    }
    return LSTUR_OK;
  }
  const float inv_keep = 1.f / (1.f - dropout);
  const int slot = L <= 31 ? 32 : 64;
  size_t smem = (size_t)2 * slot * (F / 8) * 16 + (size_t)2 * F * sizeof(float);   // two title buffers + d_pooled + att_w
  if (smem < (size_t)3 * 64 * 16 * sizeof(float)) smem = (size_t)3 * 64 * 16 * sizeof(float);   // the final reduction scratch aliases the title buffers
#define IMG_LAUNCH(CT_, SLOT_)                                                                                          \
  do {                                                                                                                  \
    if (smem > 48 * 1024) cudaFuncSetAttribute(attn_bwd_img_kernel<CT_, SLOT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    attn_bwd_img_kernel<CT_, SLOT_><<<grid, IMG_THREADS, smem, stream>>>(N, L, F, (const CT_*)Cd_16, a_in, w_in, d_pooled, lddp, \
                                                                         att_w, (uint8_t*)dpre_img, inv_keep, img_scale, partials,       \
                                                                         n_titles_dev, title_idx);                       \
  } while (0)
  if (fp16 && slot == 32) IMG_LAUNCH(__half, 32);
  else if (fp16) IMG_LAUNCH(__half, 64);
  else if (slot == 32) IMG_LAUNCH(__nv_bfloat16, 32);
  else IMG_LAUNCH(__nv_bfloat16, 64);
#undef IMG_LAUNCH
  LSTUR_CHECK_LAUNCH("lstur_attn_pool_bwd_img");
  attn_bwd_reduce_kernel<<<cdiv(2 * F + 1, 32), 256, 0, stream>>>(grid, F, partials, d_att_w, d_conv_b, d_att_b, accumulate,
                                                                     1.f / img_scale);
  LSTUR_CHECK_LAUNCH("lstur_attn_pool_bwd_img(reduce)");
  return LSTUR_OK;
}
