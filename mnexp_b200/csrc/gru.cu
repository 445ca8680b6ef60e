// Masked Keras-2.2 GRU over the clicked-news sequence: recurrent part, forward and backward.
//
// Reference call sites: keras.layers.GRU(U)(Masking()(clicked), initial_state=user_vec)
// task/paper.py:612-613 (LSTUR-ini) and :596-611 (LSTUR-con); cook twin task/cook.py:152-168.
// Library semantics restated in SURVEY.md §9.4: gates z,r,h; hard_sigmoid
// recurrent activation; reset gate applied BEFORE the recurrent matmul;
// masked steps carry the state; output = last state.
//
// The input projection XW = H.Wx + b and all weight gradients are plain GEMMs
// done outside; these kernels only run the W-step sequential dependency.
// One CTA owns BT batch rows for all W steps: h lives in registers (thread j
// owns column j of every row) and is mirrored in shared memory for the
// matvec broadcast; the recurrent weights (G x 3G fp32, L2-resident) are
// streamed with coalesced loads each step.
#include "common.cuh"

namespace lstur {

constexpr int GRU_BT = 8;

__device__ __forceinline__ float rec_act(float x, int act) {
  return act == LSTUR_ACT_HARD_SIGMOID ? hard_sigmoid_f(x) : 1.f / (1.f + expf(-x));
}
__device__ __forceinline__ float rec_act_grad(float y, int act) {
  return act == LSTUR_ACT_HARD_SIGMOID ? ((y > 0.f && y < 1.f) ? 0.2f : 0.f) : y * (1.f - y);
}

template <int BT>
__device__ __forceinline__ void gru_fwd_body(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                                             const float* __restrict__ h0, long long ldh0, const float* __restrict__ Wh,
                                             int act, float* __restrict__ hT, long long ldo, float* __restrict__ Z,
                                             float* __restrict__ R, float* __restrict__ HH, float* __restrict__ HP,
                                             float* __restrict__ RH) {
  extern __shared__ float sm[];
  // rows of the mirrored state are padded to a multiple of 4 floats (zero tail) so that any G keeps the 128-bit reads
  // aligned: G = user_embedding_dim + vertical_embedding_dim = 215 at the reference's defaults (task/paper.py:1204-1208)
  const int Gs = (G + 3) & ~3;
  float* sh = sm;              // [BT][Gs]
  float* srh = sm + BT * Gs;   // [BT][Gs]
  const int j = threadIdx.x, b0 = blockIdx.x * BT;
  const bool act_j = j < G;
  const int G3 = 3 * G;
  float h[BT];
#pragma unroll
  for (int i = 0; i < BT; ++i) {
    int b = b0 + i;
    h[i] = (act_j && b < B && h0) ? h0[(long long)b * ldh0 + j] : 0.f;
    if (act_j) sh[i * Gs + j] = h[i];
    else if (j < Gs) { sh[i * Gs + j] = 0.f; srh[i * Gs + j] = 0.f; }
  }
  __syncthreads();
  for (int t = 0; t < W; ++t) {
    unsigned mbits = 0;
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B && gm[(long long)b * W + t] != 0.f) mbits |= 1u << i;
    }
    if (mbits == 0) {  // whole tile masked at this step (left padding): carry state
      if (HP && act_j) {
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          int b = b0 + i;
          if (b < B) {
            long long o = ((long long)b * W + t) * G + j;
            Z[o] = 0.f; R[o] = 0.f; HH[o] = 0.f; RH[o] = 0.f; HP[o] = h[i];
          }
        }
      }
      continue;
    }
    float az[BT], ar[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      bool ok = act_j && b < B;
      az[i] = ok ? XW[((long long)b * W + t) * G3 + j] : 0.f;
      ar[i] = ok ? XW[((long long)b * W + t) * G3 + G + j] : 0.f;
    }
    if (act_j) {
      for (int k = 0; k < G; k += 4) {
        float wz[4], wr[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const bool in = k + q < G;
          wz[q] = in ? __ldg(Wh + (long long)(k + q) * G3 + j) : 0.f;
          wr[q] = in ? __ldg(Wh + (long long)(k + q) * G3 + G + j) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          float4 hv = *(const float4*)(sh + i * Gs + k);
          az[i] = fmaf(hv.x, wz[0], az[i]); ar[i] = fmaf(hv.x, wr[0], ar[i]);
          az[i] = fmaf(hv.y, wz[1], az[i]); ar[i] = fmaf(hv.y, wr[1], ar[i]);
          az[i] = fmaf(hv.z, wz[2], az[i]); ar[i] = fmaf(hv.z, wr[2], ar[i]);
          az[i] = fmaf(hv.w, wz[3], az[i]); ar[i] = fmaf(hv.w, wr[3], ar[i]);
        }
      }
    }
    float z[BT], r[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      z[i] = rec_act(az[i], act);
      r[i] = rec_act(ar[i], act);
      if (act_j) srh[i * Gs + j] = r[i] * h[i];
    }
    __syncthreads();
    float ah[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      ah[i] = (act_j && b < B) ? XW[((long long)b * W + t) * G3 + 2 * G + j] : 0.f;
    }
    if (act_j) {
      for (int k = 0; k < G; k += 4) {
        float wh[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) wh[q] = k + q < G ? __ldg(Wh + (long long)(k + q) * G3 + 2 * G + j) : 0.f;
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          float4 v = *(const float4*)(srh + i * Gs + k);
          ah[i] = fmaf(v.x, wh[0], ah[i]);
          ah[i] = fmaf(v.y, wh[1], ah[i]);
          ah[i] = fmaf(v.z, wh[2], ah[i]);
          ah[i] = fmaf(v.w, wh[3], ah[i]);
        }
      }
    }
    __syncthreads();  // all reads of sh / srh for this step are done
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      bool on = (mbits >> i) & 1u;
      float hh = tanhf(ah[i]);
      float hn = z[i] * h[i] + (1.f - z[i]) * hh;
      if (HP && act_j && b < B) {
        long long o = ((long long)b * W + t) * G + j;
        Z[o] = on ? z[i] : 0.f;
        R[o] = on ? r[i] : 0.f;
        HH[o] = on ? hh : 0.f;
        RH[o] = on ? r[i] * h[i] : 0.f;
        HP[o] = h[i];
      }
      if (on) h[i] = hn;
      if (act_j) sh[i * Gs + j] = h[i];
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

// BPTT through the recurrence.  WhT is Wh transposed: (3G, G) row-major, so that
// thread k reads WhT[c*G + k] coalesced.  Produces dA = d(loss)/d(pre-activations)
// (B,W,3G) in gate order z,r,h (zero on masked steps) and dh0.
template <int BT>
__device__ __forceinline__ void gru_bwd_body(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ Z,
                                             const float* __restrict__ R, const float* __restrict__ HH,
                                             const float* __restrict__ HP, const float* __restrict__ WhT, int act,
                                             const float* __restrict__ dhT, long long lddh, float* __restrict__ dA,
                                             float* __restrict__ dh0, long long lddh0) {
  extern __shared__ float sm[];
  const int Gs = (G + 3) & ~3;      // padded row stride, zero tail (see the forward kernel)
  float* s_dah = sm;                // [BT][Gs]
  float* s_daz = sm + BT * Gs;      // [BT][Gs]
  float* s_dar = sm + 2 * BT * Gs;  // [BT][Gs]
  const int k = threadIdx.x, b0 = blockIdx.x * BT;
  const bool act_k = k < G;
  const int G3 = 3 * G;
  float dh[BT];
#pragma unroll
  for (int i = 0; i < BT; ++i) {
    int b = b0 + i;
    dh[i] = (act_k && b < B) ? dhT[(long long)b * lddh + k] : 0.f;
    if (!act_k && k < Gs) { s_dah[i * Gs + k] = 0.f; s_daz[i * Gs + k] = 0.f; s_dar[i * Gs + k] = 0.f; }
  }
  for (int t = W - 1; t >= 0; --t) {
    unsigned mbits = 0;
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B && gm[(long long)b * W + t] != 0.f) mbits |= 1u << i;
    }
    if (mbits == 0) {
      if (act_k) {
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          int b = b0 + i;
          if (b < B) {
            long long o = ((long long)b * W + t) * G3;
            dA[o + k] = 0.f; dA[o + G + k] = 0.f; dA[o + 2 * G + k] = 0.f;
          }
        }
      }
      continue;
    }
    float z[BT], r[BT], hp[BT], dhp[BT], dah[BT], daz[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      bool on = act_k && b < B && ((mbits >> i) & 1u);
      long long o = ((long long)b * W + t) * G + k;
      z[i] = on ? Z[o] : 0.f;
      r[i] = on ? R[o] : 0.f;
      hp[i] = on ? HP[o] : 0.f;
      float hh = on ? HH[o] : 0.f;
      float dz = dh[i] * (hp[i] - hh);
      float dhh = dh[i] * (1.f - z[i]);
      dah[i] = on ? dhh * (1.f - hh * hh) : 0.f;
      daz[i] = on ? dz * rec_act_grad(z[i], act) : 0.f;
      dhp[i] = dh[i] * z[i];
      if (act_k) {
        s_dah[i * Gs + k] = dah[i];
        s_daz[i * Gs + k] = daz[i];
      }
    }
    __syncthreads();
    float drh[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) drh[i] = 0.f;
    if (act_k) {
      for (int j = 0; j < G; j += 4) {
        float w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] = j + q < G ? __ldg(WhT + (long long)(2 * G + j + q) * G + k) : 0.f;
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          float4 v = *(const float4*)(s_dah + i * Gs + j);
          drh[i] = fmaf(v.x, w[0], drh[i]);
          drh[i] = fmaf(v.y, w[1], drh[i]);
          drh[i] = fmaf(v.z, w[2], drh[i]);
          drh[i] = fmaf(v.w, w[3], drh[i]);
        }
      }
    }
    float dar[BT];
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      float dr = drh[i] * hp[i];
      dhp[i] = fmaf(drh[i], r[i], dhp[i]);
      dar[i] = dr * rec_act_grad(r[i], act);
      if (act_k) s_dar[i * Gs + k] = dar[i];
    }
    __syncthreads();
    if (act_k) {
      for (int j = 0; j < G; j += 4) {
        float wz[4], wr[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const bool in = j + q < G;
          wz[q] = in ? __ldg(WhT + (long long)(j + q) * G + k) : 0.f;
          wr[q] = in ? __ldg(WhT + (long long)(G + j + q) * G + k) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < BT; ++i) {
          float4 vz = *(const float4*)(s_daz + i * Gs + j);
          float4 vr = *(const float4*)(s_dar + i * Gs + j);
          dhp[i] = fmaf(vz.x, wz[0], dhp[i]); dhp[i] = fmaf(vr.x, wr[0], dhp[i]);
          dhp[i] = fmaf(vz.y, wz[1], dhp[i]); dhp[i] = fmaf(vr.y, wr[1], dhp[i]);
          dhp[i] = fmaf(vz.z, wz[2], dhp[i]); dhp[i] = fmaf(vr.z, wr[2], dhp[i]);
          dhp[i] = fmaf(vz.w, wz[3], dhp[i]); dhp[i] = fmaf(vr.w, wr[3], dhp[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (act_k && b < B) {
        long long o = ((long long)b * W + t) * G3;
        dA[o + k] = daz[i];
        dA[o + G + k] = dar[i];
        dA[o + 2 * G + k] = dah[i];
      }
      if ((mbits >> i) & 1u) dh[i] = dhp[i];
    }
    __syncthreads();  // smem reused next step
  }
  if (act_k) {
#pragma unroll
    for (int i = 0; i < BT; ++i) {
      int b = b0 + i;
      if (b < B) dh0[(long long)b * lddh0 + k] = dh[i];
    }
  }
}

// Two instances of each kernel.  GRU_BT = 8 rows per CTA keeps 8 states per thread in registers, which limits the CTA
// to fewer threads than the widest G (140 registers: 448 threads forward).  Wider G takes the _wide instance: 4 rows per
// CTA under __launch_bounds__(1024), so one thread per unit fits for every G <= 1024.
constexpr int GRU_BT_WIDE = 4;

template <int BT>
__global__ void gru_fwd_kernel(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                               const float* __restrict__ h0, long long ldh0, const float* __restrict__ Wh, int act,
                               float* __restrict__ hT, long long ldo, float* __restrict__ Z, float* __restrict__ R,
                               float* __restrict__ HH, float* __restrict__ HP, float* __restrict__ RH) {
  gru_fwd_body<BT>(B, W, G, XW, gm, h0, ldh0, Wh, act, hT, ldo, Z, R, HH, HP, RH);
}
__global__ void __launch_bounds__(1024)
gru_fwd_kernel_wide(int B, int W, int G, const float* __restrict__ XW, const float* __restrict__ gm,
                    const float* __restrict__ h0, long long ldh0, const float* __restrict__ Wh, int act,
                    float* __restrict__ hT, long long ldo, float* __restrict__ Z, float* __restrict__ R,
                    float* __restrict__ HH, float* __restrict__ HP, float* __restrict__ RH) {
  gru_fwd_body<GRU_BT_WIDE>(B, W, G, XW, gm, h0, ldh0, Wh, act, hT, ldo, Z, R, HH, HP, RH);
}

template <int BT>
__global__ void gru_bwd_kernel(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ Z,
                               const float* __restrict__ R, const float* __restrict__ HH,
                               const float* __restrict__ HP, const float* __restrict__ WhT, int act,
                               const float* __restrict__ dhT, long long lddh, float* __restrict__ dA,
                               float* __restrict__ dh0, long long lddh0) {
  gru_bwd_body<BT>(B, W, G, gm, Z, R, HH, HP, WhT, act, dhT, lddh, dA, dh0, lddh0);
}
__global__ void __launch_bounds__(1024)
gru_bwd_kernel_wide(int B, int W, int G, const float* __restrict__ gm, const float* __restrict__ Z,
                    const float* __restrict__ R, const float* __restrict__ HH, const float* __restrict__ HP,
                    const float* __restrict__ WhT, int act, const float* __restrict__ dhT, long long lddh,
                    float* __restrict__ dA, float* __restrict__ dh0, long long lddh0) {
  gru_bwd_body<GRU_BT_WIDE>(B, W, G, gm, Z, R, HH, HP, WhT, act, dhT, lddh, dA, dh0, lddh0);
}

__global__ void transpose_kernel(int rows, int cols, const float* __restrict__ in, float* __restrict__ out) {
  __shared__ float tile[32][33];
  int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    if (x < cols && y0 + i < rows) tile[i][threadIdx.x] = in[(long long)(y0 + i) * cols + x];
  __syncthreads();
  int ox = blockIdx.y * 32 + threadIdx.x, oy0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    if (ox < rows && oy0 + i < cols) out[(long long)(oy0 + i) * rows + ox] = tile[threadIdx.x][i];
}

}  // namespace lstur

using namespace lstur;

extern "C" int lstur_transpose(int rows, int cols, const float* in, float* out, cudaStream_t stream) {
  LSTUR_REQUIRE(rows > 0 && cols > 0, "lstur_transpose");
  dim3 g(cdiv(cols, 32), cdiv(rows, 32)), b(32, 8);
  transpose_kernel<<<g, b, 0, stream>>>(rows, cols, in, out);
  LSTUR_CHECK_LAUNCH("lstur_transpose");
  return LSTUR_OK;
}

// XW (B,W,3G) = H.Wx + b precomputed; h0 may be NULL (zeros).  Z,R,HH,HP,RH are
// (B,W,G) saved tensors for the backward pass, all NULL for inference.
extern "C" int lstur_gru_fwd_streaming(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                             const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH,
                             float* HP, float* RH, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && G > 0 && G <= 1024, "lstur_gru_fwd_streaming");
  LSTUR_REQUIRE((Z && R && HH && HP && RH) || (!Z && !R && !HH && !HP && !RH), "lstur_gru_fwd_streaming");
  if (B == 0) return LSTUR_OK;
  static const int narrow_max = kernel_max_threads((const void*)gru_fwd_kernel<GRU_BT>);
  const int threads = cdiv(G, 32) * 32;
  const int bt = threads <= narrow_max ? GRU_BT : GRU_BT_WIDE;
  const void* fn = bt == GRU_BT ? (const void*)gru_fwd_kernel<GRU_BT> : (const void*)gru_fwd_kernel_wide;
  const size_t smem = (size_t)2 * bt * ((G + 3) & ~3) * sizeof(float);
  if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (bt == GRU_BT)
    gru_fwd_kernel<GRU_BT><<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, XW, gm, h0, ldh0, Wh, rec_act, hT, ldo, Z, R,
                                                                    HH, HP, RH);
  else
    gru_fwd_kernel_wide<<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, XW, gm, h0, ldh0, Wh, rec_act, hT, ldo, Z, R, HH,
                                                                 HP, RH);
  LSTUR_CHECK_LAUNCH("lstur_gru_fwd_streaming");
  return LSTUR_OK;
}

extern "C" int lstur_gru_bwd_streaming(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                             const float* HP, const float* WhT, int rec_act, const float* dhT, long long lddh,
                             float* dA, float* dh0, long long lddh0, cudaStream_t stream) {
  LSTUR_REQUIRE(B >= 0 && W > 0 && G > 0 && G <= 1024, "lstur_gru_bwd_streaming");
  if (B == 0) return LSTUR_OK;
  static const int narrow_max = kernel_max_threads((const void*)gru_bwd_kernel<GRU_BT>);
  const int threads = cdiv(G, 32) * 32;
  const int bt = threads <= narrow_max ? GRU_BT : GRU_BT_WIDE;
  const void* fn = bt == GRU_BT ? (const void*)gru_bwd_kernel<GRU_BT> : (const void*)gru_bwd_kernel_wide;
  const size_t smem = (size_t)3 * bt * ((G + 3) & ~3) * sizeof(float);
  if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (bt == GRU_BT)
    gru_bwd_kernel<GRU_BT><<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, gm, Z, R, HH, HP, WhT, rec_act, dhT, lddh, dA,
                                                                    dh0, lddh0);
  else
    gru_bwd_kernel_wide<<<cdiv(B, bt), threads, smem, stream>>>(B, W, G, gm, Z, R, HH, HP, WhT, rec_act, dhT, lddh, dA, dh0,
                                                                 lddh0);
  LSTUR_CHECK_LAUNCH("lstur_gru_bwd_streaming");
  return LSTUR_OK;
}

// Dispatchers: shared-memory-resident cluster kernels (gru_cl.cu) when the shape fits, else the streaming kernels.
// row_order (optional) is honoured by the cluster kernels only; the streaming kernels process the rows in order.
extern "C" int lstur_gru_fwd(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                             const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH,
                             float* HP, float* RH, const int* row_order, cudaStream_t stream) {
  if (lstur_gru_cluster_supported(B, W, G))
    return lstur_gru_fwd_cluster(B, W, G, XW, gm, h0, ldh0, Wh, rec_act, hT, ldo, Z, R, HH, HP, RH, row_order, stream);
  return lstur_gru_fwd_streaming(B, W, G, XW, gm, h0, ldh0, Wh, rec_act, hT, ldo, Z, R, HH, HP, RH, stream);
}

extern "C" int lstur_gru_bwd(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                             const float* HP, const float* WhT, int rec_act, const float* dhT, long long lddh,
                             float* dA, float* dh0, long long lddh0, const int* row_order, cudaStream_t stream) {
  if (lstur_gru_cluster_supported(B, W, G))
    return lstur_gru_bwd_cluster(B, W, G, gm, Z, R, HH, HP, WhT, rec_act, dhT, lddh, dA, dh0, lddh0, row_order, stream);
  return lstur_gru_bwd_streaming(B, W, G, gm, Z, R, HH, HP, WhT, rec_act, dhT, lddh, dA, dh0, lddh0, stream);
}
