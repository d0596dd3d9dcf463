// CUDA-core fp32 kernels of the hot path (SYN_ENGINE_SIMT_FP32 and the non-GEMM stages of every
// engine).  Activations are NHWC fp32; BatchNorm is already folded into (weight, bias).
//
// Reference ops replaced (paths relative to the reference root):
//   stem_conv3x3s2_kernel   ConvBNReLU(3,32,stride=2)          mobilenetv2_backbone.py:127
//   pointwise_gemm_kernel   1x1 Conv2d+BN(+ReLU6)(+skip)       mobilenetv2_backbone.py:60,65,71-74,136
//   depthwise3x3_kernel     3x3 depthwise Conv2d+BN+ReLU6      mobilenetv2_backbone.py:63
//   pool_heads_kernel       adaptive_avg_pool2d + 3 Linear+cat mobilenetv2_backbone.py:179-188
//   reconstruct_kernel      reconstruct_vertex_62              model_building.py:106-139
#pragma once
#include "common.cuh"

namespace syn {

// -------------------------------------------------------------------------------------------------
// uint8 crop -> fp32, `(img - 127.5) / 128` (synergy3DMM.py:192); used by the engines whose stem reads fp32.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) normalize_u8_kernel(const uint8_t* __restrict__ in, float* __restrict__ out,
                                                           size_t n4, int border) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  uchar4 u = reinterpret_cast<const uchar4*>(in)[i];
  if (border > 0) {            // CenterCrop(border, mode='test') of the reference loader (utils/ddfa.py:162-243): zero frame
    const int col = (int)(i % (kImg / 4)) * 4, iy = (int)((i / (kImg / 4)) % kImg);
    const bool row_out = iy < border || iy >= kImg - border;
    if (row_out || col < border || col >= kImg - border) u.x = 0;
    if (row_out || col + 1 < border || col + 1 >= kImg - border) u.y = 0;
    if (row_out || col + 2 < border || col + 2 >= kImg - border) u.z = 0;
    if (row_out || col + 3 < border || col + 3 >= kImg - border) u.w = 0;
  }
  reinterpret_cast<float4*>(out)[i] = make_float4(((float)u.x - 127.5f) / 128.0f, ((float)u.y - 127.5f) / 128.0f,
                                                   ((float)u.z - 127.5f) / 128.0f, ((float)u.w - 127.5f) / 128.0f);
}

// -------------------------------------------------------------------------------------------------
// Pose decode, batched: parse_pose + predict_pose of the reference (utils/inference.py:33-62,86-92,146-157).
//   P = (param * std + mean)[:12].reshape(3,4);  r1, r2 = rows / |rows| (fp32, like numpy);  r3 = r1 x r2;
//   angles (degrees, fp64 like Python's math.asin / atan2 on the fp32 matrix), t3d = P[:,3] moved to image
//   coordinates when a crop box is given: t3d[0] * (ex-sx)/120 + sx, t3d[1] * (ey-sy)/120 + sy.
// roi rows hold the five fp32 numbers the host derived in double like numpy's scalar handling:
//   kx = (ex-sx)/120, sx, ky = (ey-sy)/120, sy, kz = (kx+ky)/2.
// -------------------------------------------------------------------------------------------------
__global__ void pose_decode_kernel(const float* __restrict__ params, const float* __restrict__ mean, const float* __restrict__ stdv,
                                   const float* __restrict__ roi, double* __restrict__ angles, float* __restrict__ t3d, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  float P[12];
#pragma unroll
  for (int j = 0; j < 12; ++j) P[j] = __fadd_rn(__fmul_rn(params[(size_t)b * kNumParams + j], stdv[j]), mean[j]);
  // numpy: norm = sqrt(sum of squares) in fp32, sequential for three elements; no fused multiply-adds
  const float n1 = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(P[0], P[0]), __fmul_rn(P[1], P[1])), __fmul_rn(P[2], P[2])));
  const float n2 = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(P[4], P[4]), __fmul_rn(P[5], P[5])), __fmul_rn(P[6], P[6])));
  const float r1[3] = {__fdiv_rn(P[0], n1), __fdiv_rn(P[1], n1), __fdiv_rn(P[2], n1)};
  const float r2[3] = {__fdiv_rn(P[4], n2), __fdiv_rn(P[5], n2), __fdiv_rn(P[6], n2)};
  // np.cross(r1, r2) row: (a1*b2 - a2*b1, a2*b0 - a0*b2, a0*b1 - a1*b0), each product rounded
  const float r3[3] = {__fsub_rn(__fmul_rn(r1[1], r2[2]), __fmul_rn(r1[2], r2[1])),
                       __fsub_rn(__fmul_rn(r1[2], r2[0]), __fmul_rn(r1[0], r2[2])),
                       __fsub_rn(__fmul_rn(r1[0], r2[1]), __fmul_rn(r1[1], r2[0]))};
  const double R00 = r1[0], R01 = r1[1], R02 = r1[2], R12 = r2[2], R20 = r3[0], R22 = r3[2];
  const double kPi = 3.14159265358979323846;
  double x, y, z;
  if (R20 != 1.0 && R20 != -1.0) {                           // matrix2angle_corr, utils/inference.py:45-62
    x = asin(R20);
    y = atan2(R12 / cos(x), R22 / cos(x));
    z = atan2(R01 / cos(x), R00 / cos(x));
  } else {                                                   // gimbal lock
    z = 0.0;
    if (R20 == -1.0) { x = kPi / 2; y = z + atan2(R01, R02); }
    else { x = -kPi / 2; y = -z + atan2(-R01, -R02); }
  }
  angles[(size_t)b * 3 + 0] = x * 180 / kPi;
  angles[(size_t)b * 3 + 1] = y * 180 / kPi;
  angles[(size_t)b * 3 + 2] = z * 180 / kPi;
  float t0 = P[3], t1 = P[7];
  if (roi != nullptr) {
    const float* r = roi + (size_t)b * 5;
    t0 = __fadd_rn(__fmul_rn(t0, r[0]), r[1]);
    t1 = __fadd_rn(__fmul_rn(t1, r[2]), r[3]);
  }
  t3d[(size_t)b * 3 + 0] = t0; t3d[(size_t)b * 3 + 1] = t1; t3d[(size_t)b * 3 + 2] = P[11];
}

// -------------------------------------------------------------------------------------------------
// Stem: (B,3,120,120) NCHW -> (B,60,60,32) NHWC, 3x3 stride 2 pad 1, +bias, then
//   kRelu6 = true:  ReLU6                       (MobileNetV2 features.0, mobilenetv2_backbone.py:127)
//   kRelu6 = false: ReLU, and max|y| per output pixel into rowmax (ResNeSt-50 deep stem conv1.0-2,
//                   ResNeSt/resnet.py:182-185; the next layer is a dynamically scaled tc_gemm conv)
// One CTA per output row (b, oy); 256 threads = 64 pixel slots x 4 channel groups of 8.
// Weights packed [27][32] with tap index (ci*3+ky)*3+kx.
// -------------------------------------------------------------------------------------------------
constexpr int kStemThreads = 256;

template <bool kRelu6>
__global__ void __launch_bounds__(kStemThreads)
stem_conv3x3s2_kernel(const float* __restrict__ x, const float* __restrict__ w,
                      const float* __restrict__ bias, float* __restrict__ y, int batch,
                      unsigned* __restrict__ rowmax) {
  constexpr int HI = kImg, HO = 60, CO = 32;
  __shared__ float s_in[3][3][HI + 4];   // [ci][ky][ix+1], column 0 is the left zero pad
  __shared__ __align__(16) float s_w[27 * CO];
  __shared__ float s_b[CO];
  const int b = blockIdx.x / HO, oy = blockIdx.x % HO;
  const int tid = threadIdx.x;
  for (int i = tid; i < 27 * CO; i += kStemThreads) s_w[i] = w[i];
  if (tid < CO) s_b[tid] = bias[tid];
  for (int i = tid; i < 9 * (HI + 1); i += kStemThreads) {
    const int c = i % (HI + 1), r = i / (HI + 1);      // r = ci*3+ky
    const int ci = r / 3, ky = r % 3;
    const int iy = 2 * oy - 1 + ky, ix = c - 1;
    float v = 0.f;
    if (iy >= 0 && iy < HI && ix >= 0) v = x[((size_t)(b * 3 + ci) * HI + iy) * HI + ix];
    s_in[ci][ky][c] = v;
  }
  __syncthreads();
  const int px = tid >> 2, cg = tid & 3;
  if (kRelu6 && px >= HO) return;
  // rowmax variant: the idle slots (px >= HO) stay for the shuffles of the pixel maximum and compute a valid pixel
  const int pxc = px < HO ? px : HO - 1;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = s_b[cg * 8 + j];
#pragma unroll
  for (int ci = 0; ci < 3; ++ci)
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const float v = s_in[ci][ky][2 * pxc + kx];
        const float4 w0 = *reinterpret_cast<const float4*>(&s_w[((ci * 3 + ky) * 3 + kx) * CO + cg * 8]);
        const float4 w1 = *reinterpret_cast<const float4*>(&s_w[((ci * 3 + ky) * 3 + kx) * CO + cg * 8 + 4]);
        acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]);
        acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
        acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]);
        acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
      }
  float4* out = reinterpret_cast<float4*>(y + ((size_t)(b * HO + oy) * HO + pxc) * CO + cg * 8);
  if (kRelu6) {
    out[0] = make_float4(relu6f(acc[0]), relu6f(acc[1]), relu6f(acc[2]), relu6f(acc[3]));
    out[1] = make_float4(relu6f(acc[4]), relu6f(acc[5]), relu6f(acc[6]), relu6f(acc[7]));
  } else {
    float m = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j] = fmaxf(acc[j], 0.f);
      m = fmaxf(m, acc[j]);
    }
    if (px < HO) {
      out[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      out[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));      // the 4 channel groups of a pixel are adjacent lanes
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
    if (px < HO && cg == 0) rowmax[((size_t)b * HO + oy) * HO + px] = __float_as_uint(m);
  }
}

// -------------------------------------------------------------------------------------------------
// Pointwise (1x1) convolution as an fp32 SIMT GEMM:
//   out[M,N] = act(A[M,K] * W[K,N] + bias[N]) (+ residual[M,N]),  M = B*H*W pixels (NHWC rows).
// BMxBN tile per CTA, BK=16, TMxTN outer product per thread.  K, N are multiples of 8.
// -------------------------------------------------------------------------------------------------
template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
pointwise_gemm_kernel(const float* __restrict__ A, const float* __restrict__ W,
                      const float* __restrict__ bias, const float* __restrict__ residual,
                      float* __restrict__ out, int M, int K, int N, int relu6) {
  constexpr int BK = 16;
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int PAD = 4;
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x;
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
    // A tile: BM rows x 4 float4 (along K), stored transposed.
    for (int i = tid; i < BM * (BK / 4); i += NT) {
      const int row = i / (BK / 4), kq = i % (BK / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + row < M && k0 + kq * 4 < K)
        v = *reinterpret_cast<const float4*>(A + (size_t)(m0 + row) * K + k0 + kq * 4);
      As[kq * 4 + 0][row] = v.x; As[kq * 4 + 1][row] = v.y;
      As[kq * 4 + 2][row] = v.z; As[kq * 4 + 3][row] = v.w;
    }
    for (int i = tid; i < BK * (BN / 4); i += NT) {
      const int kr = i / (BN / 4), nq = i % (BN / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k0 + kr < K && n0 + nq * 4 < N)
        v = *reinterpret_cast<const float4*>(W + (size_t)(k0 + kr) * N + n0 + nq * 4);
      *reinterpret_cast<float4*>(&Bs[kr][nq * 4]) = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&As[k][ty * TM + i]);
        a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
      }
#pragma unroll
      for (int j = 0; j < TN; j += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&Bs[k][tx * TN + j]);
        b[j] = v.x; b[j + 1] = v.y; b[j + 2] = v.z; b[j + 3] = v.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty * TM + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; j += 4) {
      const int n = n0 + tx * TN + j;
      if (n >= N) continue;
      const float4 bv = *reinterpret_cast<const float4*>(bias + n);
      float4 v = make_float4(acc[i][j] + bv.x, acc[i][j + 1] + bv.y, acc[i][j + 2] + bv.z,
                             acc[i][j + 3] + bv.w);
      if (relu6) { v.x = relu6f(v.x); v.y = relu6f(v.y); v.z = relu6f(v.z); v.w = relu6f(v.w); }
      if (residual != nullptr) {
        const float4 r = *reinterpret_cast<const float4*>(residual + (size_t)m * N + n);
        v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
      }
      *reinterpret_cast<float4*>(out + (size_t)m * N + n) = v;
    }
  }
}

// -------------------------------------------------------------------------------------------------
// Depthwise 3x3, pad 1, stride 1|2, +bias, ReLU6.  NHWC; one thread per (output pixel, 4 channels).
// Weights packed [9][C].
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
depthwise3x3_kernel(const float* __restrict__ x, const float* __restrict__ w,
                    const float* __restrict__ bias, float* __restrict__ y, int batch, int C,
                    int HI, int HO, int stride) {
  const int c4n = C >> 2;
  const size_t total = (size_t)batch * HO * HO * c4n;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c4 = (int)(idx % c4n);
  size_t pix = idx / c4n;
  const int ox = (int)(pix % HO);
  pix /= HO;
  const int oy = (int)(pix % HO);
  const int b = (int)(pix / HO);
  float4 acc = *reinterpret_cast<const float4*>(bias + c4 * 4);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int iy = oy * stride - 1 + ky;
    if (iy < 0 || iy >= HI) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int ix = ox * stride - 1 + kx;
      if (ix < 0 || ix >= HI) continue;
      const float4 v = *reinterpret_cast<const float4*>(x + ((size_t)(b * HI + iy) * HI + ix) * C + c4 * 4);
      const float4 wv = *reinterpret_cast<const float4*>(w + (ky * 3 + kx) * C + c4 * 4);
      acc.x = fmaf(v.x, wv.x, acc.x); acc.y = fmaf(v.y, wv.y, acc.y);
      acc.z = fmaf(v.z, wv.z, acc.z); acc.w = fmaf(v.w, wv.w, acc.w);
    }
  }
  acc.x = relu6f(acc.x); acc.y = relu6f(acc.y); acc.z = relu6f(acc.z); acc.w = relu6f(acc.w);
  *reinterpret_cast<float4*>(y + ((size_t)(b * HO + oy) * HO + ox) * C + c4 * 4) = acc;
}

// -------------------------------------------------------------------------------------------------
// Global average pool over the 4x4 map + the three Linear heads (concatenated to 62 outputs).
// One CTA per face.  feat: (B,16,1280) NHWC; Wh: (62,1280) row-major; bh: (62).
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pool_heads_kernel(const float* __restrict__ feat, const float* __restrict__ Wh,
                  const float* __restrict__ bh, float* __restrict__ params,
                  float* __restrict__ pool_out, int npix) {
  __shared__ __align__(16) float s_pool[kLastCh];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float inv = 1.0f / (float)npix;
  const float* f = feat + (size_t)b * npix * kLastCh;
  for (int c = tid; c < kLastCh; c += 256) {
    float s = 0.f;
    for (int p = 0; p < npix; ++p) s += f[(size_t)p * kLastCh + c];
    s *= inv;
    s_pool[c] = s;
    if (pool_out != nullptr) pool_out[(size_t)b * kLastCh + c] = s;
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int j = warp; j < kNumParams; j += 8) {
    const float* wr = Wh + (size_t)j * kLastCh;
    float s = 0.f;
    for (int c = lane * 4; c < kLastCh; c += 128) {
      const float4 wv = *reinterpret_cast<const float4*>(wr + c);
      const float4 pv = *reinterpret_cast<const float4*>(&s_pool[c]);
      s = fmaf(wv.x, pv.x, s); s = fmaf(wv.y, pv.y, s);
      s = fmaf(wv.z, pv.z, s); s = fmaf(wv.w, pv.w, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) params[(size_t)b * kNumParams + j] = s + bh[j];
  }
}

// -------------------------------------------------------------------------------------------------
// 3DMM reconstruction, sparse and dense (one kernel family so dense[:, :, kp] == sparse bit for
// bit when the sparse basis is the keypoint gather of the dense one).
//   basis: planar [51][3][nv_pad] fp32: plane 0 = mean shape u, planes 1..40 = w_shp columns,
//          41..50 = w_exp columns; inner [3] = x|y|z, nv_pad = nver rounded up to 128.
//   params (B,62) whitened (or already de-whitened when whitening == 0).
//   out (B,3,nver).
// Thread = vertex, F faces per CTA: the basis element is loaded once and reused for F faces.
// -------------------------------------------------------------------------------------------------
template <int F>
__global__ void __launch_bounds__(128)
reconstruct_kernel(const float* __restrict__ basis, const float* __restrict__ params,
                   const float* __restrict__ mean, const float* __restrict__ stdv,
                   float* __restrict__ out, int batch, int nver, int nv_pad, int whitening,
                   int transform) {
  __shared__ float s_par[F][kNumParams + 2];
  const int tid = threadIdx.x;
  const int b0 = blockIdx.y * F;
  for (int i = tid; i < F * kNumParams; i += 128) {
    const int f = i / kNumParams, j = i % kNumParams;
    float v = 0.f;
    if (b0 + f < batch) {
      v = params[(size_t)(b0 + f) * kNumParams + j];
      if (whitening) v = v * stdv[j] + mean[j];      // model_building.py:117 (mul then add)
    }
    s_par[f][j] = v;
  }
  __syncthreads();
  const int v = blockIdx.x * 128 + tid;              // < nv_pad by construction
  const size_t plane = (size_t)3 * nv_pad;
  float sx[F], sy[F], sz[F];
  {
    const float ux = basis[v], uy = basis[nv_pad + v], uz = basis[2 * (size_t)nv_pad + v];
#pragma unroll
    for (int f = 0; f < F; ++f) { sx[f] = ux; sy[f] = uy; sz[f] = uz; }
  }
#pragma unroll 2
  for (int k = 0; k < kNumAlpha; ++k) {
    const float* bp = basis + (size_t)(k + 1) * plane + v;
    const float bx = bp[0], by = bp[nv_pad], bz = bp[2 * (size_t)nv_pad];
#pragma unroll
    for (int f = 0; f < F; ++f) {
      const float a = s_par[f][12 + k];
      sx[f] = fmaf(bx, a, sx[f]); sy[f] = fmaf(by, a, sy[f]); sz[f] = fmaf(bz, a, sz[f]);
    }
  }
  if (v >= nver) return;
#pragma unroll
  for (int f = 0; f < F; ++f) {
    if (b0 + f >= batch) break;
    const float* p = s_par[f];                       // row-major 3x4 [R|t], model_building.py:27-29
    float X = fmaf(p[0], sx[f], fmaf(p[1], sy[f], p[2] * sz[f])) + p[3];
    float Y = fmaf(p[4], sx[f], fmaf(p[5], sy[f], p[6] * sz[f])) + p[7];
    float Z = fmaf(p[8], sx[f], fmaf(p[9], sy[f], p[10] * sz[f])) + p[11];
    if (transform) Y = (float)(kImg + 1) - Y;        // model_building.py:129,137
    float* o = out + (size_t)(b0 + f) * 3 * nver + v;
    o[0] = X; o[nver] = Y; o[2 * (size_t)nver] = Z;
  }
}

}  // namespace syn
