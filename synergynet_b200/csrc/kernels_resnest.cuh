// CUDA-core pieces of the ResNeSt-50 backbone variant (reference backbone_nets/ResNeSt/resnet.py:29-127, splat.py:11-98):
// the split-attention of SplAtConv2d (radix 2, cardinality 1), its apply step with the fused `avd` pool, and the
// avg-down pool of the shortcut.  The convolutions themselves (deep stem 2 and 3, conv1 / conv2 (grouped) / conv3, the
// shortcut conv and the heads) run on tc_gemm_kernel (kernels_gemm.cuh); the first stem conv on stem_conv3x3s2_kernel.
// Activations are NHWC fp32; every kernel whose output feeds a GEMM also records max|x| per pixel (`rowmax`).
#pragma once
#include "common.cuh"

namespace syn {

constexpr int kRnsThreads = 256;

// per-pixel maximum of a block that covers whole pixels (ppb pixels x q4 channel quads): one smem atomic per thread
__device__ __forceinline__ void rns_block_rowmax(unsigned* s_max, int ppb, int lp, bool live, float m, unsigned* rowmax,
                                                 int pix0, int npix) {
  if (live) atomicMax(&s_max[lp], __float_as_uint(m));
  __syncthreads();
  if ((int)threadIdx.x < ppb && pix0 + (int)threadIdx.x < npix) rowmax[pix0 + threadIdx.x] = s_max[threadIdx.x];
}

// SplAtConv2d attention (splat.py:55-72): x = relu(bn0(conv(.))) as (B, HW, 2C) NHWC, split r = channels [rC, (r+1)C).
//   gap = mean_HW(x0 + x1); hid = relu(fc1'(gap)) with conv2.bn1 folded into fc1 (w1 [C/2][C], b1); logit = fc2(hid)
//   (w2 [2C][C/2], b2); att[r*C + c] = softmax_r(logit[r*C + c]) (rSoftMax, splat.py:84-98).
// One CTA per face.  C in {64, 128, 256, 512}: 256 threads = (pixel slice, channel quad).
__global__ void __launch_bounds__(kRnsThreads) resnest_attention_kernel(const float* __restrict__ x, const float* __restrict__ w1,
                                                                        const float* __restrict__ b1, const float* __restrict__ w2,
                                                                        const float* __restrict__ b2, float* __restrict__ att,
                                                                        int HW, int C) {
  __shared__ __align__(16) float s_part[kRnsThreads * 4];
  __shared__ float s_gap[512], s_hid[256], s_logit[1024];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int q4 = C >> 2, slices = kRnsThreads / q4, q = tid % q4, sl = tid / q4;
  const float* xb = x + (size_t)b * HW * 2 * C + 4 * q;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = sl; p < HW; p += slices) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(xb + (size_t)p * 2 * C));
    const float4 c = __ldg(reinterpret_cast<const float4*>(xb + (size_t)p * 2 * C + C));
    s.x += a.x + c.x; s.y += a.y + c.y; s.z += a.z + c.z; s.w += a.w + c.w;
  }
  *reinterpret_cast<float4*>(s_part + sl * C + 4 * q) = s;
  __syncthreads();
  for (int c = tid; c < C; c += kRnsThreads) {
    float t = 0.f;
    for (int i = 0; i < slices; ++i) t += s_part[i * C + c];
    s_gap[c] = t / (float)HW;
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31, I = C >> 1;
  for (int j = warp; j < I; j += kRnsThreads / 32) {            // fc1 (+ bn1) + relu: one warp per output
    float t = 0.f;
    for (int c = lane; c < C; c += 32) t = fmaf(__ldg(w1 + (size_t)j * C + c), s_gap[c], t);
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_hid[j] = fmaxf(t + __ldg(b1 + j), 0.f);
  }
  __syncthreads();
  for (int n = warp; n < 2 * C; n += kRnsThreads / 32) {        // fc2
    float t = 0.f;
    for (int k = lane; k < I; k += 32) t = fmaf(__ldg(w2 + (size_t)n * I + k), s_hid[k], t);
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_logit[n] = t + __ldg(b2 + n);
  }
  __syncthreads();
  for (int c = tid; c < C; c += kRnsThreads) {                  // softmax over the radix
    const float l0 = s_logit[c], l1 = s_logit[C + c], mx = fmaxf(l0, l1);
    const float e0 = expf(l0 - mx), e1 = expf(l1 - mx), inv = 1.f / (e0 + e1);
    att[(size_t)b * 2 * C + c] = e0 * inv;
    att[(size_t)b * 2 * C + C + c] = e1 * inv;
  }
}

// out = att0 * x0 + att1 * x1 (splat.py:74-79), x (B, H, H, 2C) -> y (B, HO, HO, C), and max|y| per output pixel.
// kPool: followed by the block's avd_layer AvgPool2d(3, 2, padding=1) (resnet.py:48-50,113-114; count_include_pad, so
// the divisor is always 9), HO = (H - 1) / 2 + 1.  Otherwise HO = H.
// Thread = (output pixel, channel quad); C / 4 divides the 256 threads of a block.
template <bool kPool>
__global__ void __launch_bounds__(kRnsThreads) resnest_apply_kernel(const float* __restrict__ x, const float* __restrict__ att,
                                                                    float* __restrict__ y, unsigned* __restrict__ rowmax,
                                                                    int batch, int H, int HO, int C) {
  __shared__ unsigned s_max[kRnsThreads / 16];
  const int q4 = C >> 2, ppb = kRnsThreads / q4, tid = threadIdx.x, lp = tid / q4, q = tid % q4;
  const int npix = batch * HO * HO, pix0 = blockIdx.x * ppb, pix = pix0 + lp;
  if (tid < ppb) s_max[tid] = 0u;
  __syncthreads();
  const bool live = pix < npix;
  float m = 0.f;
  if (live) {
    const int b = pix / (HO * HO);
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(att + (size_t)b * 2 * C + 4 * q));
    const float4 a1 = __ldg(reinterpret_cast<const float4*>(att + (size_t)b * 2 * C + C + 4 * q));
    auto apply = [&](size_t ipix, float4& o) {
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(x + ipix * 2 * C + 4 * q));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(x + ipix * 2 * C + C + 4 * q));
      o.x += a0.x * v0.x + a1.x * v1.x; o.y += a0.y * v0.y + a1.y * v1.y;
      o.z += a0.z * v0.z + a1.z * v1.z; o.w += a0.w * v0.w + a1.w * v1.w;
    };
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kPool) {
      const int r = pix - b * HO * HO, oy = r / HO, ox = r - oy * HO;
      for (int ky = 0; ky < 3; ++ky) {
        const int iy = 2 * oy - 1 + ky;
        if (iy < 0 || iy >= H) continue;
        for (int kx = 0; kx < 3; ++kx) {
          const int ix = 2 * ox - 1 + kx;
          if (ix >= 0 && ix < H) apply(((size_t)b * H + iy) * H + ix, o);
        }
      }
      o.x /= 9.f; o.y /= 9.f; o.z /= 9.f; o.w /= 9.f;
    } else {
      apply((size_t)pix, o);
    }
    *reinterpret_cast<float4*>(y + (size_t)pix * C + 4 * q) = o;
    m = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w)));
  }
  rns_block_rowmax(s_max, ppb, lp, live, m, rowmax, pix0, npix);
}

// Shortcut avg-down AvgPool2d(2, 2, ceil_mode=True, count_include_pad=False) (resnet.py:248-251): x (B, H, H, C) ->
// y (B, HO, HO, C), HO = ceil(H / 2); an edge window of an odd H holds 1 or 2 pixels and divides by its own count.
__global__ void __launch_bounds__(kRnsThreads) resnest_avgdown_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                                      unsigned* __restrict__ rowmax, int batch, int H, int HO,
                                                                      int C) {
  __shared__ unsigned s_max[kRnsThreads / 16];
  const int q4 = C >> 2, ppb = kRnsThreads / q4, tid = threadIdx.x, lp = tid / q4, q = tid % q4;
  const int npix = batch * HO * HO, pix0 = blockIdx.x * ppb, pix = pix0 + lp;
  if (tid < ppb) s_max[tid] = 0u;
  __syncthreads();
  const bool live = pix < npix;
  float m = 0.f;
  if (live) {
    const int b = pix / (HO * HO), r = pix - b * HO * HO, oy = r / HO, ox = r - oy * HO;
    const int y1 = min(2 * oy + 2, H), x1 = min(2 * ox + 2, H);
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int iy = 2 * oy; iy < y1; ++iy)
      for (int ix = 2 * ox; ix < x1; ++ix) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + (((size_t)b * H + iy) * H + ix) * C + 4 * q));
        o.x += v.x; o.y += v.y; o.z += v.z; o.w += v.w;
      }
    const float n = (float)((y1 - 2 * oy) * (x1 - 2 * ox));
    o.x /= n; o.y /= n; o.z /= n; o.w /= n;
    *reinterpret_cast<float4*>(y + (size_t)pix * C + 4 * q) = o;
    m = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w)));
  }
  rns_block_rowmax(s_max, ppb, lp, live, m, rowmax, pix0, npix);
}

}  // namespace syn
