// General fp32-accurate GEMM / implicit-GEMM convolution on tcgen05 for the layers outside the fused MobileNetV2
// blocks: the PointNet refinement heads MLP_for / MLP_rev (reference backbone_nets/pointnet_backbone.py:31-64,
// 90-106; Conv1d(k=1) + BatchNorm1d + ReLU over B x 68 points), the ResNet-50 backbone variant
// (backbone_nets/resnet_backbone.py:227-249; 1x1 / 3x3 convolutions + BatchNorm2d + ReLU, NHWC here) and the
// ResNeSt-50 variant (backbone_nets/ResNeSt/resnet.py, splat.py; including the radix-2 grouped 3x3 convolution).
//
//   out[m, n] = act( sum_k A[m, k] * W[n, k] * oscale[n] + bias[n] + addend[m / group, n] + residual[m, n] )
//
// Precision: the split-fp16 x3 scheme of kernels_tc.cuh, but with a DYNAMIC power-of-two scale per A row instead of
// the fixed kActScale: the producing layer's epilogue records max|x| of every row (`rowmax`, atomicMax on the fp32
// bit pattern), and the consumer scales row m by 2^e(m) so that its largest element lands in [2^13, 2^14) before
// the hi/lo split -- exact, undone by one multiply in the epilogue, and immune to the |x| < ~937 range limit of
// the fixed scale (ReLU outputs of these layers are unbounded).
//
// Roles: warps 0-7 = producers (thread = GEMM row x half of a chunk's k groups: gathers the fp32 row -- or, in conv
// mode, the k x k x C patch of an NHWC pixel -- splits it and stores the canonical K-major operand), then the epilogue
// (lane quarter = warp & 3, column half = warp >> 2); warp 8 = bulk-copy of the
// pre-packed weight chunks + MMA issue (converged warp, elect.sync).  K streams in chunks of 32 through a 4-stage
// ring (193 KB smem): the fp32 rows come from global memory / L2 and three chunks of look-ahead cover their latency.
#pragma once
#include "common.cuh"
#include "tc_common.cuh"

namespace syn {

constexpr int kGmKC = 32;                                 // K chunk
constexpr int kGmStages = 4;                              // chunk ring: global-load latency of three chunks hidden
constexpr int kGmProducerWarps = 8;                       // thread = (GEMM row, half of the chunk's k groups)
constexpr int kGmThreads = (kGmProducerWarps + 1) * 32;
constexpr int kGmMaxNr = 256;
constexpr int kGmStageA = 128 * kGmKC * 2;                // 8 KB: one plane (hi or lo) of the A tile
constexpr int kGmStageB = kGmMaxNr * kGmKC * 2;           // 16 KB
constexpr int kGmStage = 2 * kGmStageA + 2 * kGmStageB;   // 48 KB
constexpr int kGmSmem = kGmStages * kGmStage + 1024;

enum { kActNone = 0, kActRelu6 = 1, kActRelu = 2 };

struct GemmArgs {
  const float* A;            // plain mode: [M][lda]; conv mode: NHWC activations (B, H, W, C)
  const uint8_t* Wimg;       // per n-range, per K chunk: [hi plane nr x kc][lo plane]  (pack_gemm_weights)
  const float* bias;         // [N] (BatchNorm folded), never null
  const float* oscale;       // [N]: 1 / weight scale of the channel
  const float* addend;       // nullable: [M / addend_group][N], broadcast over the rows of a group (PointNet conv6)
  const float* residual;     // nullable: [M][N], added before the activation (ResNet shortcut)
  float* out;                // nullable: [M][N]
  const unsigned* rowmax_in; // max|a| per source row as fp32 bits (conv mode: per input pixel)
  unsigned* rowmax_out;      // nullable: atomicMax of |out| per output row
  unsigned* colmax_out;      // nullable: max over the rows of a group per channel (PointNet max-pool; values >= 0)
  int addend_group, colmax_group;
  int M, K, N, Kp, nr, lda, act;
  // conv mode (ksize > 0): implicit GEMM over k = (ky * ksize + kx) * C + c
  int ksize, stride, pad, H, W, C, HO, WO;
  // grouped conv mode: C is the per-group input channel count, a_pix the channel count of an input pixel (= C when
  // ungrouped); the CTA of n-range n0 is in group n0 / n_group (n_group = output channels per group, 0 = ungrouped;
  // nr divides it) and reads input channels [group * C, (group + 1) * C)
  int n_group, a_pix;
  // accumulator split (0 = one TMEM accumulator for all three passes).  The tensor cores round each accumulator update
  // toward zero, so the error of a sum grows with the number of updates times the accumulator's magnitude; with
  // acc_slices = S > 0 the hi*hi products of chunk c go to accumulator c % S and the two small correction passes to a
  // separate one (S + 1 buffers of nr columns in a 512-column allocation), summed in fp32 by the epilogue
  int acc_slices;
  int* err;
};

// exponent e such that max * 2^e lies in [2^13, 2^14); max == 0 (all-zero row) -> 0
__device__ __forceinline__ int gemm_row_exp(unsigned maxbits) {
  const int be = (int)((maxbits >> 23) & 0xffu);
  if (be == 0 || be == 255) return 0;                 // zero / denormal row, or inf / nan (propagates unscaled)
  return max(-100, min(100, 13 - (be - 127)));
}
__device__ __forceinline__ float exp2i(int e) { return __uint_as_float((unsigned)(e + 127) << 23); }   // |e| <= 126

__global__ void __launch_bounds__(kGmThreads, 1) tc_gemm_kernel(const GemmArgs p) {
  using namespace tc;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[kGmStages], bar_empty[kGmStages], bar_acc;
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float s_bias[kGmMaxNr], s_osc[kGmMaxNr];       // epilogue constants of this n-range
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int m0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * p.nr;
  for (int i = tid; i < p.nr; i += kGmThreads) {              // the packed arrays are padded to nranges * nr entries
    s_bias[i] = p.bias[n0 + i];
    s_osc[i] = p.oscale[n0 + i];
  }
  const int nchunks = (p.Kp + kGmKC - 1) / kGmKC;
  const int nsl = min(p.acc_slices, nchunks);                  // hi*hi slices in use (split accumulators), 0 = off
  const uint8_t* wimg = p.Wimg + (size_t)blockIdx.y * (size_t)p.nr * p.Kp * 4;

  if (tid == 0) {
    for (int i = 0; i < kGmStages; ++i) {
      mbar_init(smem_u32(&bar_full[i]), kGmProducerWarps * 32 + 1);   // producer arrivals + the weight copy's expect_tx arrival
      mbar_init(smem_u32(&bar_empty[i]), 1);
    }
    mbar_init(smem_u32(&bar_acc), 1);
    fence_mbar_init();
  }
  if (warp == kGmProducerWarps) {
    if (p.acc_slices > 0) tmem_alloc<512>(smem_u32(&tmem_base_s));
    else tmem_alloc<256>(smem_u32(&tmem_base_s));
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  auto stage_a = [&](int s, int plane) { return smem + s * kGmStage + plane * kGmStageA; };
  auto stage_b = [&](int s, int plane) { return smem + s * kGmStage + 2 * kGmStageA + plane * kGmStageB; };

  if (warp < kGmProducerWarps) {
    // ------------------------------ producers ---------------------------------------------------
    const int row = tid & 127, kh = tid >> 7, m = m0 + row;        // kh: which two of the chunk's four 8-element k groups
    const bool row_ok = m < p.M;
    int b = 0, oy = 0, ox = 0;
    unsigned mx = 0;
    if (p.ksize > 0) {
      if (row_ok) {
        b = m / (p.HO * p.WO);
        const int r = m - b * p.HO * p.WO;
        oy = r / p.WO; ox = r - oy * p.WO;
        for (int ky = 0; ky < p.ksize; ++ky)
          for (int kx = 0; kx < p.ksize; ++kx) {
            const int iy = oy * p.stride - p.pad + ky, ix = ox * p.stride - p.pad + kx;
            if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) mx = max(mx, p.rowmax_in[((size_t)b * p.H + iy) * p.W + ix]);
          }
      }
    } else if (row_ok) {
      mx = p.rowmax_in[m];
    }
    const int e_row = gemm_row_exp(mx);
    const float a_scale = exp2i(e_row);
    const float* arow = p.A + (size_t)m * p.lda;
    const float* abase = p.A + (p.n_group > 0 ? (n0 / p.n_group) * p.C : 0);   // grouped conv: this CTA's input channels
    for (int c = 0; c < nchunks; ++c) {
      const int s = c % kGmStages, use = c / kGmStages;
      const int k0 = c * kGmKC;
      const int kc = min(kGmKC, p.Kp - k0);
      // gather first (the loads do not depend on the slot), then wait for the slot: the global latency overlaps the wait
      float4 va[2], ve[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int kg = kh * 2 + q, k = k0 + kg * 8;
        const float* src = nullptr;
        if (row_ok && kg * 8 < kc && k < p.K) {
          if (p.ksize > 0) {
            const int tap = k / p.C, cc = k - tap * p.C;
            const int ky = tap / p.ksize, kx = tap - ky * p.ksize;
            const int iy = oy * p.stride - p.pad + ky, ix = ox * p.stride - p.pad + kx;
            if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) src = abase + (((size_t)b * p.H + iy) * p.W + ix) * p.a_pix + cc;
          } else {
            src = arow + k;
          }
        }
        va[q] = make_float4(0.f, 0.f, 0.f, 0.f); ve[q] = va[q];
        if (src != nullptr) {                                 // K and C are multiples of 8, rows 16-byte aligned
          va[q] = __ldg(reinterpret_cast<const float4*>(src));
          ve[q] = __ldg(reinterpret_cast<const float4*>(src + 4));
        }
      }
      mbar_wait(smem_u32(&bar_empty[s]), (use & 1) ^ 1, p.err);
      uint8_t* ah = stage_a(s, 0) + (row >> 3) * 128 + (row & 7) * 16;
      uint8_t* al = stage_a(s, 1) + (row >> 3) * 128 + (row & 7) * 16;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int kg = kh * 2 + q;
        if (kg * 8 < kc) {
          uint32_t h[4], l[4];
          split2_f16(va[q].x * a_scale, va[q].y * a_scale, h[0], l[0]);
          split2_f16(va[q].z * a_scale, va[q].w * a_scale, h[1], l[1]);
          split2_f16(ve[q].x * a_scale, ve[q].y * a_scale, h[2], l[2]);
          split2_f16(ve[q].z * a_scale, ve[q].w * a_scale, h[3], l[3]);
          *reinterpret_cast<uint4*>(ah + kg * 2048) = make_uint4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<uint4*>(al + kg * 2048) = make_uint4(l[0], l[1], l[2], l[3]);
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(smem_u32(&bar_full[s]));
    }
    // ------------------------------ epilogue ----------------------------------------------------
    mbar_wait(smem_u32(&bar_acc), 0, p.err);
    tc_fence_after_sync();
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int ncols = min(p.nr, p.N - n0);
    const float inv_a = exp2i(-e_row);
    float* orow = p.out ? p.out + (size_t)m * p.N + n0 : nullptr;
    const float* rrow = p.residual ? p.residual + (size_t)m * p.N + n0 : nullptr;
    const float* arow2 = p.addend ? p.addend + (size_t)(m / p.addend_group) * p.N + n0 : nullptr;
    unsigned* crow = p.colmax_out ? p.colmax_out + (size_t)(m / p.colmax_group) * p.N + n0 : nullptr;
    float rmax = 0.f;
    const bool vec = (p.N & 3) == 0;                           // rows of out / residual / addend are 16-byte aligned
    // max-pool over the rows of a group (PointNet): the 32 rows of a warp almost always belong to one group (68 points
    // per face), so the warp reduces first (redux.sync) and issues ONE atomic per column instead of 32 on one address
    const int cgrp = crow ? m / p.colmax_group : 0;
    const bool warp_one_group = crow != nullptr && __all_sync(0xffffffffu, cgrp == __shfl_sync(0xffffffffu, cgrp, 0) && row_ok);
    auto pool_max = [&](int col, float o) {                    // warp-uniform call sites only
      const unsigned bits = row_ok ? __float_as_uint(o) : 0u;  // o >= 0 (ReLU): the bit pattern orders like the value
      if (warp_one_group) {
        const unsigned mx = __reduce_max_sync(0xffffffffu, bits);
        if ((tid & 31) == 0) atomicMax(crow + col, mx);
      } else if (row_ok) {
        atomicMax(crow + col, bits);
      }
    };
    for (int c0 = kh * 16; c0 < ncols; c0 += 32) {          // the two warps of a lane quarter interleave 16-column blocks
      float v[16];
      tmem_ld16(trow + c0, v);                              // warp-collective: the control flow below stays warp-uniform
      for (int sl = 1; sl <= nsl; ++sl) {                   // split accumulators: the other hi*hi slices, the corrections
        float u[16];
        tmem_ld16(trow + sl * p.nr + c0, u);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] += u[j];
      }
      if (vec && c0 + 16 <= ncols) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 sc = *reinterpret_cast<const float4*>(s_osc + c0 + j), bb = *reinterpret_cast<const float4*>(s_bias + c0 + j);
          float4 o = make_float4(fmaf(v[j] * inv_a, sc.x, bb.x), fmaf(v[j + 1] * inv_a, sc.y, bb.y),
                                 fmaf(v[j + 2] * inv_a, sc.z, bb.z), fmaf(v[j + 3] * inv_a, sc.w, bb.w));
          if (row_ok) {
            if (arow2) { const float4 a = *reinterpret_cast<const float4*>(arow2 + c0 + j); o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w; }
            if (rrow) { const float4 r = __ldg(reinterpret_cast<const float4*>(rrow + c0 + j)); o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w; }
          }
          if (p.act == kActRelu6) { o.x = relu6f(o.x); o.y = relu6f(o.y); o.z = relu6f(o.z); o.w = relu6f(o.w); }
          else if (p.act == kActRelu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
          if (row_ok) {
            rmax = fmaxf(rmax, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
            if (orow) *reinterpret_cast<float4*>(orow + c0 + j) = o;
          }
          if (crow) { pool_max(c0 + j, o.x); pool_max(c0 + j + 1, o.y); pool_max(c0 + j + 2, o.z); pool_max(c0 + j + 3, o.w); }
        }
        continue;
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        if (c0 + j >= ncols) break;                          // warp-uniform
        float o = fmaf(v[j] * inv_a, s_osc[c0 + j], s_bias[c0 + j]);
        if (row_ok) {
          if (arow2) o += arow2[c0 + j];
          if (rrow) o += rrow[c0 + j];
        }
        if (p.act == kActRelu6) o = relu6f(o); else if (p.act == kActRelu) o = fmaxf(o, 0.f);
        if (row_ok) {
          rmax = fmaxf(rmax, fabsf(o));
          if (orow) orow[c0 + j] = o;
        }
        if (crow) pool_max(c0 + j, o);
      }
    }
    if (row_ok && p.rowmax_out != nullptr) atomicMax(p.rowmax_out + m, __float_as_uint(rmax));
  } else {
    // ------------------------------ weight loader + MMA issuer (converged warp) -------------------
    const uint32_t idesc = make_idesc_f16(128, p.nr);
    const uint32_t lbo_b = (uint32_t)(p.nr >> 3) * 128;
    const uint32_t d_hi = smem_desc_hi(128);
    auto load_w = [&](int c) {                                // weight chunk c -> its ring slot (slot known to be free)
      const int s = c % kGmStages, k0 = c * kGmKC;
      const int kc = min(kGmKC, p.Kp - k0);
      if (elect_one()) {
        const uint32_t plane_bytes = (uint32_t)p.nr * kc * 2;
        const uint8_t* src = wimg + (size_t)p.nr * k0 * 4;    // chunks of this range are consecutive
        mbar_expect_tx(smem_u32(&bar_full[s]), 2 * plane_bytes);
        bulk_g2s(smem_u32(stage_b(s, 0)), src, plane_bytes, smem_u32(&bar_full[s]));
        bulk_g2s(smem_u32(stage_b(s, 1)), src + plane_bytes, plane_bytes, smem_u32(&bar_full[s]));
      }
      __syncwarp();
    };
    for (int c = 0; c < min(nchunks, kGmStages); ++c) load_w(c);      // the first use of every slot needs no wait
    for (int c = 0; c < nchunks; ++c) {
      const int s = c % kGmStages, use = c / kGmStages;
      const int kc = min(kGmKC, p.Kp - c * kGmKC);
      mbar_wait(smem_u32(&bar_full[s]), use & 1, p.err);
      tc_fence_after_sync();
      const uint32_t a_lo = smem_desc_lo(smem_u32(stage_a(s, 0)), 2048);
      const uint32_t b_lo = smem_desc_lo(smem_u32(stage_b(s, 0)), lbo_b);
      if (elect_one()) {
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {                 // hi*hi, hi*lo, lo*hi
          const uint32_t a_off = (pass == 2 ? kGmStageA : 0), b_off = (pass == 1 ? kGmStageB : 0);
          uint32_t d = tmem, acc = (c > 0 || pass > 0) ? 1u : 0u;
          if (nsl > 0) {                                       // split accumulators (see GemmArgs::acc_slices)
            const int sl = pass == 0 ? c % nsl : nsl;
            d = tmem + (uint32_t)(sl * p.nr);
            acc = (pass == 0 ? c >= nsl : (c > 0 || pass > 1)) ? 1u : 0u;
          }
          for (int ks = 0; ks < kc / 16; ++ks)
            umma_f16(d, desc64(d_hi, a_lo + ((a_off + ks * 4096) >> 4)), desc64(d_hi, b_lo + ((b_off + ks * 2 * lbo_b) >> 4)),
                     idesc, (acc || ks > 0) ? 1u : 0u);
        }
        umma_commit(smem_u32(&bar_empty[s]));
        if (c == nchunks - 1) umma_commit(smem_u32(&bar_acc));
      }
      __syncwarp();
      // refill the slot of chunk c - 1 (its MMAs were committed one iteration ago) with chunk c - 1 + stages
      if (c >= 1 && c - 1 + kGmStages < nchunks) {
        const int cp = c - 1, sp = cp % kGmStages;
        mbar_wait(smem_u32(&bar_empty[sp]), (uint32_t)(cp / kGmStages) & 1, p.err);
        load_w(cp + kGmStages);
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kGmProducerWarps) {
    __syncwarp();
    if (p.acc_slices > 0) tmem_dealloc<512>(tmem);
    else tmem_dealloc<256>(tmem);
  }
}

// ---- small CUDA-core helpers of the same layer families ---------------------------------------------------------
// K < 8 first layer (PointNet conv1: 3 -> 64 on the landmark coordinates): out[m, n] = act(sum_k A[m,k] W[k,n] + b[n]).
// A is read through (row stride, element stride) so that the (B,3,68) landmark tensor is consumed in place:
// row m = (b, point) reads x[b, k, point].
__global__ void small_k_layer_kernel(const float* __restrict__ x, const float* __restrict__ Wkn, const float* __restrict__ bias,
                                     float* __restrict__ out, unsigned* __restrict__ rowmax_out, int M, int K, int N, int pts,
                                     int act) {
  const int m = blockIdx.x * blockDim.y + threadIdx.y;
  if (m >= M) return;
  const int b = m / pts, pt = m - b * pts;
  float a[8];
  for (int k = 0; k < K; ++k) a[k] = x[((size_t)b * K + k) * pts + pt];
  float rmax = 0.f;
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float o = bias[n];
    for (int k = 0; k < K; ++k) o = fmaf(a[k], Wkn[k * N + n], o);
    if (act == kActRelu) o = fmaxf(o, 0.f);
    out[(size_t)m * N + n] = o;
    rmax = fmaxf(rmax, fabsf(o));
  }
  for (int o = 16; o > 0; o >>= 1) rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
  if (threadIdx.x == 0 && rowmax_out != nullptr) rowmax_out[m] = __float_as_uint(rmax);
}

// rowmax of an arbitrary [M][K] fp32 matrix (inputs that no GEMM epilogue produced)
__global__ void rowmax_kernel(const float* __restrict__ A, unsigned* __restrict__ rowmax, int M, int K, int lda) {
  const int m = blockIdx.x * blockDim.y + threadIdx.y;
  if (m >= M) return;
  float r = 0.f;
  for (int k = threadIdx.x; k < K; k += 32) r = fmaxf(r, fabsf(A[(size_t)m * lda + k]));
  for (int o = 16; o > 0; o >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, o));
  if (threadIdx.x == 0) rowmax[m] = __float_as_uint(r);
}

}  // namespace syn
