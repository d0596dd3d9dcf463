// C-ABI implementation of the SynergyNet inference hot path for B200 (sm_100a).
// See include/synergy_b200.h for the contract and the reference lines each entry replaces.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_fused.cuh"
#include "kernels_tail.cuh"
#include "kernels_dense.cuh"
#include "kernels_gemm.cuh"
#include "kernels_loss.cuh"
#include "kernels_resnet.cuh"
#include "kernels_resnest.cuh"

using namespace syn;

namespace {

struct HostConv {
  std::vector<float> w, g, b, m, v;
  float eps = 1e-5f;
  bool set = false;
};

struct DevConv {
  float* w = nullptr;     // SIMT layout (stem [27][32], pointwise [K][N], depthwise [9][C])
  float* bias = nullptr;  // folded BN bias
};

}  // namespace

struct syn_heads;       // PointNet refinement heads (heads_host.inl)
void syn_heads_destroy(syn_heads* s);
struct syn_resnet;      // ResNet-50 backbone variant (resnet_host.inl)
void syn_resnet_destroy(syn_resnet* s);
struct syn_resnest;     // ResNeSt-50 backbone variant (resnest_host.inl)
void syn_resnest_destroy(syn_resnest* s);

struct syn_handle {
  int device = 0;
  syn_heads* heads = nullptr;
  syn_resnet* resnet = nullptr;
  syn_resnest* resnest = nullptr;
  int sm_count = 0;
  int engine = SYN_ENGINE_TC_FUSED;            // default: fused tcgen05 engine; 0/1 remain for cross-checks
  int center_crop = 0;                         // CenterCrop margin applied by the uint8 entry points (syn_set_center_crop)
  int npass() const { return engine == SYN_ENGINE_TC_FUSED_1PASS ? 1 : 3; }
  bool fused() const { return engine == SYN_ENGINE_TC_FUSED || engine == SYN_ENGINE_TC_FUSED_1PASS; }
  bool committed = false;
  int64_t launches = 0;
  // optional per-launch timing (syn_set_timing): events recorded after every kernel of a call
  bool timing = false;
  std::vector<cudaEvent_t> tev;
  std::vector<const char*> tname;
  int tn = 0;

  HostConv hconv[kNumConv];
  std::vector<float> h_head_w, h_head_b;       // (62,1280), (62)
  std::vector<float> h_mean, h_std;            // 62 each
  std::vector<float> h_sparse;                 // planar [51][3][sp_pad]
  std::vector<float> h_dense;                  // planar [51][3][dn_pad]
  int n_pts = 0, sp_pad = 0;
  int64_t n_vert = 0, dn_pad = 0;
  bool heads_set = false, whiten_set = false, sparse_dirty = false, dense_dirty = false;

  // device-side constants
  float* d_weights = nullptr;                  // one slab for all conv weights + biases
  DevConv dconv[kNumConv];
  float *d_head_w = nullptr, *d_head_b = nullptr, *d_mean = nullptr, *d_std = nullptr;
  float *d_sparse = nullptr, *d_dense = nullptr;

  // tensor-core engine: bf16 hi/lo weight images of the pointwise convs (kernels_tc.cuh)
  uint8_t* d_tcw = nullptr;
  float* d_tc_oscale = nullptr;                // per layer, per output channel: 1/(kActScale*weight scale)
  size_t tc_osc_off[kNumConv] = {};
  size_t tc_off[kNumConv] = {};
  int tc_nr[kNumConv] = {}, tc_nranges[kNumConv] = {}, tc_kp[kNumConv] = {};
  int* d_err = nullptr;                        // raised by a bounded mbarrier wait that timed out: mapped pinned HOST memory,
                                               // so every entry point can look at it without synchronising the device
  int* d_sat = nullptr;                        // device flag: a block input left the fp16 range of the split engines and was clamped
  bool tc_ready = false;
  // fused stem+block1 and blocks 2..7 (kernels_fused.cuh): one weight image per fused launch
  uint8_t* d_fused = nullptr;
  size_t fused_off[18] = {};                   // index = features[] index of the block (1..17)
  uint8_t* d_tail_w = nullptr;                 // kernels_tail.cuh weight image (10 x 160 KB)
  float* d_tail_osc = nullptr;                 // 1280 epilogue scales
  float* d_pool_tmp = nullptr;                 // (ws_batch, 1280) pooled features
  // tensor-core reconstruction (kernels_dense.cuh): fp16 hi/lo basis images + per-row meta
  uint8_t *d_sp_img = nullptr, *d_dn_img = nullptr;
  float *d_sp_meta = nullptr, *d_dn_meta = nullptr, *d_ascale = nullptr;
  int sp_vtiles = 0, dn_vtiles = 0;
  uint8_t* d_alpha_img = nullptr;              // recon workspace: alpha tiles + pose rows
  float* d_pose = nullptr;
  int recon_ftiles = 0;
  float* d_x_f32 = nullptr;                    // (ws_batch,3,120,120) normalised crops for engines 0/1 fed with uint8
  int x_f32_batch = 0;
  uint8_t* d_stage_u8[2] = {nullptr, nullptr};
  int stage_u8_chunk = 0;

  // activation workspace (NHWC fp32), grown on demand
  int ws_batch = 0;
  float *buf_io[2] = {nullptr, nullptr}, *buf_hid = nullptr, *buf_dw = nullptr;
  float* d_params_tmp = nullptr;               // (ws_batch, 62) for the fused landmark call

  // host-buffer pipeline
  cudaStream_t s_copy = nullptr, s_compute = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  float* d_stage_x[2] = {nullptr, nullptr};
  float* d_stage_lmk = nullptr;
  float* d_stage_par = nullptr;
  int stage_chunk = 0, stage_batch = 0;
  int host_slot = 0;                             // staging buffer of the next chunk (persists across calls)
  unsigned long long host_chunks = 0;            // chunks issued so far
  unsigned long long host_calls = 0;             // submitted host calls = next ticket
  cudaEvent_t ev_call[2] = {nullptr, nullptr};   // results of ticket t are on the host once ev_call[t & 1] has fired
};

namespace {

// per-face activation element counts (floats) of the four workspace buffers
constexpr size_t kIoPerFace = 60 * 60 * 32;       // stem output is the largest block in/out
constexpr size_t kHidPerFace = 60 * 60 * 96;      // block 2 expand output
constexpr size_t kDwPerFace = 30 * 30 * 144;      // block 3 depthwise output (> 60*60*32)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    int cur;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// count a launch and, when timing is on, drop an event behind it
void mark(syn_handle* h, cudaStream_t st, const char* name) {
  h->launches++;
  if (!h->timing) return;
  if (h->tn >= (int)h->tev.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    h->tev.push_back(e);
    h->tname.push_back(name);
  }
  h->tname[h->tn] = name;
  cudaEventRecord(h->tev[h->tn++], st);
}

int ensure_workspace(syn_handle* h, int batch) {
  if (batch <= h->ws_batch) return SYN_OK;
  SYN_CUDA(cudaDeviceSynchronize());
  cudaFree(h->buf_io[0]); cudaFree(h->buf_io[1]); cudaFree(h->buf_hid); cudaFree(h->buf_dw);
  cudaFree(h->d_params_tmp); cudaFree(h->d_pool_tmp);
  h->buf_io[0] = h->buf_io[1] = h->buf_hid = h->buf_dw = h->d_params_tmp = h->d_pool_tmp = nullptr;
  h->ws_batch = 0;
  const size_t b = (size_t)batch;
  SYN_CUDA(cudaMalloc(&h->buf_io[0], b * kIoPerFace * sizeof(float)));
  SYN_CUDA(cudaMalloc(&h->buf_io[1], b * kIoPerFace * sizeof(float)));
  SYN_CUDA(cudaMalloc(&h->buf_hid, b * kHidPerFace * sizeof(float)));
  SYN_CUDA(cudaMalloc(&h->buf_dw, b * kDwPerFace * sizeof(float)));
  SYN_CUDA(cudaMalloc(&h->d_params_tmp, b * kNumParams * sizeof(float)));
  SYN_CUDA(cudaMalloc(&h->d_pool_tmp, b * kLastCh * sizeof(float)));
  h->ws_batch = batch;
  return SYN_OK;
}

// ---- launches -------------------------------------------------------------------------------
int launch_pointwise_simt(syn_handle* h, const float* A, const DevConv& w, const float* residual,
                          float* out, int M, int K, int N, int relu6, cudaStream_t st) {
  if (N >= 64) {
    dim3 grid((M + 127) / 128, (N + 63) / 64);
    pointwise_gemm_kernel<128, 64, 8, 4><<<grid, 256, 0, st>>>(A, w.w, w.bias, residual, out, M, K, N, relu6);
  } else if (N > 16) {
    dim3 grid((M + 127) / 128, (N + 31) / 32);
    pointwise_gemm_kernel<128, 32, 4, 4><<<grid, 256, 0, st>>>(A, w.w, w.bias, residual, out, M, K, N, relu6);
  } else {
    dim3 grid((M + 255) / 256, (N + 15) / 16);
    pointwise_gemm_kernel<256, 16, 4, 4><<<grid, 256, 0, st>>>(A, w.w, w.bias, residual, out, M, K, N, relu6);
  }
  SYN_LAUNCH_CHECK("pointwise_gemm_kernel");
  mark(h, st, "pointwise_gemm_kernel");
  return SYN_OK;
}

int launch_pointwise_tc(syn_handle* h, const float* A, int layer, const float* residual, float* out,
                        int M, cudaStream_t st) {
  const ConvDesc& c = plan().conv[layer];
  TcPointwiseArgs a;
  a.A = A; a.Wimg = h->d_tcw + h->tc_off[layer]; a.bias = h->dconv[layer].bias; a.oscale = h->d_tc_oscale + h->tc_osc_off[layer]; a.residual = residual;
  a.out = out; a.M = M; a.K = c.cin; a.N = c.cout; a.Kp = h->tc_kp[layer]; a.nr = h->tc_nr[layer];
  a.relu6 = c.relu6; a.err = h->d_err;
  dim3 grid((M + 127) / 128, h->tc_nranges[layer]);
  tc_pointwise_kernel<<<grid, kTcThreads, kTcSmemBytes, st>>>(a);
  SYN_LAUNCH_CHECK("tc_pointwise_kernel");
  mark(h, st, "tc_pointwise_kernel");
  return SYN_OK;
}

int launch_pointwise(syn_handle* h, const float* A, int layer, const float* residual, float* out,
                     int M, cudaStream_t st) {
  const ConvDesc& c = plan().conv[layer];
  if (h->engine != SYN_ENGINE_SIMT_FP32) return launch_pointwise_tc(h, A, layer, residual, out, M, st);
  return launch_pointwise_simt(h, A, h->dconv[layer], residual, out, M, c.cin, c.cout, c.relu6, st);
}

int launch_depthwise(syn_handle* h, const float* x, int layer, float* y, int batch, cudaStream_t st) {
  const ConvDesc& c = plan().conv[layer];
  const size_t total = (size_t)batch * c.h_out * c.h_out * (c.cout / 4);
  const unsigned grid = (unsigned)((total + 255) / 256);
  depthwise3x3_kernel<<<grid, 256, 0, st>>>(x, h->dconv[layer].w, h->dconv[layer].bias, y, batch,
                                           c.cout, c.h_in, c.h_out, c.stride);
  SYN_LAUNCH_CHECK("depthwise3x3_kernel");
  mark(h, st, "depthwise3x3_kernel");
  return SYN_OK;
}

template <class C>
int launch_fused(syn_handle* h, const float* x, int block, float* y, int batch, cudaStream_t st,
                 const uint8_t* x_u8 = nullptr);

// Runs the backbone.  When stop_layer >= 0 the activation of that conv is copied to dbg_out and
// the function returns early.  Otherwise params (B,62) [and pool (B,1280)] are produced.
int run_backbone(syn_handle* h, const float* x, int batch, float* params, float* pool,
                 int stop_layer, float* dbg_out, cudaStream_t st, const uint8_t* x_u8 = nullptr) {
  const Plan& P = plan();
  int rc = ensure_workspace(h, batch);
  if (rc != SYN_OK) return rc;
  if (x_u8 != nullptr && !h->fused()) {
    // engines whose stem reads fp32: normalise into a scratch buffer first
    if (batch > h->x_f32_batch) {
      SYN_CUDA(cudaDeviceSynchronize());
      cudaFree(h->d_x_f32);
      h->d_x_f32 = nullptr;
      h->x_f32_batch = 0;
      SYN_CUDA(cudaMalloc(&h->d_x_f32, (size_t)batch * 3 * kImg * kImg * sizeof(float)));
      h->x_f32_batch = batch;
    }
    const size_t n4 = (size_t)batch * 3 * kImg * kImg / 4;
    normalize_u8_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(x_u8, h->d_x_f32, n4, h->center_crop);
    SYN_LAUNCH_CHECK("normalize_u8_kernel");
    mark(h, st, "normalize_u8_kernel");
    x = h->d_x_f32;
    x_u8 = nullptr;
  }

  auto dbg = [&](int layer, const float* buf) -> int {
    const ConvDesc& c = P.conv[layer];
    const size_t n = (size_t)batch * c.h_out * c.h_out * c.cout;
    SYN_CUDA(cudaMemcpyAsync(dbg_out, buf, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return SYN_OK;
  };

  int cur = 0;
  int li = 1;
  if (h->fused()) {
    // stem + block 1, then blocks 2..7, each one fused launch; only block outputs exist
    if (stop_layer >= 0 && stop_layer <= 50 && (stop_layer < 2 || (stop_layer - 2) % 3 != 0))
      return fail(SYN_ERR_UNSUPPORTED, "conv %d lives inside a fused block and is never materialised", stop_layer);
    const float* in = x;
    for (int b = 1; b <= 17; ++b) {
      float* out = h->buf_io[cur ^ 1];
      switch (b) {
        case 1: rc = launch_fused<FusedStemB1>(h, in, b, out, batch, st, x_u8); break;
        case 2: rc = launch_fused<FusedB2>(h, in, b, out, batch, st); break;
        case 3: rc = launch_fused<FusedB3>(h, in, b, out, batch, st); break;
        case 4: rc = launch_fused<FusedB4>(h, in, b, out, batch, st); break;
        case 5: case 6: rc = launch_fused<FusedB56>(h, in, b, out, batch, st); break;
        case 7: rc = launch_fused<FusedB7>(h, in, b, out, batch, st); break;
        case 8: case 9: case 10: rc = launch_fused<FusedB8>(h, in, b, out, batch, st); break;
        case 11: rc = launch_fused<FusedB11>(h, in, b, out, batch, st); break;
        case 12: case 13: rc = launch_fused<FusedB12>(h, in, b, out, batch, st); break;
        case 14: rc = launch_fused<FusedB14>(h, in, b, out, batch, st); break;
        case 15: case 16: rc = launch_fused<FusedB15>(h, in, b, out, batch, st); break;
        default: rc = launch_fused<FusedB17>(h, in, b, out, batch, st); break;
      }
      if (rc != SYN_OK) return rc;
      cur ^= 1;
      in = h->buf_io[cur];
      if (stop_layer == 3 * b - 1) return dbg(3 * b - 1, h->buf_io[cur]);
    }
    if (stop_layer == 51)
      return fail(SYN_ERR_UNSUPPORTED, "conv 51 is fused with the average pool and never materialised");
    {
      float* pooled = pool ? pool : h->d_pool_tmp;
      TailArgs t;
      t.x = h->buf_io[cur]; t.wimg = h->d_tail_w; t.bias = h->dconv[51].bias; t.oscale = h->d_tail_osc;
      t.pooled = pooled; t.batch = batch; t.err = h->d_err; t.npass = h->npass();
      const int ntiles = (batch + kTailFaces - 1) / kTailFaces;
      t.ctas_per_slice = std::max(1, std::min(ntiles, h->sm_count / 10));
      tail_conv_pool_kernel<<<10 * t.ctas_per_slice, kTailThreads, kTailSmem, st>>>(t);
      SYN_LAUNCH_CHECK("tail_conv_pool_kernel");
      mark(h, st, "tail_conv_pool_kernel");
      heads_kernel<<<dim3((batch + 7) / 8, 2), 256, 0, st>>>(pooled, h->d_head_w, h->d_head_b, params, batch);
      SYN_LAUNCH_CHECK("heads_kernel");
      mark(h, st, "heads_kernel");
      return SYN_OK;
    }
  } else {
  stem_conv3x3s2_kernel<true><<<batch * 60, kStemThreads, 0, st>>>(x, h->dconv[0].w, h->dconv[0].bias,
                                                                  h->buf_io[cur], batch, nullptr);
  SYN_LAUNCH_CHECK("stem_conv3x3s2_kernel");
  mark(h, st, "stem_conv3x3s2_kernel");
  if (stop_layer == 0) return dbg(0, h->buf_io[cur]);
  }

  while (P.conv[li].kind != kLast) {
    const float* block_in = h->buf_io[cur];
    const float* dw_in = block_in;
    if (P.conv[li].kind == kExpand) {
      const ConvDesc& e = P.conv[li];
      rc = launch_pointwise(h, block_in, li, nullptr, h->buf_hid, batch * e.h_in * e.h_in, st);
      if (rc != SYN_OK) return rc;
      if (stop_layer == li) return dbg(li, h->buf_hid);
      dw_in = h->buf_hid;
      ++li;
    }
    rc = launch_depthwise(h, dw_in, li, h->buf_dw, batch, st);
    if (rc != SYN_OK) return rc;
    if (stop_layer == li) return dbg(li, h->buf_dw);
    ++li;
    const ConvDesc& p = P.conv[li];
    rc = launch_pointwise(h, h->buf_dw, li, p.residual ? block_in : nullptr, h->buf_io[cur ^ 1],
                          batch * p.h_out * p.h_out, st);
    if (rc != SYN_OK) return rc;
    cur ^= 1;
    if (stop_layer == li) return dbg(li, h->buf_io[cur]);
    ++li;
  }
  const ConvDesc& last = P.conv[li];
  rc = launch_pointwise(h, h->buf_io[cur], li, nullptr, h->buf_hid, batch * last.h_in * last.h_in, st);
  if (rc != SYN_OK) return rc;
  if (stop_layer == li) return dbg(li, h->buf_hid);

  pool_heads_kernel<<<batch, 256, 0, st>>>(h->buf_hid, h->d_head_w, h->d_head_b, params, pool,
                                          last.h_out * last.h_out);
  SYN_LAUNCH_CHECK("pool_heads_kernel");
  mark(h, st, "pool_heads_kernel");
  return SYN_OK;
}

// Reconstruction kernels are launched with programmatic stream serialization: they start while dense_alpha_kernel
// (which signals griddepcontrol.launch_dependents at its top) is still running, set up barriers / TMEM, stream in
// basis data, and execute griddepcontrol.wait before the first access to the pre-pass' output.
static cudaError_t launch_after_prepass(void (*kernel)(DenseArgs), int grid, int smem, cudaStream_t st, const DenseArgs& a) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kDnThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, a);
}

int run_reconstruct_tc(syn_handle* h, const float* params, int batch, int dense, int whitening, int transform,
                       float* out, cudaStream_t st, const float* roi5 = nullptr) {
  const int n_ftiles = (batch + kDnFaces - 1) / kDnFaces;
  if (n_ftiles > h->recon_ftiles) {
    SYN_CUDA(cudaDeviceSynchronize());
    cudaFree(h->d_alpha_img); cudaFree(h->d_pose);
    h->d_alpha_img = nullptr; h->d_pose = nullptr; h->recon_ftiles = 0;
    SYN_CUDA(cudaMalloc(&h->d_alpha_img, (size_t)n_ftiles * kDnBTile));
    SYN_CUDA(cudaMalloc(&h->d_pose, (size_t)n_ftiles * kDnPoseTile));
    h->recon_ftiles = n_ftiles;
  }
  dense_alpha_kernel<<<n_ftiles, kDnAlphaThreads, 0, st>>>(params, h->d_mean, h->d_std, h->d_ascale, h->d_alpha_img, h->d_pose, batch,
                                             whitening, roi5);
  SYN_LAUNCH_CHECK("dense_alpha_kernel");
  mark(h, st, "dense_alpha_kernel");
  DenseArgs a;
  a.basis_img = dense ? h->d_dn_img : h->d_sp_img;
  a.meta = dense ? h->d_dn_meta : h->d_sp_meta;
  a.alpha_img = h->d_alpha_img; a.pose = h->d_pose; a.out = out; a.batch = batch;
  a.nver = dense ? (int)h->n_vert : h->n_pts;
  a.n_vtiles = dense ? h->dn_vtiles : h->sp_vtiles;
  a.n_ftiles = n_ftiles; a.transform = transform; a.affine = roi5 != nullptr; a.err = h->d_err;
  const int items = a.n_vtiles * a.n_ftiles;
  // dense mesh: face-major walk with streamed basis planes (long contiguous output runs per CTA); the 68-landmark
  // basis is one vertex tile, where the two kernels do the same work -- keep the simpler one there.
  static const bool fm_off = getenv("SYN_DENSE_VERTEX_MAJOR") != nullptr;      // A/B switches for measurements
  static const bool wb_stores = getenv("SYN_DENSE_WB_STORES") != nullptr;
  a.stream_stores = wb_stores ? 0 : 1;
  a.trace = nullptr;
  static long long* d_dense_trace = nullptr;                                   // debug: SYN_DENSE_TRACE=file dumps CTA 0's timeline
  static const char* trace_fp = getenv("SYN_DENSE_TRACE");
  if (trace_fp != nullptr && dense) {
    if (d_dense_trace == nullptr) cudaMalloc(&d_dense_trace, 192 * 8 * sizeof(long long));
    cudaMemsetAsync(d_dense_trace, 0, 192 * 8 * sizeof(long long), st);
    a.trace = d_dense_trace;
  }
  if (dense && !fm_off) {
    // grid = face tiles x vertex bands (see the kernel): as many whole bands as fit the SMs
    const int n_bands = std::max(1, h->sm_count / a.n_ftiles);
    const int grid = a.n_ftiles * std::min(n_bands, a.n_vtiles);
    if (a.trace != nullptr) SYN_CUDA(launch_after_prepass(dense_recon_fm_kernel<true, true>, grid, kFmSmem, st, a));
    else if (a.affine) SYN_CUDA(launch_after_prepass(dense_recon_fm_kernel<false, true>, grid, kFmSmem, st, a));
    else SYN_CUDA(launch_after_prepass(dense_recon_fm_kernel<false, false>, grid, kFmSmem, st, a));
    SYN_LAUNCH_CHECK("dense_recon_fm_kernel");
    mark(h, st, "dense_recon_fm_kernel");
    if (a.trace != nullptr) {                                                  // debug only: synchronous dump
      std::vector<long long> t(192 * 8);
      cudaStreamSynchronize(st);
      cudaMemcpy(t.data(), a.trace, t.size() * sizeof(long long), cudaMemcpyDeviceToHost);
      if (FILE* f = fopen(trace_fp, "w")) {
        for (int r = 0; r < 192; ++r) {
          fprintf(f, "%s %d", r < 64 ? "epi0" : r < 128 ? "epi1" : "issuer", r & 63);
          for (int e = 0; e < 8; ++e) fprintf(f, " %lld", t[r * 8 + e]);
          fprintf(f, "\n");
        }
        fclose(f);
      }
    }
    return SYN_OK;
  }
  SYN_CUDA(launch_after_prepass(dense_recon_tc_kernel, std::min(items, h->sm_count), kDnSmem, st, a));
  SYN_LAUNCH_CHECK("dense_recon_tc_kernel");
  mark(h, st, "dense_recon_tc_kernel");
  return SYN_OK;
}

int run_reconstruct(syn_handle* h, const float* params, int batch, int dense, int whitening,
                    int transform, float* out, cudaStream_t st, const float* roi5 = nullptr) {
  if (dense && h->d_dense == nullptr) return fail(SYN_ERR_STATE, "dense basis not set (syn_set_basis_dense)");
  if (!dense && h->d_sparse == nullptr) return fail(SYN_ERR_STATE, "sparse basis not set (syn_set_basis_sparse)");
  if (h->engine != SYN_ENGINE_SIMT_FP32 || roi5 != nullptr)     // the image-space variant exists on the tensor-core kernels only
    return run_reconstruct_tc(h, params, batch, dense, whitening, transform, out, st, roi5);
  if (dense) {
    constexpr int F = 16;
    dim3 grid((unsigned)(h->dn_pad / 128), (batch + F - 1) / F);
    reconstruct_kernel<F><<<grid, 128, 0, st>>>(h->d_dense, params, h->d_mean, h->d_std, out, batch,
                                               (int)h->n_vert, (int)h->dn_pad, whitening, transform);
  } else {
    constexpr int F = 8;
    dim3 grid(h->sp_pad / 128, (batch + F - 1) / F);
    reconstruct_kernel<F><<<grid, 128, 0, st>>>(h->d_sparse, params, h->d_mean, h->d_std, out, batch,
                                               h->n_pts, h->sp_pad, whitening, transform);
  }
  SYN_LAUNCH_CHECK("reconstruct_kernel");
  mark(h, st, "reconstruct_kernel");
  return SYN_OK;
}

// ---- fp16 hi/lo weight images for the tensor-core kernels -------------------------------------------
inline void split_f16_host(float x, uint16_t& hi, uint16_t& lo) {
  const __half h = __float2half_rn(x);
  const __half l = __float2half_rn(x - __half2float(h));
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(l);
}
// power-of-two scale that brings max|w| of one output channel into [256, 512) (tc_common.cuh)
inline float channel_scale(const float* w, size_t stride, int count) {
  float m = 0.f;
  for (int i = 0; i < count; ++i) m = std::max(m, fabsf(w[(size_t)i * stride]));
  if (!(m > 0.f) || !std::isfinite(m)) return 1.f;
  int ex;
  frexpf(m, &ex);                       // m = f * 2^ex, f in [0.5, 1)
  return ldexpf(1.f, 9 - ex);
}
constexpr float kActScaleHost = 64.0f;   // == tc::kActScale

// Wkn: folded weights [K][N] fp32 (SIMT layout).  Image: for each n-range, for each K-chunk of 64:
// hi plane [nr x kc] then lo plane, canonical K-major no-swizzle (SBO = 128, LBO = nr/8*128).
// oscale[n] receives the epilogue multiplier that undoes the activation and weight scales.
void pack_tc_pointwise(std::vector<uint8_t>& img, std::vector<float>& oscale, const float* Wkn, int K, int N,
                       int Kp, int nr, int nranges) {
  img.assign((size_t)nranges * nr * Kp * 4, 0);
  oscale.assign((size_t)nranges * nr, 0.f);
  uint16_t* base = reinterpret_cast<uint16_t*>(img.data());
  const size_t lbo = (size_t)(nr / 8) * 128;
  std::vector<float> ws(N);
  for (int n = 0; n < N; ++n) {
    ws[n] = channel_scale(Wkn + n, (size_t)N, K);
    oscale[n] = 1.0f / (kActScaleHost * ws[n]);
  }
  for (int j = 0; j < nranges; ++j)
    for (int k0 = 0; k0 < Kp; k0 += kTcKChunk) {
      const int kc = std::min(kTcKChunk, Kp - k0);
      uint16_t* hi = base + ((size_t)j * nr * Kp * 4 + (size_t)nr * k0 * 4) / 2;
      uint16_t* lo = hi + (size_t)nr * kc;
      for (int nl = 0; nl < nr; ++nl) {
        const int n = j * nr + nl;
        if (n >= N) continue;
        for (int kl = 0; kl < kc; ++kl) {
          const int k = k0 + kl;
          if (k >= K) continue;
          const size_t off = ((size_t)(nl / 8) * 128 + (size_t)(kl / 8) * lbo + (nl % 8) * 16 + (kl % 8) * 2) / 2;
          split_f16_host(Wkn[(size_t)k * N + n] * ws[n], hi[off], lo[off]);
        }
      }
    }
}

// ---- weight image of one fused block (layout documented in FusedCfg) --------------------------------
// w1: [K][CHID] folded expand (or stem) weights, dw: [9][CHID], w3: [CHID][COUT] folded project weights.
template <class C>
void pack_fused(std::vector<uint8_t>& img, const float* w1, int K, const float* b1, const float* dw,
                const float* bdw, const float* w3, const float* b3) {
  img.assign(C::W_BYTES, 0);
  auto put = [&](size_t byte_off, float w, size_t plane_bytes) {
    uint16_t h, l;
    split_f16_host(w, h, l);
    *reinterpret_cast<uint16_t*>(img.data() + byte_off) = h;
    *reinterpret_cast<uint16_t*>(img.data() + byte_off + plane_bytes) = l;
  };
  float* b3p = reinterpret_cast<float*>(img.data());                   // [b3 | s3]
  std::vector<float> s3(C::COUT);
  for (int n = 0; n < C::COUT; ++n) {
    s3[n] = channel_scale(w3 + n, (size_t)C::COUT, C::CHID);
    b3p[n] = b3[n];
    b3p[C::COUT_P + n] = 1.0f / (kActScaleHost * s3[n]);
  }
  // one power-of-two scale for the whole expand layer (the kernel keeps it in a register): max |w1| in [256,512)
  const float s1 = channel_scale(w1, 1, K * C::CHID);
  for (int c = 0; c < C::NCHUNK; ++c) {
    const size_t chunk = C::B3_BYTES + (size_t)c * C::CHUNK_BYTES;
    float* d = reinterpret_cast<float*>(img.data() + chunk + C::CH_DW);
    for (int n = 0; n < C::NC; ++n) {
      const int ch = c * C::NC + n;
      for (int k = 0; k < K; ++k) {
        const size_t off = (size_t)(n / 8) * 128 + (size_t)(k / 8) * ((C::NC / 8) * 128) + (n % 8) * 16 + (k % 8) * 2;
        put(chunk + C::CH_W1 + off, w1[(size_t)k * C::CHID + ch] * s1, C::W1_PLANE);
      }
      for (int t = 0; t < 9; ++t) d[t * C::DWS + n] = dw[(size_t)t * C::CHID + ch];
      // the hidden activation is kept as relu6(h)/6 in [0,1] (kernels_fused.cuh): fold the 1/6 here
      d[9 * C::DWS + n] = bdw[ch] / 6.0f;
      d[10 * C::DWS + n] = b1[ch] / 6.0f;
      d[11 * C::DWS + n] = 1.0f / (6.0f * kActScaleHost * s1);
    }
    for (int n = 0; n < C::COUT; ++n)
      for (int k = 0; k < C::NC; ++k) {
        const size_t off = (size_t)(n / 8) * 128 + (size_t)(k / 8) * ((C::COUT_P / 8) * 128) + (n % 8) * 16 + (k % 8) * 2;
        put(chunk + C::CH_W3 + off, w3[(size_t)(c * C::NC + k) * C::COUT + n] * s3[n], C::W3_PLANE);
      }
  }
}

// Worker warps of the fused kernel: 16 by default (4 per SM sub-partition, measured best); SYN_FUSED_WARPS=8|12|16
// selects another instantiation for tuning runs.
inline int fused_worker_warps(int block) {
  static const struct Table {
    int v[18];
    Table() {
      const char* e = getenv("SYN_FUSED_WARPS");
      const int n = e ? atoi(e) : 16;
      const int all = (n == 8 || n == 12 || n == 16 || n == 20 || n == 24) ? n : 16;
      for (int i = 0; i < 18; ++i) v[i] = all;
      // per block: SYN_FUSED_WARPS_MAP="1:24,2:20" (tuning runs)
      const char* m = getenv("SYN_FUSED_WARPS_MAP");
      while (m && *m) {
        const int b = atoi(m);
        const char* c = strchr(m, ':');
        if (!c) break;
        const int w = atoi(c + 1);
        if (b >= 1 && b <= 17 && (w == 8 || w == 12 || w == 16 || w == 20 || w == 24)) v[b] = w;
        m = strchr(c, ',');
        if (m) ++m;
      }
    }
  } t;
  return t.v[block];
}

template <class C, int NWW>
int launch_fused_nww(syn_handle* h, const FusedArgs& a, int grid, cudaStream_t st) {
  static bool attr_set[16] = {};
  if (!attr_set[h->device & 15]) {
    SYN_CUDA(cudaFuncSetAttribute(fused_mbconv_kernel<C, NWW>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set[h->device & 15] = true;
    if (getenv("SYN_DEBUG_OCC") != nullptr) {
      int nb = -1;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fused_mbconv_kernel<C, NWW>, (NWW + 1) * 32, C::SMEM_BYTES);
      fprintf(stderr, "[syn] fused CIN=%d CHID=%d W=%d: %d worker warps, %d B smem, %d TMEM cols -> %d CTA(s)/SM\n",
              C::CIN, C::CHID, C::W, NWW, C::SMEM_BYTES, C::TM_COLS, nb);
    }
  }
#if SYN_PDL
  // programmatic dependent launch (experimental, see kernels_fused.cuh): the kernel may start while its
  // predecessor in the stream drains; it waits (griddepcontrol.wait) before touching the predecessor's output
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3((NWW + 1) * 32);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  SYN_CUDA(cudaLaunchKernelEx(&cfg, fused_mbconv_kernel<C, NWW>, a));
#else
  fused_mbconv_kernel<C, NWW><<<grid, (NWW + 1) * 32, C::SMEM_BYTES, st>>>(a);
#endif
  return SYN_OK;
}

template <class C>
int launch_fused(syn_handle* h, const float* x, int block, float* y, int batch, cudaStream_t st, const uint8_t* x_u8) {
  FusedArgs a;
  a.x_u8 = x_u8;
  a.x = x; a.wimg = h->d_fused + h->fused_off[block]; a.y = y; a.batch = batch; a.err = h->d_err; a.sat = h->d_sat; a.npass = h->npass(); a.border = h->center_crop;
#ifdef SYN_FUSED_TRACE
  a.trace_id = block;
#endif
  fused_tile_plan<C>(batch, h->sm_count, a.split, a.face_groups);
  const int ntiles = a.face_groups * C::STRIPS;
  const int grid = std::min(ntiles, h->sm_count);
  int rc;
  switch (fused_worker_warps(block)) {
    case 8: rc = launch_fused_nww<C, 8>(h, a, grid, st); break;
    case 12: rc = launch_fused_nww<C, 12>(h, a, grid, st); break;
#ifdef SYN_MORE_WARPS
    case 20: rc = launch_fused_nww<C, 20>(h, a, grid, st); break;
    case 24: rc = launch_fused_nww<C, 24>(h, a, grid, st); break;
#endif
    default: rc = launch_fused_nww<C, 16>(h, a, grid, st); break;
  }
  if (rc != SYN_OK) return rc;
  SYN_LAUNCH_CHECK("fused_mbconv_kernel");
  static const char* const names[18] = {"", "fused_stem_block1", "fused_block2", "fused_block3", "fused_block4",
                                        "fused_block5", "fused_block6", "fused_block7", "fused_block8", "fused_block9",
                                        "fused_block10", "fused_block11", "fused_block12", "fused_block13", "fused_block14",
                                        "fused_block15", "fused_block16", "fused_block17"};
  mark(h, st, names[block]);
  return SYN_OK;
}

// ---- tensor-core reconstruction images (kernels_dense.cuh) from the planar [51][3][pad] basis --------------
// alpha coefficient k is pre-multiplied by ascale[k] on the device, so column k of the basis is divided by it
// here (exact: powers of two); each (vertex, coordinate) row is then scaled into [256, 512).
void pack_recon_tc(std::vector<uint8_t>& img, std::vector<float>& meta, const std::vector<float>& planar, int64_t n,
                   int64_t pad, const float* ascale) {
  const int64_t vtiles = pad / 128;
  img.assign((size_t)vtiles * kDnATile, 0);
  meta.assign((size_t)vtiles * 6 * 128, 0.f);
  float row[kNumAlpha];
  for (int64_t vt = 0; vt < vtiles; ++vt)
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 128; ++r) {
        const int64_t v = vt * 128 + r;
        float* m = meta.data() + (size_t)vt * 6 * 128;
        m[(3 + c) * 128 + r] = 1.f;
        if (v >= n) continue;
        m[c * 128 + r] = planar[(size_t)(0 * 3 + c) * pad + v];
        for (int k = 0; k < kNumAlpha; ++k) row[k] = planar[(size_t)((1 + k) * 3 + c) * pad + v] / ascale[k];
        const float rs = channel_scale(row, 1, kNumAlpha);
        m[(3 + c) * 128 + r] = 1.0f / rs;
        uint8_t* base = img.data() + (size_t)vt * kDnATile + (size_t)(c * 2) * kDnAPlane;
        for (int k = 0; k < kNumAlpha; ++k) {
          const size_t off = (size_t)(r / 8) * 128 + (size_t)(k / 8) * 2048 + (r % 8) * 16 + (k % 8) * 2;
          uint16_t hi, lo;
          split_f16_host(row[k] * rs, hi, lo);
          *reinterpret_cast<uint16_t*>(base + off) = hi;
          *reinterpret_cast<uint16_t*>(base + kDnAPlane + off) = lo;
        }
      }
}

int upload_bytes(uint8_t** dptr, const std::vector<uint8_t>& src) {
  if (*dptr != nullptr) { cudaFree(*dptr); *dptr = nullptr; }
  SYN_CUDA(cudaMalloc(dptr, src.size()));
  SYN_CUDA(cudaMemcpy(*dptr, src.data(), src.size(), cudaMemcpyHostToDevice));
  return SYN_OK;
}

// planar [51][3][pad] from the reference's interleaved (3N,1)/(3N,40)/(3N,10) buffers
void pack_basis(std::vector<float>& dst, const float* u, const float* ws, const float* we, int64_t n,
                int64_t pad) {
  dst.assign((size_t)(kNumAlpha + 1) * 3 * pad, 0.f);
  for (int64_t v = 0; v < n; ++v)
    for (int c = 0; c < 3; ++c) {
      const int64_t row = 3 * v + c;
      dst[(size_t)(0 * 3 + c) * pad + v] = u[row];
      for (int k = 0; k < kNumShp; ++k) dst[(size_t)((1 + k) * 3 + c) * pad + v] = ws[row * kNumShp + k];
      for (int k = 0; k < kNumExp; ++k)
        dst[(size_t)((1 + kNumShp + k) * 3 + c) * pad + v] = we[row * kNumExp + k];
    }
}

int upload(float** dptr, const std::vector<float>& src) {
  if (*dptr != nullptr) { cudaFree(*dptr); *dptr = nullptr; }
  SYN_CUDA(cudaMalloc(dptr, src.size() * sizeof(float)));
  SYN_CUDA(cudaMemcpy(*dptr, src.data(), src.size() * sizeof(float), cudaMemcpyHostToDevice));
  return SYN_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int syn_abi_version(void) { return SYN_ABI_VERSION; }
const char* syn_last_error(void) { return last_error_buf(); }
int syn_num_conv_layers(void) { return kNumConv; }

int syn_conv_desc(int layer, syn_conv_desc_t* out) {
  if (layer < 0 || layer >= kNumConv || out == nullptr) return fail(SYN_ERR_INVALID, "syn_conv_desc: bad layer %d", layer);
  const ConvDesc& c = plan().conv[layer];
  out->cin = c.cin; out->cout = c.cout; out->ksize = c.ksize; out->stride = c.stride;
  out->groups = c.groups; out->relu6 = c.relu6; out->h_in = c.h_in; out->h_out = c.h_out;
  out->residual = c.residual;
  return SYN_OK;
}

int syn_create(int device, syn_handle_t** out) {
  if (out == nullptr) return fail(SYN_ERR_INVALID, "syn_create: out is null");
  *out = nullptr;
  int ndev = 0;
  SYN_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(SYN_ERR_INVALID, "syn_create: device %d of %d", device, ndev);
  cudaDeviceProp prop;
  SYN_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(SYN_ERR_UNSUPPORTED, "syn_create: device %d is sm_%d%d; this library is built for sm_100a only",
                device, prop.major, prop.minor);
  DeviceGuard g(device);
  if (!g.ok) return fail(SYN_ERR_CUDA, "syn_create: cannot select device %d", device);
  syn_handle* h = new (std::nothrow) syn_handle();
  if (h == nullptr) return fail(SYN_ERR_NOMEM, "syn_create: out of host memory");
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  SYN_CUDA(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
  SYN_CUDA(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    SYN_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
    SYN_CUDA(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
    SYN_CUDA(cudaEventCreateWithFlags(&h->ev_call[i], cudaEventDisableTiming));
  }
  *out = h;
  return SYN_OK;
}

void syn_destroy(syn_handle_t* h) {
  if (h == nullptr) return;
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  syn_heads_destroy(h->heads);
  syn_resnet_destroy(h->resnet);
  syn_resnest_destroy(h->resnest);
  cudaFree(h->d_weights); cudaFree(h->d_head_w); cudaFree(h->d_head_b); cudaFree(h->d_mean);
  cudaFree(h->d_std); cudaFree(h->d_sparse); cudaFree(h->d_dense); cudaFree(h->d_tcw); cudaFreeHost(h->d_err); cudaFree(h->d_sat); cudaFree(h->d_fused); cudaFree(h->d_tc_oscale);
  cudaFree(h->buf_io[0]); cudaFree(h->buf_io[1]); cudaFree(h->buf_hid); cudaFree(h->buf_dw);
  cudaFree(h->d_params_tmp); cudaFree(h->d_pool_tmp); cudaFree(h->d_tail_w); cudaFree(h->d_tail_osc); cudaFree(h->d_x_f32);
  cudaFree(h->d_sp_img); cudaFree(h->d_dn_img); cudaFree(h->d_sp_meta); cudaFree(h->d_dn_meta); cudaFree(h->d_ascale);
  cudaFree(h->d_alpha_img); cudaFree(h->d_pose);
  cudaFree(h->d_stage_u8[0]); cudaFree(h->d_stage_u8[1]);
  cudaFree(h->d_stage_x[0]); cudaFree(h->d_stage_x[1]); cudaFree(h->d_stage_lmk); cudaFree(h->d_stage_par);
  for (int i = 0; i < 2; ++i) {
    if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
    if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]);
    if (h->ev_call[i]) cudaEventDestroy(h->ev_call[i]);
  }
  for (cudaEvent_t e : h->tev) cudaEventDestroy(e);
  if (h->s_copy) cudaStreamDestroy(h->s_copy);
  if (h->s_compute) cudaStreamDestroy(h->s_compute);
  delete h;
}

int syn_set_conv_bn(syn_handle_t* h, int layer, const float* w, int64_t w_numel, const float* g,
                    const float* b, const float* m, const float* v, float eps) {
  if (h == nullptr || w == nullptr || g == nullptr || b == nullptr || m == nullptr || v == nullptr)
    return fail(SYN_ERR_INVALID, "syn_set_conv_bn: null argument");
  if (layer < 0 || layer >= kNumConv) return fail(SYN_ERR_INVALID, "syn_set_conv_bn: layer %d out of range", layer);
  const ConvDesc& c = plan().conv[layer];
  const int64_t expect = (int64_t)c.cout * (c.cin / c.groups) * c.ksize * c.ksize;
  if (w_numel != expect)
    return fail(SYN_ERR_SHAPE, "syn_set_conv_bn: layer %d expects %lld weights, got %lld", layer,
                (long long)expect, (long long)w_numel);
  HostConv& hc = h->hconv[layer];
  hc.w.assign(w, w + w_numel);
  hc.g.assign(g, g + c.cout); hc.b.assign(b, b + c.cout);
  hc.m.assign(m, m + c.cout); hc.v.assign(v, v + c.cout);
  hc.eps = eps;
  hc.set = true;
  h->committed = false;
  return SYN_OK;
}

int syn_set_heads(syn_handle_t* h, const float* w_ori, const float* b_ori, const float* w_shape,
                  const float* b_shape, const float* w_exp, const float* b_exp) {
  if (h == nullptr || !w_ori || !b_ori || !w_shape || !b_shape || !w_exp || !b_exp)
    return fail(SYN_ERR_INVALID, "syn_set_heads: null argument");
  h->h_head_w.resize((size_t)kNumParams * kLastCh);
  h->h_head_b.resize(kNumParams);
  memcpy(h->h_head_w.data(), w_ori, sizeof(float) * 12 * kLastCh);
  memcpy(h->h_head_w.data() + 12 * kLastCh, w_shape, sizeof(float) * 40 * kLastCh);
  memcpy(h->h_head_w.data() + 52 * kLastCh, w_exp, sizeof(float) * 10 * kLastCh);
  memcpy(h->h_head_b.data(), b_ori, sizeof(float) * 12);
  memcpy(h->h_head_b.data() + 12, b_shape, sizeof(float) * 40);
  memcpy(h->h_head_b.data() + 52, b_exp, sizeof(float) * 10);
  h->heads_set = true;
  h->committed = false;
  return SYN_OK;
}

int syn_set_whitening(syn_handle_t* h, const float* mean, const float* stdv) {
  if (h == nullptr || mean == nullptr || stdv == nullptr) return fail(SYN_ERR_INVALID, "syn_set_whitening: null argument");
  h->h_mean.assign(mean, mean + kNumParams);
  h->h_std.assign(stdv, stdv + kNumParams);
  h->whiten_set = true;
  h->committed = false;
  return SYN_OK;
}

int syn_set_basis_sparse(syn_handle_t* h, const float* u, const float* ws, const float* we, int n_pts) {
  if (h == nullptr || !u || !ws || !we || n_pts <= 0) return fail(SYN_ERR_INVALID, "syn_set_basis_sparse: bad argument");
  h->n_pts = n_pts;
  h->sp_pad = (n_pts + 127) / 128 * 128;
  pack_basis(h->h_sparse, u, ws, we, n_pts, h->sp_pad);
  h->sparse_dirty = true;
  h->committed = false;
  return SYN_OK;
}

int syn_set_basis_dense(syn_handle_t* h, const float* u, const float* ws, const float* we, int64_t n_vert) {
  if (h == nullptr || !u || !ws || !we || n_vert <= 0 || n_vert > (1 << 28))
    return fail(SYN_ERR_INVALID, "syn_set_basis_dense: bad argument");
  h->n_vert = n_vert;
  h->dn_pad = (n_vert + 127) / 128 * 128;
  pack_basis(h->h_dense, u, ws, we, n_vert, h->dn_pad);
  h->dense_dirty = true;
  h->committed = false;
  return SYN_OK;
}

int syn_commit(syn_handle_t* h) {
  if (h == nullptr) return fail(SYN_ERR_INVALID, "syn_commit: null handle");
  for (int l = 0; l < kNumConv; ++l)
    if (!h->hconv[l].set) return fail(SYN_ERR_STATE, "syn_commit: conv layer %d was never set", l);
  if (!h->heads_set) return fail(SYN_ERR_STATE, "syn_commit: heads not set");
  if (!h->whiten_set) return fail(SYN_ERR_STATE, "syn_commit: whitening not set");
  DeviceGuard g(h->device);
  SYN_CUDA(cudaDeviceSynchronize());

  // ---- fold BN (eval) into conv weight/bias and lay out for the SIMT kernels -----------------
  const Plan& P = plan();
  size_t total = 0;
  size_t w_off[kNumConv], b_off[kNumConv];
  for (int l = 0; l < kNumConv; ++l) {
    const ConvDesc& c = P.conv[l];
    const size_t nw = (size_t)c.cout * (c.cin / c.groups) * c.ksize * c.ksize;
    w_off[l] = total; total += (nw + 63) / 64 * 64;
    b_off[l] = total; total += ((size_t)c.cout + 63) / 64 * 64;
  }
  std::vector<float> slab(total, 0.f);
  for (int l = 0; l < kNumConv; ++l) {
    const ConvDesc& c = P.conv[l];
    const HostConv& hc = h->hconv[l];
    float* W = slab.data() + w_off[l];
    float* B = slab.data() + b_off[l];
    const int cpg = c.cin / c.groups, kk = c.ksize * c.ksize;
    for (int co = 0; co < c.cout; ++co) {
      const double scale = (double)hc.g[co] / sqrt((double)hc.v[co] + (double)hc.eps);
      B[co] = (float)((double)hc.b[co] - (double)hc.m[co] * scale);
      for (int ci = 0; ci < cpg; ++ci)
        for (int t = 0; t < kk; ++t) {
          const float wf = (float)((double)hc.w[((size_t)co * cpg + ci) * kk + t] * scale);
          size_t dst;
          if (c.kind == kStem) dst = (size_t)(ci * kk + t) * c.cout + co;           // [27][32]
          else if (c.kind == kDepthwise) dst = (size_t)t * c.cout + co;              // [9][C]
          else dst = (size_t)ci * c.cout + co;                                       // [K][N]
          W[dst] = wf;
        }
    }
  }
  if (h->d_weights) { cudaFree(h->d_weights); h->d_weights = nullptr; }
  SYN_CUDA(cudaMalloc(&h->d_weights, total * sizeof(float)));
  SYN_CUDA(cudaMemcpy(h->d_weights, slab.data(), total * sizeof(float), cudaMemcpyHostToDevice));
  for (int l = 0; l < kNumConv; ++l) {
    h->dconv[l].w = h->d_weights + w_off[l];
    h->dconv[l].bias = h->d_weights + b_off[l];
  }
  // ---- tensor-core engine images ---------------------------------------------------------------
  {
    std::vector<uint8_t> all;
    std::vector<float> osc_all, osc;
    for (int l = 0; l < kNumConv; ++l) {
      const ConvDesc& c = P.conv[l];
      if (c.ksize != 1) continue;
      const int Kp = (c.cin + 15) / 16 * 16, Np = (c.cout + 15) / 16 * 16;
      const int nranges = (Np + kTcMaxNr - 1) / kTcMaxNr;
      const int nr = ((Np + nranges - 1) / nranges + 15) / 16 * 16;
      std::vector<uint8_t> img;
      pack_tc_pointwise(img, osc, slab.data() + w_off[l], c.cin, c.cout, Kp, nr, nranges);
      h->tc_osc_off[l] = osc_all.size();
      osc_all.insert(osc_all.end(), osc.begin(), osc.end());
      h->tc_off[l] = all.size();
      h->tc_nr[l] = nr; h->tc_nranges[l] = nranges; h->tc_kp[l] = Kp;
      all.insert(all.end(), img.begin(), img.end());
      all.resize((all.size() + 1023) / 1024 * 1024);
    }
    if (h->d_tcw) { cudaFree(h->d_tcw); h->d_tcw = nullptr; }
    SYN_CUDA(cudaMalloc(&h->d_tcw, all.size()));
    SYN_CUDA(cudaMemcpy(h->d_tcw, all.data(), all.size(), cudaMemcpyHostToDevice));
    int rc_o = upload(&h->d_tc_oscale, osc_all);
    if (rc_o != SYN_OK) return rc_o;
    if (h->d_err == nullptr) {
      SYN_CUDA(cudaHostAlloc(&h->d_err, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));   // UVA: same pointer on the device
      SYN_CUDA(cudaMalloc(&h->d_sat, sizeof(int)));
    }
    *reinterpret_cast<volatile int*>(h->d_err) = 0;
    SYN_CUDA(cudaMemset(h->d_sat, 0, sizeof(int)));
    SYN_CUDA(cudaFuncSetAttribute(tc_pointwise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
    h->tc_ready = true;
  }
  // ---- fused-block images: conv indices: stem 0 | b1: dw 1, proj 2 | block k>=2: 3k-3, 3k-2, 3k-1 ------
  {
    std::vector<uint8_t> all, img;
    auto W = [&](int l) { return slab.data() + w_off[l]; };
    auto Bv = [&](int l) { return slab.data() + b_off[l]; };
    auto add = [&](int block) {
      h->fused_off[block] = all.size();
      all.insert(all.end(), img.begin(), img.end());
      all.resize((all.size() + 1023) / 1024 * 1024);
    };
    pack_fused<FusedStemB1>(img, W(0), 27, Bv(0), W(1), Bv(1), W(2), Bv(2)); add(1);
    auto blk = [&](int b, auto tag) {      // block b >= 2: convs 3b-3 (expand), 3b-2 (dw), 3b-1 (project)
      using Cfg = decltype(tag);
      const int e = 3 * b - 3;
      pack_fused<Cfg>(img, W(e), Cfg::CIN, Bv(e), W(e + 1), Bv(e + 1), W(e + 2), Bv(e + 2));
      add(b);
    };
    blk(2, FusedB2{}); blk(3, FusedB3{}); blk(4, FusedB4{}); blk(5, FusedB56{}); blk(6, FusedB56{});
    blk(7, FusedB7{}); blk(8, FusedB8{}); blk(9, FusedB8{}); blk(10, FusedB8{}); blk(11, FusedB11{});
    blk(12, FusedB12{}); blk(13, FusedB12{}); blk(14, FusedB14{}); blk(15, FusedB15{}); blk(16, FusedB15{});
    blk(17, FusedB17{});
    {   // tail: features[18] weights as the A operand of the transposed GEMM (kernels_tail.cuh)
      const float* w = W(51);                       // [K=320][N=1280]
      std::vector<uint8_t> timg((size_t)10 * kTailWBytes, 0);
      std::vector<float> tosc(kTailN);
      for (int n = 0; n < kTailN; ++n) {
        const float sc = channel_scale(w + n, (size_t)kTailN, kTailK);
        tosc[n] = 1.0f / (kActScaleHost * sc);
        const int slice = n / 128, r = n % 128;
        for (int k = 0; k < kTailK; ++k) {
          const int kc = k / kTailKC, kl = k % kTailKC;
          const size_t off = (size_t)slice * kTailWBytes + (size_t)kc * 2 * kTailPlane + (size_t)(r / 8) * 128 +
                             (size_t)(kl / 8) * 2048 + (r % 8) * 16 + (kl % 8) * 2;
          uint16_t hi, lo;
          split_f16_host(w[(size_t)k * kTailN + n] * sc, hi, lo);
          *reinterpret_cast<uint16_t*>(timg.data() + off) = hi;
          *reinterpret_cast<uint16_t*>(timg.data() + off + kTailPlane) = lo;
        }
      }
      if (h->d_tail_w) { cudaFree(h->d_tail_w); h->d_tail_w = nullptr; }
      SYN_CUDA(cudaMalloc(&h->d_tail_w, timg.size()));
      SYN_CUDA(cudaMemcpy(h->d_tail_w, timg.data(), timg.size(), cudaMemcpyHostToDevice));
      int rc_t = upload(&h->d_tail_osc, tosc);
      if (rc_t != SYN_OK) return rc_t;
      SYN_CUDA(cudaFuncSetAttribute(tail_conv_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmem));
    }
    if (h->d_fused) { cudaFree(h->d_fused); h->d_fused = nullptr; }
    SYN_CUDA(cudaMalloc(&h->d_fused, all.size()));
    SYN_CUDA(cudaMemcpy(h->d_fused, all.data(), all.size(), cudaMemcpyHostToDevice));
  }
  int rc;
  if ((rc = upload(&h->d_head_w, h->h_head_w)) != SYN_OK) return rc;
  if ((rc = upload(&h->d_head_b, h->h_head_b)) != SYN_OK) return rc;
  if ((rc = upload(&h->d_mean, h->h_mean)) != SYN_OK) return rc;
  if ((rc = upload(&h->d_std, h->h_std)) != SYN_OK) return rc;
  // alpha scales of the tensor-core reconstruction: |alpha_k * ascale_k| <= 2^10 within 8 sigma of the mean
  std::vector<float> ascale(kNumAlpha);
  for (int k = 0; k < kNumAlpha; ++k) {
    const float bound = fabsf(h->h_mean[12 + k]) + 8.f * fabsf(h->h_std[12 + k]);
    int ex = 0;
    if (bound > 0.f && std::isfinite(bound)) frexpf(bound, &ex);
    ascale[k] = ldexpf(1.f, 10 - ex);
  }
  if ((rc = upload(&h->d_ascale, ascale)) != SYN_OK) return rc;
  {
    std::vector<uint8_t> img;
    std::vector<float> meta;
    if (!h->h_sparse.empty()) {
      if (h->sparse_dirty && (rc = upload(&h->d_sparse, h->h_sparse)) != SYN_OK) return rc;
      h->sparse_dirty = false;
      pack_recon_tc(img, meta, h->h_sparse, h->n_pts, h->sp_pad, ascale.data());
      h->sp_vtiles = h->sp_pad / 128;
      if ((rc = upload_bytes(&h->d_sp_img, img)) != SYN_OK) return rc;
      if ((rc = upload(&h->d_sp_meta, meta)) != SYN_OK) return rc;
    }
    if (!h->h_dense.empty()) {                 // kept on the host (32 MB): whitening changes re-scale the image
      if (h->dense_dirty && (rc = upload(&h->d_dense, h->h_dense)) != SYN_OK) return rc;
      h->dense_dirty = false;
      pack_recon_tc(img, meta, h->h_dense, h->n_vert, h->dn_pad, ascale.data());
      h->dn_vtiles = (int)(h->dn_pad / 128);
      if ((rc = upload_bytes(&h->d_dn_img, img)) != SYN_OK) return rc;
      if ((rc = upload(&h->d_dn_meta, meta)) != SYN_OK) return rc;
    }
    SYN_CUDA(cudaFuncSetAttribute(dense_recon_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDnSmem));
    SYN_CUDA(cudaFuncSetAttribute(dense_recon_fm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFmSmem));
    SYN_CUDA(cudaFuncSetAttribute(dense_recon_fm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFmSmem));
    SYN_CUDA(cudaFuncSetAttribute(dense_recon_fm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFmSmem));
  }
  h->committed = true;
  return SYN_OK;
}

int syn_set_engine(syn_handle_t* h, int engine) {
  if (h == nullptr) return fail(SYN_ERR_INVALID, "syn_set_engine: null handle");
  if (engine != SYN_ENGINE_SIMT_FP32 && engine != SYN_ENGINE_TC_BF16X3 && engine != SYN_ENGINE_TC_FUSED &&
      engine != SYN_ENGINE_TC_FUSED_1PASS)
    return fail(SYN_ERR_UNSUPPORTED, "syn_set_engine: engine %d not available in this build", engine);
  h->engine = engine;
  return SYN_OK;
}
int syn_get_engine(const syn_handle_t* h) { return h ? h->engine : -1; }

// The time-out flag of the bounded in-kernel waits is sticky and lives in mapped host memory: a call that finds it
// raised (by a kernel of an earlier call) refuses to run instead of returning garbage with SYN_OK;
// syn_poll_error reports and clears it.
#define SYN_CHECK_READY(h, name)                                                         \
  if ((h) == nullptr) return fail(SYN_ERR_INVALID, name ": null handle");                \
  if (!(h)->committed) return fail(SYN_ERR_STATE, name ": weights not committed (syn_commit)"); \
  if ((h)->d_err != nullptr && *reinterpret_cast<volatile int*>((h)->d_err) != 0)        \
    return fail(SYN_ERR_CUDA, name ": a kernel of an earlier call timed out in a pipeline wait; its results and " \
                              "everything after it are invalid (syn_poll_error reports and clears the flag)"); \
  (h)->tn = 0

int syn_forward(syn_handle_t* h, const float* x, int batch, float* params, float* pool, void* stream) {
  SYN_CHECK_READY(h, "syn_forward");
  if (x == nullptr || params == nullptr || batch <= 0) return fail(SYN_ERR_INVALID, "syn_forward: bad argument");
  DeviceGuard g(h->device);
  if (h->timing) { mark(h, (cudaStream_t)stream, "start"); h->launches--; }
  return run_backbone(h, x, batch, params, pool, -1, nullptr, (cudaStream_t)stream);
}

int syn_reconstruct(syn_handle_t* h, const float* params, int batch, int dense, int whitening,
                    int transform, float* out, void* stream) {
  SYN_CHECK_READY(h, "syn_reconstruct");
  if (params == nullptr || out == nullptr || batch <= 0) return fail(SYN_ERR_INVALID, "syn_reconstruct: bad argument");
  DeviceGuard g(h->device);
  if (h->timing) { mark(h, (cudaStream_t)stream, "start"); h->launches--; }
  return run_reconstruct(h, params, batch, dense, whitening, transform, out, (cudaStream_t)stream);
}

int syn_reconstruct_image(syn_handle_t* h, const float* params, int batch, int dense, const float* roi5_dev, float* out,
                          void* stream) {
  SYN_CHECK_READY(h, "syn_reconstruct_image");
  if (params == nullptr || out == nullptr || roi5_dev == nullptr || batch <= 0)
    return fail(SYN_ERR_INVALID, "syn_reconstruct_image: bad argument");
  DeviceGuard g(h->device);
  if (h->timing) { mark(h, (cudaStream_t)stream, "start"); h->launches--; }
  return run_reconstruct(h, params, batch, dense, 1, 1, out, (cudaStream_t)stream, roi5_dev);
}

int syn_forward_landmarks(syn_handle_t* h, const float* x, int batch, float* params, float* lmk,
                          void* stream) {
  SYN_CHECK_READY(h, "syn_forward_landmarks");
  if (x == nullptr || lmk == nullptr || batch <= 0) return fail(SYN_ERR_INVALID, "syn_forward_landmarks: bad argument");
  DeviceGuard g(h->device);
  int rc = ensure_workspace(h, batch);
  if (rc != SYN_OK) return rc;
  float* p = params ? params : h->d_params_tmp;
  if (h->timing) { mark(h, (cudaStream_t)stream, "start"); h->launches--; }
  rc = run_backbone(h, x, batch, p, nullptr, -1, nullptr, (cudaStream_t)stream);
  if (rc != SYN_OK) return rc;
  return run_reconstruct(h, p, batch, 0, 1, 1, lmk, (cudaStream_t)stream);
}

static int host_submit_impl(syn_handle_t* h, const void* x_host, int is_u8, int batch, float* params_host, float* lmk_host,
                            int* ticket, bool blocking);
static int host_wait_impl(syn_handle_t* h, int ticket);
static int forward_landmarks_host_impl(syn_handle_t* h, const void* x_host, int is_u8, int batch,
                                       float* params_host, float* lmk_host) {
  int ticket = 0;
  const int rc = host_submit_impl(h, x_host, is_u8, batch, params_host, lmk_host, &ticket, true);
  return rc != SYN_OK ? rc : host_wait_impl(h, ticket);
}

int syn_forward_landmarks_host(syn_handle_t* h, const float* x_host, int batch, float* params_host,
                               float* lmk_host) {
  SYN_CHECK_READY(h, "syn_forward_landmarks_host");
  if (x_host == nullptr || lmk_host == nullptr || batch <= 0)
    return fail(SYN_ERR_INVALID, "syn_forward_landmarks_host: bad argument");
  return forward_landmarks_host_impl(h, x_host, 0, batch, params_host, lmk_host);
}

int syn_forward_landmarks_u8(syn_handle_t* h, const uint8_t* x_u8, int batch, float* params, float* lmk, void* stream) {
  SYN_CHECK_READY(h, "syn_forward_landmarks_u8");
  if (x_u8 == nullptr || lmk == nullptr || batch <= 0) return fail(SYN_ERR_INVALID, "syn_forward_landmarks_u8: bad argument");
  DeviceGuard g(h->device);
  int rc = ensure_workspace(h, batch);
  if (rc != SYN_OK) return rc;
  float* p = params ? params : h->d_params_tmp;
  rc = run_backbone(h, nullptr, batch, p, nullptr, -1, nullptr, (cudaStream_t)stream, x_u8);
  if (rc != SYN_OK) return rc;
  return run_reconstruct(h, p, batch, 0, 1, 1, lmk, (cudaStream_t)stream);
}

// Faces per pipeline chunk: large enough that the 8x8 / 4x4 blocks still fill the 148 SMs, small enough that the copies
// hide behind compute.  The FIRST chunk is small: its host->device copy is the only one nothing can overlap.
// SYN_HOST_CHUNK / SYN_HOST_CHUNK0 override both for measurements.
static int host_chunk_faces() {
  static const int v = [] {
    const char* e = getenv("SYN_HOST_CHUNK");
    const int c = e ? atoi(e) : 0;
    return c > 0 ? c : 512;
  }();
  return v;
}
static int host_submit_chunk_faces() {
  static const int v = [] {
    const char* e = getenv("SYN_HOST_CHUNK_SUBMIT");
    const int c = e ? atoi(e) : 0;
    return c > 0 ? c : 1024;
  }();
  return v;
}
static int host_first_chunk_faces() {
  static const int v = [] {
    const char* e = getenv("SYN_HOST_CHUNK0");
    const int c = e ? atoi(e) : 0;
    return c > 0 ? c : 512;   // measured: [512, 512] beats [128, 448, 448] and [256, 448, 320] (round 2)
  }();
  return v;
}

// Shared host pipeline: chunks of host_chunk_faces() faces, H2D on s_copy overlapped with compute on s_compute.
// Everything is stream-ordered, so a second call may be submitted while the first one computes: its H2D copies then run
// under the first call's kernels (the staging slots and their events persist across calls; the result staging buffers
// are reused in s_compute order, after the previous call's D2H).  At most two calls are in flight.
static int host_submit_impl(syn_handle_t* h, const void* x_host, int is_u8, int batch, float* params_host, float* lmk_host,
                            int* ticket, bool blocking) {
  if (h->n_pts <= 0) return fail(SYN_ERR_STATE, "forward_landmarks_host: sparse basis not set");
  DeviceGuard g(h->device);
  const unsigned long long seq = h->host_calls;
  if (seq >= 2) SYN_CUDA(cudaEventSynchronize(h->ev_call[seq & 1]));   // ticket seq - 2 owns this event: it must be done
  // A blocking call can only overlap its own chunks (512 + 512 measured best); a submitted call overlaps with its
  // neighbours in the queue, so it runs whole 1024-face launches (uint8: 409 K faces/s against 350 K with 512 + 512).
  const int chunk = std::min(batch, blocking ? host_chunk_faces() : host_submit_chunk_faces());
  const size_t x_face = (size_t)3 * kImg * kImg;
  const size_t elt = is_u8 ? 1 : sizeof(float);
  const size_t lmk_face = (size_t)3 * h->n_pts;
  if (batch > h->stage_batch) {
    SYN_CUDA(cudaDeviceSynchronize());
    cudaFree(h->d_stage_lmk); cudaFree(h->d_stage_par);
    h->d_stage_lmk = h->d_stage_par = nullptr;
    h->stage_batch = 0;
    SYN_CUDA(cudaMalloc(&h->d_stage_lmk, batch * lmk_face * sizeof(float)));
    SYN_CUDA(cudaMalloc(&h->d_stage_par, (size_t)batch * kNumParams * sizeof(float)));
    h->stage_batch = batch;
  }
  void* stage[2];
  if (is_u8) {
    if (chunk > h->stage_u8_chunk) {
      SYN_CUDA(cudaDeviceSynchronize());
      cudaFree(h->d_stage_u8[0]); cudaFree(h->d_stage_u8[1]);
      h->d_stage_u8[0] = h->d_stage_u8[1] = nullptr;
      h->stage_u8_chunk = 0;
      SYN_CUDA(cudaMalloc(&h->d_stage_u8[0], chunk * x_face));
      SYN_CUDA(cudaMalloc(&h->d_stage_u8[1], chunk * x_face));
      h->stage_u8_chunk = chunk;
    }
    stage[0] = h->d_stage_u8[0]; stage[1] = h->d_stage_u8[1];
  } else {
    if (chunk > h->stage_chunk) {
      SYN_CUDA(cudaDeviceSynchronize());
      cudaFree(h->d_stage_x[0]); cudaFree(h->d_stage_x[1]);
      h->d_stage_x[0] = h->d_stage_x[1] = nullptr;
      h->stage_chunk = 0;
      SYN_CUDA(cudaMalloc(&h->d_stage_x[0], chunk * x_face * sizeof(float)));
      SYN_CUDA(cudaMalloc(&h->d_stage_x[1], chunk * x_face * sizeof(float)));
      h->stage_chunk = chunk;
    }
    stage[0] = h->d_stage_x[0]; stage[1] = h->d_stage_x[1];
  }
  int rc = ensure_workspace(h, chunk);
  if (rc != SYN_OK) return rc;
  int issued = 0;
  for (int b0 = 0, nb = 0; b0 < batch; b0 += nb, h->host_slot ^= 1, ++h->host_chunks, ++issued) {
    const int slot = h->host_slot;
    nb = std::min(issued == 0 && blocking ? std::min(chunk, host_first_chunk_faces()) : chunk, batch - b0);
    if (h->host_chunks >= 2) SYN_CUDA(cudaStreamWaitEvent(h->s_copy, h->ev_done[slot], 0));   // the slot's last reader
    SYN_CUDA(cudaMemcpyAsync(stage[slot], (const uint8_t*)x_host + (size_t)b0 * x_face * elt, nb * x_face * elt,
                             cudaMemcpyHostToDevice, h->s_copy));
    SYN_CUDA(cudaEventRecord(h->ev_h2d[slot], h->s_copy));
    SYN_CUDA(cudaStreamWaitEvent(h->s_compute, h->ev_h2d[slot], 0));
    float* par = h->d_stage_par + (size_t)b0 * kNumParams;
    rc = run_backbone(h, is_u8 ? nullptr : (const float*)stage[slot], nb, par, nullptr, -1, nullptr, h->s_compute,
                      is_u8 ? (const uint8_t*)stage[slot] : nullptr);
    if (rc != SYN_OK) return rc;
    SYN_CUDA(cudaEventRecord(h->ev_done[slot], h->s_compute));
    rc = run_reconstruct(h, par, nb, 0, 1, 1, h->d_stage_lmk + (size_t)b0 * lmk_face, h->s_compute);
    if (rc != SYN_OK) return rc;
  }
  SYN_CUDA(cudaMemcpyAsync(lmk_host, h->d_stage_lmk, batch * lmk_face * sizeof(float), cudaMemcpyDeviceToHost, h->s_compute));
  if (params_host != nullptr)
    SYN_CUDA(cudaMemcpyAsync(params_host, h->d_stage_par, (size_t)batch * kNumParams * sizeof(float),
                             cudaMemcpyDeviceToHost, h->s_compute));
  SYN_CUDA(cudaEventRecord(h->ev_call[seq & 1], h->s_compute));
  h->host_calls = seq + 1;
  if (ticket != nullptr) *ticket = (int)(seq & 0x7fffffff);
  return SYN_OK;
}

static int host_wait_impl(syn_handle_t* h, int ticket) {
  DeviceGuard g(h->device);
  const unsigned long long next = h->host_calls;
  const unsigned long long t = (next & ~0x7fffffffull) | (unsigned)ticket;
  if (t >= next) return fail(SYN_ERR_INVALID, "syn_host_wait: unknown ticket");
  if (t + 2 >= next) SYN_CUDA(cudaEventSynchronize(h->ev_call[t & 1]));   // older tickets were waited for at submit
  if (h->d_err != nullptr && *reinterpret_cast<volatile int*>(h->d_err) != 0)
    return fail(SYN_ERR_CUDA, "forward_landmarks_host: a kernel timed out in a pipeline wait; the outputs are invalid "
                              "(syn_poll_error reports and clears the flag)");
  return SYN_OK;
}

int syn_forward_landmarks_host_submit(syn_handle_t* h, const void* x_host, int x_is_u8, int batch, float* params_host,
                                      float* lmk_host, int* ticket) {
  SYN_CHECK_READY(h, "syn_forward_landmarks_host_submit");
  if (x_host == nullptr || lmk_host == nullptr || batch <= 0 || ticket == nullptr)
    return fail(SYN_ERR_INVALID, "syn_forward_landmarks_host_submit: bad argument");
  return host_submit_impl(h, x_host, x_is_u8 != 0, batch, params_host, lmk_host, ticket, false);
}

int syn_host_wait(syn_handle_t* h, int ticket) {
  if (h == nullptr) return fail(SYN_ERR_INVALID, "syn_host_wait: null handle");
  return host_wait_impl(h, ticket);
}

int syn_forward_landmarks_host_u8(syn_handle_t* h, const uint8_t* x_host, int batch, float* params_host, float* lmk_host) {
  SYN_CHECK_READY(h, "syn_forward_landmarks_host_u8");
  if (x_host == nullptr || lmk_host == nullptr || batch <= 0)
    return fail(SYN_ERR_INVALID, "syn_forward_landmarks_host_u8: bad argument");
  return forward_landmarks_host_impl(h, x_host, 1, batch, params_host, lmk_host);
}

int syn_set_center_crop(syn_handle_t* h, int margin) {
  if (h == nullptr || margin < 0 || margin >= kImg / 2) return fail(SYN_ERR_INVALID, "syn_set_center_crop: margin must be in [0, 60)");
  h->center_crop = margin;
  return SYN_OK;
}

int syn_pose_decode(syn_handle_t* h, const float* params62_dev, int batch, const float* roi5_dev, double* angles_dev,
                    float* t3d_dev, void* stream) {
  SYN_CHECK_READY(h, "syn_pose_decode");
  if (params62_dev == nullptr || angles_dev == nullptr || t3d_dev == nullptr || batch <= 0)
    return fail(SYN_ERR_INVALID, "syn_pose_decode: bad argument");
  if (h->d_mean == nullptr) return fail(SYN_ERR_STATE, "syn_pose_decode: whitening not set");
  DeviceGuard g(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  pose_decode_kernel<<<(batch + 127) / 128, 128, 0, st>>>(params62_dev, h->d_mean, h->d_std, roi5_dev, angles_dev, t3d_dev, batch);
  SYN_LAUNCH_CHECK("pose_decode_kernel");
  mark(h, st, "pose_decode_kernel");
  return SYN_OK;
}

int syn_peek_error(const syn_handle_t* h, int* flag_out) {
  if (h == nullptr || flag_out == nullptr) return fail(SYN_ERR_INVALID, "syn_peek_error: null argument");
  *flag_out = h->d_err != nullptr ? *reinterpret_cast<volatile int*>(h->d_err) : 0;
  return SYN_OK;
}

int syn_poll_saturation(syn_handle_t* h, int* flag_out) {
  if (h == nullptr || flag_out == nullptr) return fail(SYN_ERR_INVALID, "syn_poll_saturation: null argument");
  DeviceGuard g(h->device);
  SYN_CUDA(cudaDeviceSynchronize());
  *flag_out = 0;
  if (h->d_sat != nullptr) {
    SYN_CUDA(cudaMemcpy(flag_out, h->d_sat, sizeof(int), cudaMemcpyDeviceToHost));
    SYN_CUDA(cudaMemset(h->d_sat, 0, sizeof(int)));
  }
  return SYN_OK;
}

int64_t syn_launch_count(const syn_handle_t* h) { return h ? h->launches : -1; }

int syn_set_timing(syn_handle_t* h, int on) {
  if (h == nullptr) return fail(SYN_ERR_INVALID, "syn_set_timing: null handle");
  h->timing = on != 0;
  h->tn = 0;
  return SYN_OK;
}

int syn_get_timings(syn_handle_t* h, float* ms_out, const char** names_out, int max_entries, int* n_out) {
  if (h == nullptr || ms_out == nullptr || n_out == nullptr) return fail(SYN_ERR_INVALID, "syn_get_timings: null argument");
  DeviceGuard g(h->device);
  SYN_CUDA(cudaDeviceSynchronize());
  int n = 0;
  for (int i = 1; i < h->tn && n < max_entries; ++i, ++n) {
    SYN_CUDA(cudaEventElapsedTime(&ms_out[n], h->tev[i - 1], h->tev[i]));
    if (names_out != nullptr) names_out[n] = h->tname[i];
  }
  *n_out = n;
  return SYN_OK;
}

int syn_poll_error(syn_handle_t* h, int* flag_out) {
  if (h == nullptr || flag_out == nullptr) return fail(SYN_ERR_INVALID, "syn_poll_error: null handle");
  DeviceGuard g(h->device);
  SYN_CUDA(cudaDeviceSynchronize());
  *flag_out = 0;
  if (h->d_err != nullptr) {
    *flag_out = *reinterpret_cast<volatile int*>(h->d_err);
    *reinterpret_cast<volatile int*>(h->d_err) = 0;
  }
  return SYN_OK;
}

#ifdef SYN_FUSED_TRACE
// Debug builds only: copy the phase trace of the fused kernels (kernels_fused.cuh) to the host.
int syn_debug_read_trace(long long* out, int n) {
  SYN_CUDA(cudaDeviceSynchronize());
  SYN_CUDA(cudaMemcpyFromSymbol(out, g_fused_trace, std::min<size_t>((size_t)n, 18 * 2 * 64 * 8) * sizeof(long long)));
  return SYN_OK;
}
#endif

int syn_debug_tile_plan(int batch, int sms, int faces_per_tile, int* split, int* face_groups) {
  if (batch <= 0 || sms <= 0 || split == nullptr || face_groups == nullptr)
    return fail(SYN_ERR_INVALID, "syn_debug_tile_plan: bad argument");
  switch (faces_per_tile) {     // one representative configuration per tile size
    case 1: fused_tile_plan<FusedB3>(batch, sms, *split, *face_groups); break;
    case 2: fused_tile_plan<FusedB8>(batch, sms, *split, *face_groups); break;
    case 8: fused_tile_plan<FusedB15>(batch, sms, *split, *face_groups); break;
    default: return fail(SYN_ERR_INVALID, "syn_debug_tile_plan: faces_per_tile must be 1, 2 or 8");
  }
  return SYN_OK;
}

int syn_debug_forward_until(syn_handle_t* h, const float* x, int batch, int layer, float* out, void* stream) {
  SYN_CHECK_READY(h, "syn_debug_forward_until");
  if (x == nullptr || out == nullptr || batch <= 0 || layer < 0 || layer >= kNumConv)
    return fail(SYN_ERR_INVALID, "syn_debug_forward_until: bad argument");
  DeviceGuard g(h->device);
  return run_backbone(h, x, batch, h->d_params_tmp, nullptr, layer, out, (cudaStream_t)stream);
}

}  // extern "C"

#include "heads_host.inl"
#include "resnet_host.inl"
#include "resnest_host.inl"
