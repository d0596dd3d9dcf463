/*
 * synergy_b200.h -- C ABI of the B200 (sm_100a) SynergyNet inference hot path.
 *
 * The reference (choyingw/SynergyNet) has no native boundary for this path: it is a Python
 * nn.Module API (model_building.py:65-165, synergy3DMM.py:70-207) whose arithmetic runs inside
 * PyTorch.  This library sits *under* a Python shim with the same class/method names
 * (synergynet_b200/model_building.py, synergynet_b200/synergy3DMM.py) and is bound with ctypes
 * (synergynet_b200/_lib.py); INTEGRATION.md shows the stub a reference maintainer would add.
 * Each entry point cites the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns SYN_OK (0) or a SYN_ERR_* code; no exceptions cross the boundary;
 *     syn_last_error() returns a thread-local message for the last failing call.
 *   - plain pointers and sizes only.  "_dev" pointers are device memory on the handle's GPU and
 *     are owned by the caller; "_host" pointers are host memory.  `stream` is a cudaStream_t
 *     (passed as void*); work is enqueued on it and NOT synchronised unless stated.
 *   - one handle per device; a handle is not re-entrant (one call at a time per handle), but
 *     different handles may be driven from different host threads (nn.DataParallel replicas,
 *     main_train.py:176).
 *   - tensors are fp32 and contiguous in the layouts the reference uses.
 */
#ifndef SYNERGY_B200_H_
#define SYNERGY_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SYN_ABI_VERSION 1

enum {
  SYN_OK = 0,
  SYN_ERR_INVALID = 1,   /* bad argument (null pointer, negative size, unknown layer ...)      */
  SYN_ERR_CUDA = 2,      /* a CUDA runtime call or kernel launch failed                         */
  SYN_ERR_STATE = 3,     /* call order violated (e.g. forward before syn_commit)               */
  SYN_ERR_SHAPE = 4,     /* "length of params mismatch" (model_building.py:116-119) and alike  */
  SYN_ERR_NOMEM = 5,
  SYN_ERR_UNSUPPORTED = 6 /* not an sm_100 device, or an engine the build does not contain      */
};

/* Compute engines for the 1x1 convolutions / basis products (syn_set_engine). */
enum {
  SYN_ENGINE_SIMT_FP32 = 0,   /* CUDA-core fp32 FMA everywhere (bring-up / cross-check path)     */
  SYN_ENGINE_TC_SPLIT3 = 1,   /* tcgen05.mma, operands split in fp16 hi+lo with exact power-of-two  */
                              /* pre-scaling, 3 MMAs per product (hi*hi + hi*lo + lo*hi), fp32      */
                              /* accumulation in TMEM: meets the 1e-4 parity bar (a bf16 split, the  */
                              /* first version, measured 1.7e-4 and was dropped); convs unfused      */
  SYN_ENGINE_TC_BF16X3 = 1,   /* old name of SYN_ENGINE_TC_SPLIT3                                    */
  SYN_ENGINE_TC_FUSED = 2,    /* default: the same arithmetic with the stem + all 17 inverted-       */
                              /* residual blocks each fused into one kernel (expand -> depthwise ->  */
                              /* project, hidden tensor on chip), last conv fused with the pooling   */
  SYN_ENGINE_TC_FUSED_1PASS = 3 /* NOT parity-grade, never the default: engine 2 with ONE fp16 MMA per */
                              /* product (hi*hi only) in the backbone.  Exists to show how much of    */
                              /* the step is the 3x precision tax; misses the 1e-4 bar (SURVEY fact 6) */
};

typedef struct syn_handle syn_handle_t;

/* Geometry of convolution `layer` (0..51) in execution order; lets the host check a checkpoint
 * against the compiled-in MobileNetV2 plan (mobilenetv2_backbone.py:108-138). */
typedef struct {
  int32_t cin, cout, ksize, stride, groups, relu6, h_in, h_out, residual;
} syn_conv_desc_t;

int         syn_abi_version(void);
const char* syn_last_error(void);
int         syn_num_conv_layers(void);                       /* 52 */
int         syn_conv_desc(int layer, syn_conv_desc_t* out);

/* Lifetime.  Replaces nn.Module construction + .cuda() (model_building.py:66-101). */
int  syn_create(int device, syn_handle_t** out);
void syn_destroy(syn_handle_t* h);

/* ---- weights: host pointers in the reference's own layouts; copied during the call ----------
 * Conv2d weight is OIHW fp32 (cout, cin/groups, k, k); BatchNorm2d is eval-mode
 * (weight, bias, running_mean, running_var, eps) and is folded into the convolution by
 * syn_commit.  Replaces ConvBNReLU / InvertedResidual parameter storage
 * (mobilenetv2_backbone.py:33-68). */
int syn_set_conv_bn(syn_handle_t* h, int layer, const float* w_host, int64_t w_numel,
                    const float* bn_weight_host, const float* bn_bias_host,
                    const float* bn_mean_host, const float* bn_var_host, float eps);
/* classifier_ori / classifier_shape / classifier_exp Linear layers, weights (out,1280) row
 * major (mobilenetv2_backbone.py:147-158). */
int syn_set_heads(syn_handle_t* h, const float* w_ori_host, const float* b_ori_host,
                  const float* w_shape_host, const float* b_shape_host,
                  const float* w_exp_host, const float* b_exp_host);
/* param_mean / param_std, 62 floats each (model_building.py:87-88). */
int syn_set_whitening(syn_handle_t* h, const float* mean_host, const float* std_host);
/* Landmark basis buffers u_base (3*n_pts), w_shp_base (3*n_pts,40), w_exp_base (3*n_pts,10),
 * rows xyz-interleaved (model_building.py:99-101, utils/params.py:30-32). */
int syn_set_basis_sparse(syn_handle_t* h, const float* u_base_host, const float* w_shp_base_host,
                         const float* w_exp_base_host, int n_pts);
/* Dense basis buffers u (3*n_vert), w_shp (3*n_vert,40), w_exp (3*n_vert,10)
 * (model_building.py:89-91).  Optional: only needed for dense reconstruction. */
int syn_set_basis_dense(syn_handle_t* h, const float* u_host, const float* w_shp_host,
                        const float* w_exp_host, int64_t n_vert);
/* Fold BN, re-lay-out for the kernels, upload.  Must follow the setters, may be repeated. */
int syn_commit(syn_handle_t* h);

int syn_set_engine(syn_handle_t* h, int engine);
int syn_get_engine(const syn_handle_t* h);

/* ---- compute, device buffers ------------------------------------------------------------------
 * syn_forward: I2P.forward_test / MobileNetV2._forward_impl (model_building.py:59-62,
 * mobilenetv2_backbone.py:173-189).  x_dev (B,3,120,120) NCHW -> params62_dev (B,62) whitened
 * parameters [ori12|shape40|exp10]; pool1280_dev (B,1280) may be NULL. */
int syn_forward(syn_handle_t* h, const float* x_dev, int batch, float* params62_dev,
                float* pool1280_dev, void* stream);
/* syn_reconstruct: reconstruct_vertex_62 (model_building.py:106-139; benchmark.py:76-97).
 * params62_dev (B,62) -> out_dev (B,3,N) with N = n_pts (dense=0) or n_vert (dense=1). */
int syn_reconstruct(syn_handle_t* h, const float* params62_dev, int batch, int dense,
                    int whitening, int transform, float* out_dev, void* stream);
/* forward_test + reconstruct_vertex_62(dense=False) without leaving the device
 * (benchmark.py:125-127 then :153-166).  params62_dev may be NULL. */
int syn_forward_landmarks(syn_handle_t* h, const float* x_dev, int batch, float* params62_dev,
                          float* lmk_dev, void* stream);

/* ---- image-space outputs of get_all_outputs (SURVEY.md section 8 f1) ----------------------------------------
 * _predict_vertices (utils/inference.py:127-138) fused into the reconstruction: vertices leave the GPU already in the
 * coordinates of the original image.  roi5_dev (B,5) fp32 = kx, sx, ky, sy, kz with kx = (ex-sx)/120, ky = (ey-sy)/120,
 * kz = (kx+ky)/2 evaluated in double on the host like the reference's Python scalars; whitening and the y flip are on. */
int syn_reconstruct_image(syn_handle_t* h, const float* params62_dev, int batch, int dense, const float* roi5_dev,
                          float* out_dev, void* stream);
/* parse_pose + predict_pose (utils/inference.py:33-62,86-92,146-157) for B whitened vectors: angles_dev (B,3) fp64
 * degrees [pitch-like x, yaw-like y, roll-like z in the reference's order], t3d_dev (B,3) fp32 (image coordinates when
 * roi5_dev is given, crop coordinates when NULL). */
int syn_pose_decode(syn_handle_t* h, const float* params62_dev, int batch, const float* roi5_dev, double* angles_dev,
                    float* t3d_dev, void* stream);
/* CenterCrop(margin, mode='test') of the reference loader (utils/ddfa.py:162-243, benchmark.py:116): the uint8 entry
 * points read the `margin`-pixel frame of every crop as 0 before normalising.  0 (default) = off. */
int syn_set_center_crop(syn_handle_t* h, int margin);

/* ---- compute, host buffers (the end-to-end call: H2D of the crops, forward, landmarks, D2H) --
 * x_host (B,3,120,120) fp32, lmk_host (B,3,68), params62_host (B,62) or NULL.  Pinned host
 * memory is recommended; chunks are pipelined over internal streams.  Synchronous. */
int syn_forward_landmarks_host(syn_handle_t* h, const float* x_host, int batch,
                               float* params62_host, float* lmk_host);

/* ---- uint8 crops (SURVEY.md section 8 f1): the reference normalises on the host,
 * `(img - 127.5) / 128` (synergy3DMM.py:192, benchmark.py:116 Normalize(mean=127.5, std=128)); these
 * entry points take the raw uint8 (B,3,120,120) planar crops and apply the same fp32 arithmetic on the
 * device (bit-identical values, 4x fewer bytes over PCIe / HBM). */
int syn_forward_landmarks_u8(syn_handle_t* h, const uint8_t* x_u8_dev, int batch, float* params62_dev,
                             float* lmk_dev, void* stream);
int syn_forward_landmarks_host_u8(syn_handle_t* h, const uint8_t* x_u8_host, int batch,
                                  float* params62_host, float* lmk_host);
/* The same call split in two, for a loader loop that keeps the GPU busy (benchmark.py:119-132 iterates a DataLoader
 * with pinned memory and non_blocking copies): submit enqueues H2D + forward + landmarks + D2H and returns a ticket;
 * syn_host_wait(ticket) returns once lmk_host / params62_host of that call are filled.  Up to two calls may be in flight
 * (the second one's copies run under the first one's kernels); a third submit waits for the oldest.  The host buffers
 * (pinned) must stay valid until their ticket has been waited for.  x_is_u8: 0 = fp32 normalised crops, 1 = raw uint8. */
int syn_forward_landmarks_host_submit(syn_handle_t* h, const void* x_host, int x_is_u8, int batch, float* params62_host,
                                      float* lmk_host, int* ticket);
int syn_host_wait(syn_handle_t* h, int ticket);

/* ---- PointNet refinement heads and the training-forward losses (SURVEY.md section 8 a10 / f4) -------------
 * net 0 = MLP_for (backbone_nets/pointnet_backbone.py:7-64): layer 0..8 = conv1..conv9 (+bn1..bn9);
 * net 1 = MLP_rev (:67-106): layer 0..4 = conv1..conv5, 5/6/7 = conv6_1 / conv6_2 / conv6_3 (+their BN).
 * Conv1d weights are (cout, cin, 1) fp32 host arrays, BatchNorm1d is eval-mode and folded at commit. */
int syn_pointnet_set_layer(syn_handle_t* h, int net, int layer, const float* w_host, int cout, int cin,
                           const float* conv_bias_host, const float* bn_weight_host, const float* bn_bias_host,
                           const float* bn_mean_host, const float* bn_var_host, float eps);
int syn_pointnet_commit(syn_handle_t* h, int net);            /* after syn_commit */
/* MLP_for.forward(x, avgpool, shape_code, expr_code) (pointnet_backbone.py:31-64) as called at
 * model_building.py:149-150: lmk_dev (B,3,68), pool1280_dev (B,1280), params62_dev (B,62; columns 12:52 and
 * 52:62 are the shape / expression codes) -> residual_dev (B,3,68) = point_residual and/or
 * refined_dev (B,3,68) = lmk + 0.05 * point_residual (either may be NULL). */
int syn_mlp_for(syn_handle_t* h, const float* lmk_dev, const float* pool1280_dev, const float* params62_dev,
                int batch, float* residual_dev, float* refined_dev, void* stream);
/* MLP_rev.forward (pointnet_backbone.py:90-106, model_building.py:153): lmk_dev (B,3,68) -> (B,62). */
int syn_mlp_rev(syn_handle_t* h, const float* lmk_dev, int batch, float* params62_dev, void* stream);
/* WingLoss(omega=10, epsilon=2) (loss_definition.py:8-27): mean over the B*3*n_pts coordinates -> out_dev[0]. */
int syn_wing_loss(syn_handle_t* h, const float* pred_dev, const float* target_dev, int batch, int n_pts,
                  float* out_dev, void* stream);
/* ParamLoss (loss_definition.py:29-42), one value per sample -> out_dev (B): mode 0 = 'normal', 1 = 'only_3dmm'
 * (input[:, :50] against target[:, 12:62], as the reference does). */
int syn_param_loss(syn_handle_t* h, const float* input_dev, const float* target_dev, int batch, int mode,
                   float* out_dev, void* stream);

/* ---- ResNet-50 backbone variant (BASELINE.json configs[4]; backbone_nets/resnet_backbone.py:227-249) -----------
 * 53 convolutions in execution order: 0 = conv1 (7x7/s2); then per Bottleneck conv1, conv2, conv3 and -- first block of a
 * stage -- downsample.0 (syn_resnet_conv_desc gives each one's geometry).  Weights OIHW fp32 + eval BatchNorm2d, as
 * for syn_set_conv_bn.  Heads: the four Linear layers concatenated in the reference's OUTPUT order
 * fc_ori | fc_shape | fc_exp | fc_tex -> (102, 2048) weights, (102) bias (:242-246).
 * syn_resnet50_forward: x_dev (B,3,120,120) NCHW -> out102_dev (B,102) exactly what ResNet._forward_impl returns;
 * pool2048_dev (B,2048) = the flattened avgpool, may be NULL.  (The reference's I2P unpacks two values from this
 * backbone and fails, SURVEY.md fact 4; the Python shim adapts: params = out[:, :62], pool = the 2048-d feature.) */
int syn_resnet_num_convs(void);                              /* 53 */
int syn_resnet_conv_desc(int idx, syn_conv_desc_t* out);
int syn_resnet_set_conv(syn_handle_t* h, int idx, const float* w_host, int64_t w_numel, const float* bn_weight_host,
                        const float* bn_bias_host, const float* bn_mean_host, const float* bn_var_host, float eps);
int syn_resnet_set_heads(syn_handle_t* h, const float* w102x2048_host, const float* b102_host);
int syn_resnet_commit(syn_handle_t* h);                      /* after syn_commit */
int syn_resnet50_forward(syn_handle_t* h, const float* x_dev, int batch, float* out102_dev, float* pool2048_dev,
                         void* stream);

/* ---- ResNeSt-50 backbone variant (model_building.py:48-49, I2P with any arch containing 'resnest';
 * backbone_nets/ResNeSt/resnest.py:33-41, resnet.py:29-324, splat.py:11-98) -------------------------------------------
 * 87 parameterised layers in execution order: the deep stem conv1.0, conv1.3, conv1.6 (resnet.py:182-190; conv1.6 is
 * followed by the top-level bn1, :299-300); then per Bottleneck conv1, conv2.conv (3x3, groups 2), conv2.fc1,
 * conv2.fc2, conv3 and -- first block of a stage -- downsample.1, the 1x1 conv behind the avg-down pool (:246-261).
 * syn_resnest_layer_desc names each with the checkpoint's own key prefixes: name = the conv ("<name>.weight",
 * "<name>.bias" when has_bias), bn_name = its eval-mode BatchNorm2d ("<bn_name>.weight/.bias/.running_mean/
 * .running_var") or NULL for conv2.fc2, the one layer without one (splat.py:42).  h_in / h_out are the spatial sizes
 * the layer runs at (conv2 runs at stride 1: the avd AvgPool2d(3, 2, 1) after it downsamples, resnet.py:45-50).
 * syn_resnest_set_layer: w_host OIHW fp32 of cout * cin/groups * ksize^2 values (else SYN_ERR_SHAPE); bias_host and
 * the four BatchNorm tensors must be given exactly when the layer has them (else SYN_ERR_INVALID).
 * Heads: fc_ori | fc_shape | fc_exp concatenated in the reference's output order -> (62, 2048), (62) (resnet.py:316-320;
 * fc_tex is in the checkpoint but never evaluated, :319).
 * syn_resnest50_forward: x_dev (B,3,120,120) NCHW -> out62_dev (B,62) and pool2048_dev (B,2048) (may be NULL), the
 * (x, avgpool) pair ResNet.forward returns (:298-324).  SYN_ERR_STATE before syn_resnest_commit. */
typedef struct {
  const char* name;
  const char* bn_name;
  int32_t cin, cout, ksize, stride, groups, has_bias, h_in, h_out;
} syn_resnest_layer_desc_t;
int syn_resnest_num_layers(void);                            /* 87 */
int syn_resnest_layer_desc(int idx, syn_resnest_layer_desc_t* out);
int syn_resnest_set_layer(syn_handle_t* h, int idx, const float* w_host, int64_t w_numel, const float* bias_host,
                          const float* bn_weight_host, const float* bn_bias_host, const float* bn_mean_host,
                          const float* bn_var_host, float eps);
int syn_resnest_set_heads(syn_handle_t* h, const float* w62x2048_host, const float* b62_host);
int syn_resnest_commit(syn_handle_t* h);                     /* after syn_commit */
int syn_resnest50_forward(syn_handle_t* h, const float* x_dev, int batch, float* out62_dev, float* pool2048_dev,
                          void* stream);

/* ---- Sim3DR: vertex normals, lighting, z-buffer rasterisation (SURVEY.md section 8 row f2) -------------------------
 * Handle-free; every pointer is caller-owned device memory unless it says _host.  B meshes share one triangle list
 * tri_dev (ntri,3) int32, 0-based (utils/render.py:32-33).  Vertices are read in place through element strides:
 * coordinate k of vertex i of mesh b = vertices_dev[b*stride_mesh + i*stride_vertex + k*stride_coord], i.e.
 * (nver, 1) for the dense output (B,3,nver) of syn_reconstruct / syn_reconstruct_image (stride_mesh = 3*nver) and
 * (3, 1) for the (nver,3) arrays the reference passes (Sim3DR/Sim3DR.py:8-29).  normals / colours are (B,nver,3).
 * Normals and rasterisation return the reference's bits (csrc/render_math.h explains how); lighting is its float32
 * arithmetic except x**5, where numpy's powf has no portable bit pattern (<= 1 ulp). */
typedef struct {        /* Sim3DR/lighting.py:24-32 (RenderPipeline.__init__) */
  float intensity_ambient, intensity_directional, intensity_specular;
  float color_ambient[3], color_directional[3], light_pos[3], view_pos[3];
  int32_t specular_exp;
} syn_light_cfg_t;

/* One-time index work per topology: the triangles incident to each vertex, ascending (start_out: nver+1 entries,
 * list_out: 3*ntri), so that vertex normals add up in the reference's order (rasterize_kernel.cpp:189-199).
 * SYN_ERR_SHAPE if a triangle references a vertex outside [0, nver). */
int syn_mesh_incidence_host(const int32_t* tri_host, int ntri, int nver, int32_t* start_out, int32_t* list_out);
/* Sim3DR.get_normal (Sim3DR/Sim3DR.py:8-11 -> rasterize_kernel.cpp:158-213).  tri_normals_ws_dev: B*ntri*3 floats. */
int syn_mesh_normals(const float* vertices_dev, int64_t stride_mesh, int stride_vertex, int stride_coord, int batch, int nver,
                     const int32_t* tri_dev, int ntri, const int32_t* inc_start_dev, const int32_t* inc_tri_dev,
                     float* tri_normals_ws_dev, float* normals_dev, void* stream);
/* RenderPipeline.__call__ up to the rasterize call (Sim3DR/lighting.py:37-75): colours = clip(ambient + diffuse +
 * specular, 0, 1), times texture_dev (nver,3) when that is not NULL.  stats_ws_dev: 6*B uint32. */
int syn_mesh_lighting(const float* vertices_dev, int64_t stride_mesh, int stride_vertex, int stride_coord, int batch, int nver,
                      const float* normals_dev, const syn_light_cfg_t* cfg, const float* texture_dev, uint32_t* stats_ws_dev,
                      float* colors_dev, void* stream);
/* Sim3DR.rasterize (Sim3DR/Sim3DR.py:14-29 -> rasterize_kernel.cpp:217-287): draws the B meshes, in order, onto
 * image_dev (height,width,channels) uint8, each with its own depth buffer as the reference's per-face calls have
 * (utils/render.py:41-45).  colors_dev (B,nver,channels).  alpha must be 1 (the only value the reference's Python
 * API can pass; SYN_ERR_UNSUPPORTED otherwise).  keys_ws_dev: B*height*width uint64.  depth_out_dev: NULL, or
 * (B,height,width) floats that receive each mesh's final depth buffer (-1e8 where nothing was drawn). */
int syn_rasterize(uint8_t* image_dev, int height, int width, int channels, const float* vertices_dev, int64_t stride_mesh,
                  int stride_vertex, int stride_coord, int batch, int nver, const int32_t* tri_dev, int ntri,
                  const float* colors_dev, float alpha, int reverse, uint64_t* keys_ws_dev, float* depth_out_dev, void* stream);

/* ---- FaceBoxes post-processing (SURVEY.md section 8 row f3) -----------------------------------------------------------
 * These entries take the detector network's outputs (syn_fb_forward below, or any other producer). */
enum {
  SYN_NMS_CPU_NMS = 0,     /* FaceBoxes/utils/nms/cpu_nms.pyx:17-68, the path nms_wrapper.py:13-18 takes: suppress on   */
                           /* ovr >= thresh, compared in double                                                       */
  SYN_NMS_PY_CPU_NMS = 1   /* FaceBoxes/utils/nms/py_cpu_nms.py:10-38: keep on ovr <= thresh, compared in float32     */
};
/* Greedy NMS of dets_dev (n,5) fp32 rows [x1 y1 x2 y2 score] ALREADY in descending score order (FaceBoxes.py:116-121
 * sorts before it calls nms).  keep_dev (n) int32 receives the kept row indices in order, *n_keep_dev their count:
 * the index list either reference function returns, bit for bit.  mask_ws_dev: n * ceil(n/64) uint64. */
int syn_nms(const float* dets_dev, int n, double thresh, int mode, uint64_t* mask_ws_dev, int32_t* keep_dev, int32_t* n_keep_dev,
            void* stream);
/* Number of prior boxes for an im_height x im_width network input (utils/prior_box.py:19-43); -1 on bad sizes. */
int syn_faceboxes_num_priors(int im_height, int im_width);
/* FaceBoxes.__call__ between the network and the NMS (FaceBoxes/FaceBoxes.py:98-121): priors, decode
 * (utils/box_utils.py:177-195, variances 0.1 / 0.2), `boxes * scale_bbox / scale`, `scores > conf_thresh`, descending
 * order (ties: higher prior index first), first top_k.  loc_dev (P,4), conf_dev (P,2) softmax output, P =
 * syn_faceboxes_num_priors.  dets_dev (top_k,5), *n_dets_dev = rows written.  cand_ws_dev: P+1 int32. */
int syn_faceboxes_decode(const float* loc_dev, const float* conf_dev, int im_height, int im_width, float box_scale_w,
                         float box_scale_h, float scale, float conf_thresh, int top_k, int32_t* cand_ws_dev, float* dets_dev,
                         int32_t* n_dets_dev, void* stream);

/* The detector network (FaceBoxes/models/faceboxes.py:68-150, FaceBoxesNet in 'test' phase) on ONE image of any size.
 * A separate handle: the detector has its own weights and workspace and does not touch syn_handle_t.  Like syn_handle_t
 * it is bound to one device and is not re-entrant (its activation workspace is shared by consecutive calls, which are
 * ordered by the stream they are enqueued on; a change of image size synchronises the device and reallocates).
 * 33 convolutions in execution order (syn_fb_layer_desc names them with the reference's state_dict prefixes:
 * "conv1", "inception2.branch3x3_2", "loc.0" ...): layers with has_bn take the conv weight (OIHW fp32, no bias) and
 * the eval-mode BatchNorm2d of the same block (<name>.conv.weight / <name>.bn.*), the six head layers take weight +
 * bias.  activation: 0 none, 1 ReLU (BasicConv2d, :8-18), 2 CReLU (:50-64, output has 2*cout channels). */
typedef struct syn_fb syn_fb_t;
typedef struct {
  const char* name;
  int32_t cin, cout, ksize, stride, pad, has_bn, activation;
} syn_fb_layer_desc_t;
int  syn_fb_num_layers(void);                                 /* 33 */
int  syn_fb_layer_desc(int idx, syn_fb_layer_desc_t* out);
int  syn_fb_create(int device, syn_fb_t** out);
void syn_fb_destroy(syn_fb_t* f);
int  syn_fb_set_layer(syn_fb_t* f, int idx, const float* w_host, int64_t w_numel, const float* bias_host, const float* bn_weight_host,
                      const float* bn_bias_host, const float* bn_mean_host, const float* bn_var_host, float eps);
int  syn_fb_commit(syn_fb_t* f);
/* FaceBoxes.__call__ lines 88-96: image_dev (height,width,3) uint8 BGR as cv2 delivers it (already rescaled by the caller,
 * :62-79); the mean (104,117,123) is subtracted on the fly.  loc_dev (P,4) and conf_dev (P,2, softmax applied) are what
 * `self.net(img)` returns, P = syn_faceboxes_num_priors(height, width); feed them to syn_faceboxes_decode + syn_nms. */
int  syn_fb_forward(syn_fb_t* f, const uint8_t* image_dev, int height, int width, float* loc_dev, float* conf_dev, void* stream);
int64_t syn_fb_launch_count(const syn_fb_t* f);

/* ---- introspection ---------------------------------------------------------------------------*/
/* Number of kernels this handle has launched since creation (bench.py "gpu_launches"). */
int64_t syn_launch_count(const syn_handle_t* h);
/* Per-launch device timing of the LAST device-buffer call (syn_forward / syn_forward_landmarks[_u8] /
 * syn_reconstruct): with timing on, a CUDA event is recorded on the caller's stream behind every kernel.
 * syn_get_timings synchronises and returns up to max_entries durations (ms) with the kernel labels
 * (static strings; names_out may be NULL).  Used by bench.py for the per-kernel roofline. */
int syn_set_timing(syn_handle_t* h, int on);
int syn_get_timings(syn_handle_t* h, float* ms_out, const char** names_out, int max_entries, int* n_out);
/* Synchronise the device and report (then clear) the sticky flag a bounded in-kernel wait raises
 * when it times out (pipeline protocol bug); *flag_out = 0 means no kernel ever timed out.
 * While the flag is raised every compute entry point returns SYN_ERR_CUDA instead of results. */
int syn_poll_error(syn_handle_t* h, int* flag_out);
/* The same flag WITHOUT synchronising or clearing (it lives in mapped host memory): cheap enough to
 * call after any host-side synchronisation point. */
int syn_peek_error(const syn_handle_t* h, int* flag_out);
/* Synchronise and report (then clear) the "activation clamped" flag: the split-fp16 engines scale
 * block inputs by 64 and clamp to the fp16 range, i.e. |x| > ~937 saturates; the fp32 engine
 * (SYN_ENGINE_SIMT_FP32) has no such limit.  *flag_out != 0: results of engines 1-3 are suspect. */
int syn_poll_saturation(syn_handle_t* h, int* flag_out);
/* Run the backbone on x_dev but stop after convolution `layer` (0..51) and copy its NHWC
 * activation (batch*h_out*h_out*cout floats, residual already added for project convs) to
 * out_dev.  Per-layer parity tests only. */
int syn_debug_forward_until(syn_handle_t* h, const float* x_dev, int batch, int layer,
                            float* out_dev, void* stream);

/* Debug only: one workspace buffer of the PointNet heads after syn_mlp_for / syn_mlp_rev (synchronises). */
int syn_debug_heads_buffer(syn_handle_t* h, int which, float* out_host, int64_t n);

/* Host-only: the face-group plan the fused engine uses for a launch over `batch` faces on a GPU with
 * `sms` SMs and `faces_per_tile` (1, 2 or 8) faces per full tile.  Groups [0, *split) hold
 * faces_per_tile faces each; for two-face tiles the groups [*split, *face_groups) hold ONE face each
 * (the partial last wave is split so that more SMs share it), otherwise the last group may be
 * partial.  Lets the host logic be tested without a GPU. */
int syn_debug_tile_plan(int batch, int sms, int faces_per_tile, int* split, int* face_groups);

#ifdef __cplusplus
}
#endif
#endif  /* SYNERGY_B200_H_ */
