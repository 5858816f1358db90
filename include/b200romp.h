/*
 * b200romp.h - C ABI of libb200romp.so: the B200 (sm_100a) implementation of ROMP's per-frame
 * inference hot path.
 *
 * The reference (Arthur151/ROMP, simple_romp) has no FFI on this path: it is a Python class API whose
 * four internal seams call PyTorch ops (SURVEY.md section 8b).  Each entry point below replaces one
 * seam; the reference file:line it stands in for is cited next to it.  All pointers are plain device
 * (or, where noted, host) pointers, all sizes are ints, nothing torch-typed crosses the boundary.
 * Every call enqueues work on the caller's CUDA stream and returns immediately; the caller owns all
 * input/output buffers; the library owns only packed constants and the conv-graph workspace.
 *
 * Device selection: entry points that take a handle (net, smpl, bev, tracks) make the handle's device current themselves;
 * the handle-less ones (parse, project, preprocess_bgr, pack_rows, bev_bv_input / parse3d / post, gather_rows) launch on
 * the CURRENT device - the caller must have made the device that owns the stream and the buffers current.
 *
 * Return convention: 0 = OK, negative = error (b200romp_last_error() gives the text).  "Nobody
 * detected" is NOT an error: the person count simply comes back as 0 (reference: post_parser.py:138-140).
 * There is no CPU fallback anywhere in this library.
 */
#ifndef B200ROMP_H_
#define B200ROMP_H_

#ifdef __cplusplus
extern "C" {
#endif

#define B200ROMP_VERSION 200   /* round 2: b200romp_sum_desc.term_c_off, preprocess / temporal / pack entry points */

enum { B200ROMP_OK = 0, B200ROMP_EINVAL = -1, B200ROMP_ECUDA = -2, B200ROMP_ENOMEM = -3, B200ROMP_ESTATE = -4 };
enum { B200ROMP_F32 = 0, B200ROMP_BF16 = 1, B200ROMP_U8 = 2 };
/* conv engines */
/* AUTO: bf16 tensors -> tcgen05 (kind::f16), fp32 tensors -> SIMT fp32.  TF32: fp32 tensors -> tcgen05 kind::tf32 (operands
 * rounded to TF32 with cvt.rna like the reference's cuDNN TF32 convs, fp32 accumulate, fp32 tensors in HBM) where the
 * shape tiles onto the engine, SIMT fp32 otherwise. */
enum { B200ROMP_ENGINE_AUTO = 0, B200ROMP_ENGINE_SIMT = 1, B200ROMP_ENGINE_TCGEN05 = 2, B200ROMP_ENGINE_TF32 = 3 };

typedef struct b200romp_net b200romp_net;    /* a conv graph: backbone + heads                          */
typedef struct b200romp_smpl b200romp_smpl;  /* packed SMPL constants                                     */
typedef void* b200romp_stream;               /* cudaStream_t                                              */

int b200romp_version(void);
const char* b200romp_last_error(void);
/* number of SMs / compute capability of the current device, -1 on error (used to size persistent grids) */
int b200romp_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------------
 * Seam S1: `center_maps, params_maps = self.model(image)`  (simple_romp/romp/main.py:112;
 * ROMPv1.forward model.py:470-481; HigherResolutionNet.forward model.py:382-417).
 *
 * The model is handed over as a graph of fused conv ops on NHWC activation tensors (BatchNorm already
 * folded into weight/bias by the host layer, which reads the reference's state-dict keys).
 * One op computes, for every output pixel p and channel c,
 *     v = sum_{tap,ci} W[c][ci][tap] * in[p*stride + tap - pad][in_c_off + ci] + bias[c]
 *     for each (dy,dx) in the upsample x upsample block of p:   (nearest upsample, model.py:197)
 *         o = v + res[...]            (residual / running fuse sum, model.py:80,239-241)
 *         o = relu ? max(o,0) : o     (model.py:81,242)
 *         o = (c == pow_channel) ? 1.1**o : o        (main.py:113)
 *         out[..][out_c_off + c] = o
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200romp_conv_desc {
  int in, in_c_off;        /* input tensor id, first input channel                                      */
  int out, out_c_off;      /* output tensor id, first output channel                                    */
  int res, res_c_off;      /* residual tensor id or -1, first residual channel                          */
  int res_broadcast;       /* 1 = residual has no batch dimension (per-pixel bias map)                  */
  int cin, cout;           /* channels consumed / produced                                              */
  int ksize, stride;       /* 1|3|7 (padding = ksize/2), stride 1|2; 13 = Conv1d 1x3 along W (BEV); 42 = ConvTranspose2d(4, stride 2,
                              padding 1) with weight [cin][cout][4][4] (ResNet-50 deconv layers, resnet_50.py:93-120)     */
  int relu;                /* 1 = ReLU after the residual add                                           */
  int upsample;            /* 1, 2, 4, 8: nearest-neighbour replication of each conv output             */
  int input_norm;          /* 1 = input tensor holds raw 0..255 frames: x/255*2-1 on load (model.py:384) */
  int pow_channel;         /* output channel (before out_c_off) that gets 1.1**x, or -1                 */
  int engine;              /* B200ROMP_ENGINE_*                                                          */
} b200romp_conv_desc;

b200romp_net* b200romp_net_create(int device);
void b200romp_net_destroy(b200romp_net* net);
/* Declares a per-frame tensor [H,W,C] (NHWC; `nchw`=1 declares [C,H,W], only valid for fp32 outputs).
 * `external`=1: the buffer is caller-owned and bound with b200romp_net_bind before each run.
 * Returns the tensor id (>=0) or a negative error. */
int b200romp_net_add_tensor(b200romp_net* net, int H, int W, int C, int dtype, int nchw, int external);
/* Constant [H,W,C] tensor without batch dimension, uploaded now (e.g. the coord-conv bias map that
 * replaces `torch.cat((x, coordmaps))`, model.py:473). */
int b200romp_net_add_const_tensor(b200romp_net* net, int H, int W, int C, int dtype, const void* host_data);
/* weight: host fp32 [cout][cin][k][k] (PyTorch OIHW), bias: host fp32 [cout] or NULL. Returns op id. */
int b200romp_net_add_conv(b200romp_net* net, const b200romp_conv_desc* desc, const float* weight, const float* bias);
/* Fuse-layer summation of HighResolutionModule.forward (simple_romp/romp/model.py:226-244, nearest upsampling of the
 * higher-index branches :188-197) as ONE elementwise op instead of a chain of residual adds:
 *   out[n,y,x,c] = act( base[n,y,x,c] + sum_k term_k[n, y/up_k, x/up_k, c] ),  summed in fp32 in the order base, term 0, 1, ..
 * All tensors NHWC, C a multiple of 8; term k is [H/up_k, W/up_k, C_k] with C_k >= C and contributes its channel slice
 * [term_c_off_k, term_c_off_k + C) - several fuse terms computed from one branch by ONE merged 1x1 conv live in one tensor;
 * dtypes per tensor (bf16/fp32). */
typedef struct b200romp_sum_desc {
  int out, base;           /* output / identity-term tensor ids, both [H,W,C]                           */
  int n_terms;             /* 1..4                                                                      */
  int term[4];             /* tensor ids                                                                */
  int up[4];               /* 1, 2, 4, 8: nearest-neighbour replication factor of term k                */
  int relu;                /* 1 = ReLU after the sum (model.py:243)                                     */
  int term_c_off[4];       /* first channel of term k inside its tensor (multiple of 8; 0 = whole tensor) */
} b200romp_sum_desc;
/* Returns op id (ops run in the order they were added, convs and sums alike). */
int b200romp_net_add_sum(b200romp_net* net, const b200romp_sum_desc* desc);
/* MaxPool2d(kernel 3, stride 2, padding 1) of the ResNet-50 stem (romp/lib/models/resnet_50.py:42): out [ceil(H/2), ceil(W/2), C]. */
int b200romp_net_add_maxpool(b200romp_net* net, int in, int out);
/* Concurrency lane (0..3) of an op inside the captured CUDA graph: ops of different lanes that do not depend on each other
 * through a tensor (or a recycled workspace buffer) may overlap - the parallel branches of a HighResolutionModule
 * (model.py:226-233) and the three ROMP heads (model.py:475-478).  Default lane 0.  Call before finalize. */
int b200romp_net_set_lane(b200romp_net* net, int op, int lane);
/* Packs weights for the chosen engines, uploads them, plans buffer reuse and allocates the workspace. */
int b200romp_net_finalize(b200romp_net* net, int max_batch);
int b200romp_net_bind(b200romp_net* net, int tensor, void* device_ptr);
/* Enqueue the whole graph for `batch` frames on `stream` (replays a cached CUDA graph when possible). */
int b200romp_net_run(b200romp_net* net, int batch, b200romp_stream stream);
/* Debug/validation: copy an internal tensor ([batch,H,W,C] in its own dtype) to a device buffer. */
int b200romp_net_read_tensor(b200romp_net* net, int tensor, int batch, void* dst_device, b200romp_stream stream);
/* Text description of the plan (one line per op: engine, shapes, buffers); returns bytes written. */
int b200romp_net_describe(b200romp_net* net, char* buf, int len);
/* Number of kernels one b200romp_net_run launches (gpu_launches accounting in bench.py). */
int b200romp_net_num_launches(b200romp_net* net);
/* Per-op device time of one net_run (measurement aid, bench.py / tools/op_profile.py): runs the ops one by one without
 * the CUDA graph, `iters` passes, each op bracketed by CUDA events on `stream`; us_per_op[num_launches] receives the mean. */
int b200romp_net_profile(b200romp_net* net, int batch, int iters, float* us_per_op, b200romp_stream stream);
/* Diagnostics: nets finalized under B200ROMP_TC_STAMPS=1 make the CTA-pair conv kernels record %globaltimer stamps
 * (ns) of their phases; out[op][cta 0..3][16]: 0 entry, 1 prologue done, 2 predecessor grid complete, 3 weights resident,
 * 4 first activation tile landed, 5 last MMA issued, 6 epilogue done, 7 exit.  Synchronises the device. */
int b200romp_net_read_stamps(b200romp_net* net, unsigned long long* out, int n_ops);
/* workspace bytes currently held */
long long b200romp_net_workspace_bytes(b200romp_net* net);

/* Stand-alone conv op on caller buffers (kernel unit tests / microbenchmarks).  Tensors are
 * [batch,H,W,C]; weights as in add_conv. `in_dtype`/`out_dtype`/`res_dtype` are B200ROMP_* codes. */
int b200romp_conv2d(const b200romp_conv_desc* desc, const float* weight_host, const float* bias_host,
                    const void* in, int in_dtype, int in_H, int in_W, int in_C,
                    void* out, int out_dtype, int out_C, int out_nchw,
                    const void* res, int res_dtype, int batch, b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Seam S2: `parsing_outputs(center_maps, params_maps, parser)` (post_parser.py:135-146):
 * CenterMap.parse_centermap (:27-47: 5x5 max-pool NMS :50-54, top-64, threshold), parameter_sampling
 * (:128-133), pack_params_dict (:66-79) incl. rot6D_to_angular (utils.py:471-682).
 * center_maps [B,1,S,S] fp32, params_maps [B,P,S,S] fp32 (channel 0 already 1.1**x).
 * Outputs are written for persons 0..N-1 in (frame asc, score desc; ties: flat index asc) order,
 * N = min(*d_count, capacity); rows >= N are left untouched.
 *   d_count[1] i32 | batch_ids[cap] i64 | flat_inds[cap] i64 | center_confs[cap] f32 |
 *   params_pred[cap,P] f32 | cam[cap,3] | thetas[cap,72] (6 trailing zeros) | betas[cap,n_betas] |
 *   center_preds[cap,2] i64 = (x,y)*512//S
 * P = 3 + 22*6 + n_betas.  `thresh` must be >= 0 (with a negative threshold the reference's result
 * depends on torch.topk's unspecified tie order among suppressed cells).
 * ------------------------------------------------------------------------------------------------ */
int b200romp_parse(const float* center_maps, const float* params_maps, int batch, int map_size, int n_betas,
                   float thresh, int capacity, int* d_count, long long* batch_ids, long long* flat_inds,
                   float* center_confs, float* params_pred, float* cam, float* thetas, float* betas,
                   long long* center_preds, void* workspace, b200romp_stream stream);
/* bytes of device scratch `workspace` must provide for `batch` frames */
long long b200romp_parse_workspace_bytes(int batch);

/* ------------------------------------------------------------------------------------------------
 * Seam S3: `self.smpl_parser(outputs, root_align)` (main.py:168 -> smpl.py:62-108: lbs :111-188,
 * batch_rodrigues :191-222, batch_rigid_transform :236-290, VertexJointSelector :24-35).
 * Constant arrays are host fp32 / int64 with the packed-SMPL schema of pack_smpl_info.py:70-111.
 * ------------------------------------------------------------------------------------------------ */
b200romp_smpl* b200romp_smpl_create(int device, int n_betas, const float* v_template /*[6890,3]*/,
                                    const float* shapedirs /*[6890,3,n_betas]*/, const float* posedirs /*[207,20670]*/,
                                    const float* J_regressor /*[24,6890]*/, const float* weights /*[6890,24]*/,
                                    const long long* parents /*[24]*/, const long long* extra_joints_index /*[21]*/,
                                    const float* J_regressor_extra9 /*[9,6890]*/, const float* J_regressor_h36m17 /*[17,6890]*/);
void b200romp_smpl_destroy(b200romp_smpl* smpl);
/* floats of caller-provided device workspace needed per person: smpl_forward(n, ...) uses n x this many floats; the
 * contents are opaque scratch (per-person operands followed by the coordinate-tile-major v_posed of the blend GEMM) */
int b200romp_smpl_workspace_floats(void);
/* betas [n,betas_stride>=n_betas] (first n_betas used), thetas [n,72] -> verts [n,6890,3], joints [n,71,3].
 * If d_count != NULL the number of persons is min(n, *d_count) read on the device (no host sync). */
int b200romp_smpl_forward(b200romp_smpl* smpl, const float* betas, int betas_stride, const float* thetas, int n,
                          const int* d_count, int root_align, float* workspace, float* verts, float* joints,
                          b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Seam S4: `body_mesh_projection2image(joints, cam, verts, offsets)` (post_parser.py:104-114;
 * batch_orth_proj utils.py:309-315; convert_proejection_from_input_to_orgimg post_parser.py:81-88) and
 * `convert_cam_to_3d_trans` (utils.py:303-307).  cam_trans_lsq is the closed-form least squares of
 * utils.py:347-389 (the reference's own fallback for cv2.solvePnPRansac, utils.py:429-434), focal
 * 443.4, image 512 (post_parser.py:99-100), solved in fp64 per person.
 * offsets6 = host [top,bottom,left,right,h,w].  Optional outputs may be NULL.
 * ------------------------------------------------------------------------------------------------ */
int b200romp_project(const float* joints /*[n,71,3]*/, const float* verts /*[n,6890,3] or NULL*/, const float* cam /*[n,3]*/,
                     int n, const int* d_count, const float* offsets6, float* pj2d_org /*[n,71,2]*/,
                     float* verts_camed_org /*[n,6890,3] or NULL*/, float* cam_trans_weak /*[n,3] or NULL*/,
                     float* cam_trans_lsq /*[n,3] or NULL*/, b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * BEV variant (simple_romp/bev): the stages of BEVv1.forward (bev/model.py:232-250) and of
 * BEV.process_normal_image (bev/main.py:158-181) that are not 2-D/1-D convolutions.  The convolutions
 * (backbone, det_head, param_head, bv_pre_layers, bv_out_layers' Conv1d as ksize code 13 = 1x3) run on
 * b200romp_net graphs.  All maps are 128x128, 64 depth levels.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200romp_bev b200romp_bev;
typedef struct b200romp_bev_weights {   /* host fp32 arrays */
  const float* center_ref;  /* [56]  center_map_refiner, BatchNorm3d folded: w1[27], b1, w2[27], b2   (bev/model.py:185)  */
  const float* cam_ref;     /* [492] cam_map_refiner: w1[3][3][27], b1[3], w2[3][3][27], b2[3]          (bev/model.py:186)  */
  const float* coordmap;    /* [64,128,128,3] coordmap_3d buffer                                       (bev/model.py:128)  */
  const float* anchors;     /* [64]  cam3dmap_anchor                                                   (bev/model.py:77-87) */
  const float* embed;       /* [128,128] position_embeddings.weight                                    (bev/model.py:132)  */
  const float *w0, *b0, *w1, *b1, *w2, *b2;   /* transformer.{0,3,6}: [512,128],[512],[512,512],[512],[143,512],[143]   */
} b200romp_bev_weights;
b200romp_bev* b200romp_bev_create(int device, const b200romp_bev_weights* w);
void b200romp_bev_destroy(b200romp_bev* bev);
/* summon_feats = cat([center_fv, cam_offset, img_feats],1).view(B,2560,128) (bev/model.py:190), stored as the NHWC
 * "image" [B,1,128(w),2560] consumed by the Conv1d graph.  maps_fv [B,4,128,128] fp32 NCHW, img_feats [B,128,128,feats_C]
 * whose first 16 channels are bv_pre_layers' output (feats_C = 32 when that stack runs zero-padded on the tcgen05 engine). */
int b200romp_bev_bv_input(const float* maps_fv, const void* img_feats, int feats_dtype, int feats_C, int batch, void* out, int out_dtype,
                          b200romp_stream stream);
/* center_maps_3d [B,64,128,128] = refiner(center_fv (x) center_bv) (bev/model.py:195-196,206); bv_out = output of
 * bv_out_layers as NHWC [B,1,128(w),128(ch)] (ch < 64: center_maps_bv, >= 64: cam_maps_offset_bv); tmp: same size scratch. */
int b200romp_bev_center3d(b200romp_bev* bev, const float* maps_fv, const void* bv_out, int bv_dtype, int batch, float* tmp,
                          float* center3d, b200romp_stream stream);
/* CenterMap3D.parse_3dcentermap (bev/post_parser.py:44-66): 5x5x5 NMS, top-64 per frame, > thresh.  Order: frame asc,
 * score desc (ties: voxel index asc).  Exact as long as a frame has <= 4096 local maxima above thresh. */
long long b200romp_bev_parse_workspace_bytes(int batch);
int b200romp_bev_parse3d(const float* center3d, int batch, float thresh, int capacity, int* d_count, long long* batch_ids,
                         long long* czyx /*[cap,3]*/, float* conf, void* workspace, b200romp_stream stream);
/* cams = cam_maps_3d[b,:,z,y,x] (refiner evaluated lazily at the detections), mesh_parameter_regression
 * (bev/model.py:225-230) -> params_pred [cap,146], cam_czyx [cap,3]; then pack_params_dict / denormalize_cam_params_to_trans
 * (bev/post_parser.py:240-253,114-128) -> cam [cap,3], thetas [cap,72], betas [cap,11], cam_trans [cap,3].
 * fv_feats = param_head output NHWC [B,128,128,128]. */
int b200romp_bev_regress(b200romp_bev* bev, const float* maps_fv, const void* bv_out, int bv_dtype, const void* fv_feats,
                         int fv_dtype, int capacity, const int* d_count, const long long* batch_ids, const long long* czyx,
                         float* params_pred, long long* cam_czyx, float* cam, float* thetas, float* betas, float* cam_trans,
                         b200romp_stream stream);
/* After SMPL-A (into verts/joints) and SMIL (into verts_smil/joints_smil, may be NULL): merge babies (betas[:,10] > 0.8,
 * bev/post_parser.py:255-278), perspective projection to original-image pixels (:68-107,129-152), then per frame
 * suppressing_redundant_prediction_via_projection and remove_outlier (:167-222).  keep[cap] flags, sel[cap] = indices of
 * the survivors in order, *d_count_out = their number. */
int b200romp_bev_post(const float* betas, const float* verts_smil, const float* joints_smil, float* verts, float* joints,
                      const float* cam, const float* cam_trans, const long long* batch_ids, int batch, int capacity,
                      const int* d_count, const float* offsets6, float nms_thresh, float rel_scale_thresh, float img_max_side,
                      float* pj2d_org, int* keep, int* sel, int* d_count_out, b200romp_stream stream);
/* dst[i] = src[sel[i]] for i < *d_count; rows of row_bytes (multiple of 4) bytes. */
int b200romp_gather_rows(const void* src, int row_bytes, const int* sel, const int* d_count, int capacity, void* dst,
                         b200romp_stream stream);
/* the same with dst row offset *d_base (device int32): dst[*d_base + i] = src[sel[i]] - appends rows without a host sync */
int b200romp_gather_rows_at(const void* src, int row_bytes, const int* sel, const int* d_count, const int* d_base, int capacity,
                            void* dst, b200romp_stream stream);

/* BEV crowd mode, BEV.process_long_image (bev/main.py:184-258, bev/split2process.py) for images with w/h >= 2.
 * plan = DEVICE int32 [n_crops][2]: crop c covers rows 0..h-1 and columns [plan[c][0], plan[c][1]) of the image padded by
 * `pad` zero columns on each side (padding_image_overlap / get_image_split_plan, split2process.py:6-39; the last crop is
 * narrower than h).
 *
 * Per chunk of crops first_crop .. first_crop+batch-1 whose detections (batch_ids = crop - first_crop) went through
 * b200romp_bev_regress and SMPL-A / SMIL:  SMIL baby merge (post_parser.py:255-278); exclude_boudary_subjects
 * (split2process.py:41-46) on every crop but the last (cam_x > 1 - r_c, main.py:209-215) and on crops 2..S-1
 * (cam_x < r_{c-1} - 1, :221-226; crop 1 is never tested); projection in crop pixels (offsets [0,h,0,cw,h,cw], :216-218);
 * per crop suppressing_redundant_prediction_via_projection(conf_based=True) and remove_outlier(scale_thresh=1) (:228-232)
 * with crop_nms_thr_px = nms_thresh * h / 640 (fp32); convert_crop_cam_params2full_image (split2process.py:48-58, :242-248)
 * into cam_full [cap,3].  The survivors' indices go to sel / *d_count_sel in order, *d_base receives the device counter
 * *d_merged, which advances by their number (at most merged_capacity): append them with b200romp_gather_rows_at.
 * flags: int32 [2*capacity] scratch. */
int b200romp_bev_long_crops(const float* betas, const float* verts_smil, const float* joints_smil, float* verts, float* joints,
                            const float* cam, const float* cam_trans, const float* conf, const long long* batch_ids, int batch,
                            int capacity, const int* d_count, const int* plan, int n_crops, int first_crop, int h, int w, int pad,
                            float crop_nms_thr_px, float rel_scale_thresh, float* pj2d_org, float* cam_full, int* flags, int* sel,
                            int* d_count_sel, int* d_base, int* d_merged, int merged_capacity, b200romp_stream stream);
/* The final stage over the *d_count merged people (main.py:253-256): cam_trans from the full-image cams
 * (denormalize_cam_params_to_trans), projection with image_pad_info [(w-h)/2, ., 0, w, h, w] (split2process.py:16-21),
 * suppressing_redundant_prediction_via_projection(conf_based=True) with nms_thr_px = nms_thresh * max(h, w) / 640 (fp32)
 * over all pairs at once, then remove_outlier(scale_thresh=0.5).  Survivors -> sel / *d_count_out in order.
 * workspace: int32 [3*capacity + 1]; capacity <= 65535. */
int b200romp_bev_long_merge(const float* joints, const float* cam, const float* conf, int capacity, const int* d_count, int h, int w,
                            float nms_thr_px, float rel_scale_thresh, float* cam_trans, float* pj2d_org, int* workspace, int* sel,
                            int* d_count_out, b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Row a1/f2: `img_preprocess(image)` (simple_romp/romp/utils.py:16-30, called from ROMP.forward main.py:161): BGR->RGB,
 * centre zero-pad to a square (padding_image :16-24), cv2.resize(INTER_CUBIC) to out_size x out_size, uint8 - one kernel
 * from the raw BGR image in device memory to the network's input frame.  Bit-exact with OpenCV's own 8-bit bicubic
 * resize (resize.cpp; not with the closed-source IPP fast path some OpenCV builds dispatch to, which differs by +-1 LSB).
 * pad_info6 (HOST, may be NULL) receives [top, bottom, left, right, h, w] like padding_image. */
int b200romp_preprocess_bgr(const unsigned char* img_bgr_device, int h, int w, int row_stride_bytes, int out_size,
                            unsigned char* out_rgb_device, float* pad_info6_host, b200romp_stream stream);
/* BEV crowd mode (bev/main.py:193-199): img_preprocess of crops first_crop .. first_crop+n_crops-1 of the padded wide
 * image in one launch, without materialising the padding: columns outside the unpadded image (pad zero columns on each
 * side, split2process.py:6-13) and the centre padding of a crop narrower than h read as zero.  plan = DEVICE int32
 * [.][2] as for b200romp_bev_long_crops.  out_rgb [n_crops, out_size, out_size, 3]; bit-exact like b200romp_preprocess_bgr. */
int b200romp_preprocess_crops_bgr(const unsigned char* img_bgr_device, int h, int w, int row_stride_bytes, int pad,
                                  const int* plan_device, int first_crop, int n_crops, int out_size, unsigned char* out_rgb_device,
                                  b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Row f4: the temporal stage of ROMP.forward with --temporal_optimize (main.py:117-157): One-Euro smoothing of
 * (smpl_thetas, smpl_betas, cam) per tracked person, between seams S2 and S3.  Restates LowPassFilter / OneEuroFilter /
 * create_OneEuroFilter / smooth_results / smooth_global_rot_matrix (utils.py:188-192,203-270) in fp32 on the device; the
 * filter state of every track lives in device memory inside the handle.  slot[i] (device int32) = state slot of person i
 * (0 <= slot < max_tracks; a slot whose state was reset initialises on its next sample) or -1 = leave person i untouched.
 * thetas [n,72], betas [n,betas_stride] (first n_betas smoothed), cam [n,3] are updated IN PLACE; the person count is
 * min(n, *d_count) when d_count != NULL.  The track association (norfair in the reference) is the caller's. */
typedef struct b200romp_tracks b200romp_tracks;
b200romp_tracks* b200romp_tracks_create(int device, int max_tracks);
void b200romp_tracks_destroy(b200romp_tracks* tracks);
/* forget the state of one slot (slot >= 0) or of all slots (slot = -1) */
int b200romp_tracks_reset(b200romp_tracks* tracks, int slot, b200romp_stream stream);
int b200romp_one_euro_smooth(b200romp_tracks* tracks, const int* slot, int n, const int* d_count, float* thetas, float* betas,
                             int betas_stride, int n_betas, float* cam, float smooth_coeff, float freq, b200romp_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Frame-sharded multi-GPU collection (SURVEY 8e; the reference's DataParallel bookkeeping it stands in for:
 * romp/lib/maps_utils/result_parser.py:59-64,123-124).  Packs the per-person output arrays of one rank into the
 * fixed-width record buffer that a single NCCL all-gather ships:
 *   dst = [1 header row | capacity rows] x dst_row_bytes;  row 1+i = concatenation of srcs[s][i] (seg_bytes[s] bytes each);
 *   header int32 = {magic 0x0B200B20, count, user0, user1, dst_row_bytes}.
 * The person count is min(*d_count, capacity) read on the device (d_count may be NULL: then count_host is used), so
 * neither this call nor the all-gather that follows needs a host synchronisation.  srcs / seg_bytes are HOST arrays
 * (nseg <= 16) of device pointers / byte counts (multiples of 4). */
int b200romp_pack_rows(const void* const* srcs, const int* seg_bytes, int nseg, const int* d_count, int count_host,
                       int capacity, int user0, int user1, void* dst, int dst_row_bytes, b200romp_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ROMP_H_ */
