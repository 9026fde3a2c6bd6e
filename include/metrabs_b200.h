/*
 * metrabs_b200.h - C ABI of libmetrabs_b200.so: the B200 (sm_100a) implementation of the MeTRAbs per-crop
 * inference hot path   crops -> CNN backbone -> 1x1-conv head -> 2D + volumetric soft-argmax -> metric scaling
 * -> reconstruct_absolute -> joints [B,J,3].
 *
 * The reference (isarandi/metrabs) is pure Python and has no FFI; its boundary for this path is the nn.Module
 * contract consumed at metrabs_pytorch/multiperson/multiperson_model.py:240-242.  Each entry point below names
 * the reference function it replaces (file:line relative to /root/reference/metrabs_pytorch/).  INTEGRATION.md
 * shows the ctypes binding a maintainer would add on the reference side.
 *
 * Conventions: plain C, raw pointers + sizes, no torch types.  Unless a function says "host", pointers are
 * DEVICE pointers on the handle's device and work is enqueued on `stream` (a cudaStream_t passed as void*;
 * NULL = legacy default stream) without synchronising the host and without allocating: the caller owns inputs,
 * outputs and the workspace; the library owns only its weight arena.  Every function returns 0 (MTB_OK) or a
 * negative mtb_status; mtb_last_error() gives the message of the last failure on that handle (or the global
 * one when the handle is NULL).  A handle is bound to one device and is not re-entrant; distinct handles are
 * independent (one process per GPU drives one handle).
 */
#ifndef METRABS_B200_H_
#define METRABS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTB_ABI_VERSION 1

typedef enum {
  MTB_OK = 0,
  MTB_ERR_INVALID_ARG = -1,
  MTB_ERR_CUDA = -2,
  MTB_ERR_NOT_FINALIZED = -3,
  MTB_ERR_MISSING_WEIGHT = -4,
  MTB_ERR_WORKSPACE = -5,
  MTB_ERR_UNSUPPORTED = -6,
  MTB_ERR_NCCL = -7
} mtb_status;

typedef enum { MTB_DTYPE_F32 = 0, MTB_DTYPE_BF16 = 1, MTB_DTYPE_F16 = 2, MTB_DTYPE_I64 = 3 } mtb_dtype;

/* Backbone families of BASELINE.json's configs.  EFFNET covers EfficientNetV2-S/M/L and any table in the same
 * block grammar (backbones/efficientnet.py:379-433); RESNET50 / MOBILENETV3_SMALL follow the TF-only
 * metrabs_tf/backbones/{resnet,mobilenet_v3}.py. */
typedef enum { MTB_ARCH_EFFNET = 0, MTB_ARCH_RESNET50 = 1, MTB_ARCH_MOBILENETV3_SMALL = 2,
               MTB_ARCH_HEAD_ONLY = 3 } mtb_arch;

/* Arithmetic of the conv/GEMM kernels.  FP32: CUDA-core fp32 FMA everywhere (the 1e-3 parity mode).
 * BF16_TC: bf16 operands on tcgen05 tensor cores with fp32 accumulation in TMEM, bf16 activations in HBM
 * (the throughput mode; the reference itself deploys under fp16 autocast, multiperson_model.py:241). */
typedef enum { MTB_PRECISION_FP32 = 0, MTB_PRECISION_BF16_TC = 1,
               /* verification mode: same bf16 storage and bf16-rounded weights as BF16_TC, but every conv on CUDA
                * cores (fp32 FMA) - lets tests separate tensor-core kernel bugs from bf16 rounding effects */
               MTB_PRECISION_BF16_SIMT = 2,
               /* the 1e-3 parity mode ON TENSOR CORES: fp32 storage, every conv/GEMM as three tcgen05 kind::tf32
                * products of hi/lo-split operands (a_hi*b_hi + a_lo*b_hi + a_hi*b_lo) with fp32 accumulation in TMEM;
                * conv outputs agree with the fp32 FMA chain to ~1e-6 */
               MTB_PRECISION_TF32X3 = 3 } mtb_precision;

/* Layout of a logits tensor handed to the standalone soft-argmax. */
typedef enum {
  MTB_LAYOUT_BDJHW = 0, /* reference layout after rearrange 'b (d j) h w -> b d j h w' (models/metrabs.py:79) */
  MTB_LAYOUT_BHWN = 1   /* library-internal NHWC, channel n = J + d*J + j (2D logits in n < J) */
} mtb_layout;

#define MTB_MAX_STAGES 16

/* One row of EfficientNet's inverted_residual_setting (backbones/efficientnet.py:47-107). */
typedef struct {
  int32_t block;       /* 0 = FusedMBConv (:176-234), 1 = MBConv (:110-173) */
  int32_t expand;      /* expand_ratio */
  int32_t kernel;      /* 3 */
  int32_t stride;      /* stride of the first block of the stage */
  int32_t cin, cout;
  int32_t layers;
  int32_t bottomright; /* bottomright_stride: pad (pb-1, pe+1) on the first block (:140-141, :195-196) */
} mtb_stage;

/* Frozen copy of the get_config() keys the path reads (util.py:41-57; config/config_l.yaml:1-21). */
typedef struct {
  int32_t abi_version;                /* MTB_ABI_VERSION */
  int32_t arch;                       /* mtb_arch */
  int32_t precision;                  /* mtb_precision */
  int32_t device;                     /* CUDA device ordinal */
  int32_t proc_side;                  /* S */
  int32_t stride_train, stride_test;
  int32_t centered_stride;
  int32_t legacy_centered_stride_bug; /* models/util.py:17-18 */
  int32_t depth;                      /* D */
  int32_t n_joints;                   /* J (n_raw_points) */
  int32_t feature_channels;           /* C: channels entering the head (needed for MTB_ARCH_HEAD_ONLY) */
  float box_size_mm;
  float mix_3d_inside_fov;            /* < 0 means None (ptu3d.py:28) */
  int32_t weak_perspective;           /* must be 0: the reference's weak-perspective solve crashes (ptu.py:30) */
  int32_t n_stages;                   /* EFFNET only */
  int32_t last_channel;               /* EFFNET only: 1280 */
  mtb_stage stages[MTB_MAX_STAGES];
} mtb_config;

typedef struct mtb_handle mtb_handle;

/* Metrabs.__init__ (models/metrabs.py:12-45) + backbone construction (backbones/efficientnet.py:237-357). */
int mtb_create(const mtb_config* cfg, mtb_handle** out);
int mtb_destroy(mtb_handle* h);
const char* mtb_last_error(const mtb_handle* h);
const char* mtb_version(void);

/* load_state_dict (scripts/demo_image.py:73): one call per entry, `name` in the reference key schema
 * ("backbone.1.<stage>.<block>.block.<i>.0.weight", "heatmap_heads.conv_final.bias", ...).  `data` is a HOST
 * pointer to a contiguous tensor in torch layout; it is copied.  Unknown names are ignored
 * (num_batches_tracked).  mtb_finalize_weights folds BN, repacks to NHWC / K-major, uploads, and fails with
 * MTB_ERR_MISSING_WEIGHT naming the first absent key. */
int mtb_load_weight(mtb_handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim);
int mtb_finalize_weights(mtb_handle* h);

size_t mtb_workspace_bytes(const mtb_handle* h, int batch);
/* Elements per crop of the feature map [H*W*C] and its spatial side, after finalize. */
int mtb_feature_shape(const mtb_handle* h, int* hw_side, int* channels);

/* self.backbone(image) (models/metrabs.py:50): crops fp32 NCHW [B,3,S,S] in [0,1] -> features NHWC
 * [B,S/s,S/s,C] (fp32, or bf16 in BF16_TC mode). */
int mtb_backbone_forward(mtb_handle* h, const float* crops, int batch, void* features, void* workspace,
                         size_t workspace_bytes, void* stream);

/* MetrabsHeads.forward (models/metrabs.py:75-85) incl. heatmap_to_image / heatmap_to_metric
 * (models/util.py:6-33): features NHWC -> coords2d [B,J,2] px, coords3d_rel [B,J,3] mm (fp32). */
int mtb_head_decode(mtb_handle* h, const void* features, int batch, float* coords2d, float* coords3d_rel,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ptu.soft_argmax (ptu.py:54-75), standalone over materialised logits (config c5 / roofline sweep); dtype f32, bf16 or
 * f16 (f16: what the reference's head emits under autocast, multiperson_model.py:241; reference layout only).
 * BDJHW: logits [B,D,J,H,W] -> out [B,J,3] = (x,y,z) in [0,1];  with depth == 0: logits [B,J,H,W] -> out
 * [B,J,2].  BHWN: logits [B,H,W,J*(1+D)] -> out2d [B,J,2] and out3d [B,J,3] (either may be NULL). */
int mtb_softargmax(const void* logits, int dtype, int layout, int batch, int n_joints, int depth, int height,
                   int width, float* out2d, float* out3d, void* stream);

/* ptu3d.reconstruct_absolute (ptu3d.py:9-33) with reconstruct_ref_fullpersp (:56-105), is_within_fov
 * (:113-121), back_project (:108-110).  scratch: >= mtb_reconstruct_scratch_bytes(batch) bytes. */
size_t mtb_reconstruct_scratch_bytes(int batch);
int mtb_reconstruct_absolute(mtb_handle* h, const float* coords2d, const float* coords3d_rel,
                             const float* intrinsics, int batch, float* coords3d_abs, void* scratch,
                             void* stream);

/* Metrabs.forward (models/metrabs.py:47-64): crops [B,3,S,S] fp32 + intrinsics [B,3,3] fp32 -> [B,J,3] fp32. */
int mtb_forward(mtb_handle* h, const float* crops, const float* intrinsics, int batch, float* coords3d_abs,
                void* workspace, size_t workspace_bytes, void* stream);

/* Same call for HOST buffers (the reference-facing end-to-end path): pinned or pageable host crops/intrinsics
 * in, host joints out; H2D/D2H copies and the forward are enqueued on `stream`, then the stream is
 * synchronised.  The library keeps a device staging area sized by the largest batch seen. */
int mtb_forward_host(mtb_handle* h, const float* host_crops, const float* host_intrinsics, int batch,
                     float* host_coords3d_abs, void* stream);

/* Pipelined form of the same call for back-to-back batches (the reference's caller feeds chunk after chunk,
 * multiperson_model.py:190-207): `submit` enqueues the H2D copies of this batch on an internal copy stream and the forward +
 * joints read-back on `stream` behind them, and returns without synchronising; `wait` blocks until that slot's joints are
 * in `host_coords3d_abs`.  Two slots (0/1): submit batch i+1 on the other slot before waiting for batch i, and its
 * host->device copy overlaps batch i's forward.  Host buffers must be pinned for the copies to be asynchronous and must
 * stay valid until the matching wait. */
int mtb_forward_host_submit(mtb_handle* h, const float* host_crops, const float* host_intrinsics, int batch,
                            float* host_coords3d_abs, int slot, void* stream);
int mtb_forward_host_wait(mtb_handle* h, int slot);

/* Multi-GPU (SURVEY.md 8e): crops shard across ranks; one all-gather of the decoded joints over NVLink.
 * mtb_comm_* wrap a NCCL communicator owned by the handle (libnccl is dlopen'ed). */
int mtb_comm_unique_id(void* id128 /* host, 128 bytes */);
int mtb_comm_init(mtb_handle* h, const void* id128, int rank, int world_size);
int mtb_allgather_joints(mtb_handle* h, const float* local, int floats_per_rank, float* all, void* stream);
/* The sharded forward in one call, no allocation: this rank's `batch_local` crops (the same count on every rank) ->
 * backbone -> head decode -> ONE ncclAllGather of [coords2d | coords3d_rel] (5 floats per joint) -> absolute reconstruction
 * of the full batch on every rank (reconstruct_ref_fullpersp uses batch-global RMS scalars, ptu3d.py:71-74, so the result
 * equals the unsharded Metrabs.forward on the concatenated batch).  intrinsics_all [world*batch_local,3,3] and
 * coords3d_abs_all [world*batch_local,J,3] are in rank order; scratch >= mtb_sharded_scratch_bytes(h, batch_local). */
size_t mtb_sharded_scratch_bytes(const mtb_handle* h, int batch_local);
int mtb_forward_sharded(mtb_handle* h, const float* crops_local, int batch_local, const float* intrinsics_all,
                        float* coords3d_abs_all, void* scratch, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * The callers either side of the crop model (SURVEY.md 8f; /root/reference/metrabs_pytorch/multiperson/).  Handle-free
 * device functions: every pointer is a DEVICE pointer, work is enqueued on `stream`, nothing is allocated or synchronised.
 * Crop order: flat index = aug * n_boxes + box (multiperson_model.py:236-239).
 * ------------------------------------------------------------------------------------------------------------------ */

/* Gamma decoding `(images / 255) ** 2.2` (multiperson_model.py:200) + the box-filter pyramid of warp_images_with_pyramid
 * (warping.py:9-13).  images: u8 NCHW [n,3,H,W].  level1 [n,3,H/2,W/2] and level2 [n,3,H/4,W/4] are fp32 (floor sizes);
 * level 0 is decoded on the fly by mtb_warp_crops. */
int mtb_image_pyramid(const uint8_t* images, int n_images, int height, int width, float* level1, float* level2,
                      void* stream);

/* _get_new_rotation_and_scale (multiperson_model.py:321-355) + the per-crop matrices of _get_crops (:264-293) + the
 * pyramid level choice (warping.py:20-21). */
typedef struct {
  const float* boxes;            /* [n_boxes, box_stride]: x, y, w, h(, score) in image pixels */
  int32_t box_stride;
  const float* intrinsics;       /* [n_boxes,3,3] of the image each box lives in */
  const float* distortion;       /* [n_boxes, n_dist] OpenCV order (k1,k2,p1,p2,k3,k4,k5,k6,s1..s4), zero padded */
  int32_t n_dist;                /* 0..12 */
  const float* camspace_up;      /* [n_boxes,3] */
  const float* aug_rotflipmat;   /* [num_aug,3,3] */
  const float* aug_scales;       /* [num_aug] */
  int32_t n_boxes, num_aug, resolution, antialias_factor;
  float* new_intrinsics;         /* out [num_aug*n_boxes,3,3] (the intrinsics mtb_forward takes) */
  float* rotations;              /* out [num_aug*n_boxes,3,3] R = aug_rotflipmat @ R_noaug */
  float* inv_projections;        /* out [num_aug*n_boxes,3,3] inv(new_intrinsics @ R) (@ antialias scaling) */
  int32_t* pyramid_levels;       /* out [num_aug*n_boxes] */
} mtb_crop_setup_args;
int mtb_crop_setup(const mtb_crop_setup_args* args, void* stream);

/* warp_images_with_pyramid + the gamma of _get_crops (warping.py:6-52, multiperson_model.py:295-319): every crop of the
 * batch in ONE launch, written as the fp32 NCHW [num_aug*n_boxes,3,res,res] tensor mtb_forward reads.  antialias_factor
 * 1, 2 or 4 (rendered by supersampling = the reference's larger render followed by avg_pool2d). */
typedef struct {
  const uint8_t* images;         /* [n_images,3,H,W] u8 */
  const float* level1;           /* from mtb_image_pyramid */
  const float* level2;
  int32_t n_images, height, width;
  const float* intrinsics;       /* [n_boxes,3,3] */
  const float* distortion;       /* [n_boxes, n_dist] */
  int32_t n_dist;
  const int32_t* image_ids;      /* [n_boxes] */
  const float* inv_projections;  /* [num_aug*n_boxes,3,3] */
  const int32_t* pyramid_levels; /* [num_aug*n_boxes] */
  const float* gamma_exponents;  /* [num_aug] = aug_gammas / 2.2 */
  int32_t n_boxes, num_aug, resolution, antialias_factor;
  float* crops;                  /* out [num_aug*n_boxes,3,res,res] */
} mtb_warp_args;
int mtb_warp_crops(const mtb_warp_args* args, void* stream);

/* The epilogue of _predict_single_batch (mirror swap, poses @ R; multiperson_model.py:246-259) and of
 * _estimate_poses_batched (joint transform, 2D projection with distortion + intrinsics, inverse extrinsics, skeleton
 * gather, mean over augmentations; :143-182). */
typedef struct {
  const float* poses;            /* [num_aug*n_boxes, J, 3] crop-model output */
  const float* rotations;        /* [num_aug*n_boxes,3,3] */
  const uint8_t* aug_should_flip;/* [num_aug] */
  const int32_t* mirror_mapping; /* [J] */
  const float* joint_transform;  /* [J, J2] or NULL (J2 = J) */
  const int32_t* skeleton;       /* [Js] indices into J2, or NULL (Js = J2) */
  const float* intrinsics;       /* [n_boxes,3,3] */
  const float* distortion;       /* [n_boxes, n_dist] */
  int32_t n_dist;
  const float* extrinsics_inv;   /* [n_boxes,4,4] inverse extrinsic matrix of the box's image */
  int32_t n_boxes, num_aug, n_joints, n_joints_transformed, n_skeleton, average_aug;
  float* poses3d;                /* out [n_boxes,(num_aug,)Js,3] */
  float* poses2d;                /* out [n_boxes,(num_aug,)Js,2] */
} mtb_tta_args;
int mtb_tta_merge(const mtb_tta_args* args, void* stream);

/* plausibility_check.py:8-119: is_pose_plausible, are_augmentation_results_consistent, is_pose_consistent_with_box and
 * pose_non_max_suppression (similarity threshold 0.4) per image.  At most 128 boxes per image, num_aug <= 16. */
typedef struct {
  const float* poses3d;          /* [n_boxes, num_aug, J, 3] camera space */
  const float* poses2d;          /* [n_boxes, num_aug, J, 2] */
  const float* boxes;            /* [n_boxes, box_stride] x, y, w, h, score */
  int32_t box_stride;
  const int32_t* bones;          /* [n_bones,2] joint pairs (rows of joint2bone_mat) */
  const float* mean_bones;       /* [n_bones] mm */
  int32_t n_bones;
  const int32_t* image_start;    /* [n_images+1] box range of each image */
  int32_t n_images, n_boxes, num_aug, n_joints;
  uint8_t* plausible;            /* out [n_boxes] */
  uint8_t* keep;                 /* out [n_boxes]: plausible and not suppressed */
  float* scratch;                /* [n_boxes, J, 3] */
} mtb_filter_args;
int mtb_filter_poses(const mtb_filter_args* args, void* stream);

/* Introspection for tests / profiling. */
int mtb_num_ops(const mtb_handle* h);
const char* mtb_op_name(const mtb_handle* h, int op);
/* Runs the first `n_ops` backbone ops and copies that op's NHWC output (as fp32) to `out` (device). */
int mtb_debug_run_ops(mtb_handle* h, const float* crops, int batch, int n_ops, float* out, size_t out_floats,
                      void* workspace, size_t workspace_bytes, void* stream);
int mtb_op_output_shape(const mtb_handle* h, int op, int* height, int* width, int* channels);
int mtb_op_input_shape(const mtb_handle* h, int op, int* height, int* width, int* channels, int* has_residual,
                       int* has_scale);
/* Runs ONE backbone op in isolation on caller-provided fp32 NHWC device tensors (converted to the handle's
 * storage type): in [B,Hin,Win,Cin] (the stem takes NCHW crops), optional residual [B,Hout,Wout,Cout] and
 * squeeze-excitation scale [B,Cin]; out receives [B,Hout,Wout,Cout] as fp32.  Lets tests compare the tcgen05
 * kernels with the CUDA-core kernels on identical inputs. */
int mtb_debug_run_op(mtb_handle* h, int op_index, const float* in, const float* res, const float* scale, int batch,
                     float* out, size_t out_floats, void* workspace, size_t workspace_bytes, void* stream);
/* FusedMBConv block fusion (bf16 tensor-core mode): 1 when backbone op `op_index` (a 3x3 stride-1 expand conv) and the op
 * after it (the 1x1 projection, + residual) run as ONE fmb_kernel launch (reference block:
 * metrabs_pytorch/backbones/efficientnet.py:176-234).  mtb_debug_run_fused_block runs that pair in isolation on a
 * caller-provided fp32 NHWC device tensor `in` [B,H,W,Cin] (also the residual when the block has one); `out` receives the
 * block output [B,H,W,Cout] as fp32. */
int mtb_op_is_fused_block(const mtb_handle* h, int op_index);
int mtb_debug_run_fused_block(mtb_handle* h, int op_index, const float* in, int batch, float* out, size_t out_floats,
                              void* workspace, size_t workspace_bytes, void* stream);
/* MBConv front-half fusion (bf16 tensor-core mode, 16x16 and 8x8 maps): 1 when backbone op `op_index` (a 1x1 stride-1 expand
 * conv + SiLU) and the op after it (depthwise 3x3 stride 1 + SiLU, squeeze-excitation squeeze) run as ONE expdw_kernel launch
 * (reference block: metrabs_pytorch/backbones/efficientnet.py:110-173).  mtb_debug_run_expdw runs that pair in isolation on a
 * caller-provided fp32 NHWC device tensor `in` [B,H,W,Cin], fused (fused != 0) or as the two launches of the unfused path;
 * `out` receives the depthwise output [B,H,W,Cexp] and `pooled` the squeeze-excitation means [B,Cexp], both fp32. */
int mtb_op_is_expdw(const mtb_handle* h, int op_index);
int mtb_debug_run_expdw(mtb_handle* h, int op_index, const float* in, int batch, float* out, size_t out_floats, float* pooled,
                        size_t pooled_floats, int fused, void* workspace, size_t workspace_bytes, void* stream);
/* CUDA-event profiler (bench.py's live roofline measurement): between begin and end, every kernel launch of the
 * classes selected by `class_mask` (bit i = class i) is bracketed by cudaEventRecord on the launching stream.
 * mtb_profile_end synchronises those events and returns, per class, the summed device time (ms), algorithmic
 * FLOPs, algorithmic bytes and launch count; arrays must hold mtb_num_kernel_classes() entries. */
int mtb_profile_begin(mtb_handle* h, unsigned class_mask);
int mtb_profile_end(mtb_handle* h, double* ms, double* flops, double* bytes, int64_t* launches);
/* Per-op view of the last profiling window: device ms per backbone op, its algorithmic FLOPs and bytes per crop and
 * its kernel class; arrays hold mtb_num_ops() entries. */
int mtb_profile_op_times(const mtb_handle* h, double* ms, double* flops_per_crop, double* bytes_per_crop, int* cls, int n);
/* Weight bytes the op reads once per launch (bf16 on the tensor-core path, fp32 otherwise); `bytes_per_crop` above counts
 * activations (input + output + residual) only, so a launch on B crops moves B * bytes_per_crop + weight bytes. */
double mtb_op_weight_bytes(const mtb_handle* h, int op);
int mtb_num_kernel_classes(void);
const char* mtb_kernel_class_name(int cls);
/* Number of kernels the last mtb_forward / mtb_backbone_forward / ... call on this handle launched. */
int64_t mtb_last_launch_count(const mtb_handle* h);
double mtb_backbone_flops_per_crop(const mtb_handle* h);
/* Host-side tiling plan of the TMA-staged depthwise 3x3 kernel for an HxW map (no device needed): crops per item, output
 * rows per item, row bands per crop (= SE pooling slices) and bytes of one shared-memory stage; all 0 when the shape falls
 * back to the strip kernel. */
int mtb_debug_dw_plan(int height, int width, int* crops_per_item, int* rows_per_item, int* row_bands, int* stage_bytes);

/* Host-side plan and weight re-pack of the fused FusedMBConv kernel (no device needed; tests/test_host_plans.py): the shared-memory
 * plan for a block shape (all outputs 0 when the shape is not covered) and the stage images of the two weight matrices
 * (w1 [cexp][9*cin], w2 [cout][cexp], any 16-bit element type; pair = 1: the half-per-CTA images of the cta_group::2 kernel). */
int mtb_debug_fmb_plan(int cin, int cexp, int cout, int pair, int* nstages, int* npatch, int* stage_bytes, int* smem_bytes);
/* Host-side plan of the fused expand + depthwise kernel for an (H, W, Cin, Cexp) block shape (no device needed): pixels and
 * crops per tile, weight ring stages and dynamic shared-memory bytes; all 0 when the shape keeps the two launches. */
int mtb_debug_expdw_plan(int height, int width, int cin, int cexp, int* pixels_per_tile, int* crops_per_tile, int* nstages,
                         int* smem_bytes);
int mtb_debug_fmb_pack(const uint16_t* w1, const uint16_t* w2, int cin, int cexp, int cout, int pair, uint16_t* img1, uint16_t* img2);

#ifdef __cplusplus
}
#endif
#endif /* METRABS_B200_H_ */
