/*
 * p3p.h -- C ABI of libp3p.so: the B200 (sm_100a) LiDAR pillar-encode +
 * early-fusion hot path of PixelsPointsPolygons.
 *
 * Plain C: device pointers, sizes, a CUDA stream handle passed as void*.
 * No allocation, no host synchronisation and no host<->device copy happens
 * inside any p3p_* compute call; the caller owns every buffer (workspace
 * included) and the stream.  All device pointers must be 16-byte aligned.
 * Every function returns 0 on success or a negative P3P_ERR_* code;
 * p3p_last_error() gives the message of the last failure on this thread.
 *
 * What each entry point replaces in the reference (R: = /root/reference):
 *
 *   p3p_voxelize          R:pixelspointspolygons/models/pointpillars/pointpillars_o3d.py:92
 *                         `self.voxelize(x_lidar)` = Open3D-ML PointPillars.voxelize ->
 *                         PointPillarsVoxelization.forward -> open3d.ml.torch.ops.voxelize +
 *                         ragged_to_dense + x/y bound filter (SURVEY 8a rows a4, a5), for the
 *                         whole jagged batch in one call instead of a Python loop per tile.
 *   p3p_pfn_prepare       folds the eval-mode BatchNorm1d of the two PFNLayers into the linears
 *                         (Open3D-ML PFNLayer; state_dict keys of SURVEY Appendix C) and packs the
 *                         second linear in the tensor-core operand layout.
 *   p3p_pillar_features   pointpillars_o3d.py:93 `self.voxel_encoder(voxels, num_points, coors)`
 *                         (PillarFeatureNet.forward, rows a6, a7) -> (V, C) in voxel order.
 *   p3p_encode            pointpillars_o3d.py:92-107: voxelize -> voxel_encoder -> middle_encoder
 *                         (PointPillarsScatter, row a8) -> NCHW or NLC, optionally straight into the
 *                         LiDAR half of the early-fusion concat buffer
 *                         (R:pixelspointspolygons/models/fusion_layers/early_fusion_vit.py:100,113-121,
 *                         rows a10, a11).
 *   p3p_patch_embed       early_fusion_vit.py:99 `self.image_embed(x_image)` (timm PatchEmbed conv
 *                         PxP/P, flatten=False, row a9), written into the image half of the concat
 *                         buffer (early_fusion_vit.py:121 puts image channels first).
 */
#ifndef P3P_H_
#define P3P_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P3P_VERSION 200

enum {
    P3P_OK = 0,
    P3P_ERR_INVALID_ARGUMENT = -1, /* null / misaligned pointer, bad size or enum */
    P3P_ERR_UNSUPPORTED = -2,      /* configuration outside what the kernels implement */
    P3P_ERR_WORKSPACE = -3,        /* workspace too small */
    P3P_ERR_CUDA = -4              /* a CUDA runtime call failed (message has the detail) */
};

/* Arithmetic of the second PFN linear (the dense 32 -> C contraction). */
enum {
    P3P_PRECISION_FP32 = 0, /* exact fp32 FMA on CUDA cores (any M; slow; GPU-side cross-check) */
    P3P_PRECISION_TF32 = 1, /* tcgen05 kind::tf32, fp32 accumulate -- the fp32 (1e-3) contract */
    P3P_PRECISION_BF16 = 2, /* tcgen05 kind::f16 (bf16 operands), fp32 accumulate -- the bf16 (1e-2) contract */
    P3P_PRECISION_FP16 = 3  /* tcgen05 kind::f16 (fp16 operands: 10 mantissa bits like tf32, half the operand bytes), fp32
                               accumulate -- meets the fp32 (1e-3) contract while the layer-0 activations and the folded
                               weights stay inside the fp16 range (|v| < 65504); the caller checks that (the Python
                               module bounds it from the weights and the grid extent and falls back to TF32) */
};

/* Output tensor layouts of p3p_encode. */
enum {
    P3P_LAYOUT_NCHW = 0, /* (B, c_total, ny, nx), LiDAR channels at [c_offset, c_offset + C) */
    P3P_LAYOUT_NLC = 1   /* (B, ny*nx, C) contiguous tokens == x.flatten(2).transpose(1,2) values */
};

enum { P3P_DTYPE_F32 = 0, P3P_DTYPE_BF16 = 1, P3P_DTYPE_F16 = 2 };

/*
 * Voxel grid and limits.  Mirrors the constructor arguments the reference derives from
 * cfg.experiment.encoder.* (pointpillars_o3d.py:39-47) plus PointPillarsScatter's output_shape
 * (R:pixelspointspolygons/models/pointpillars/pointpillars_vit.py:55,60-63).
 */
typedef struct p3p_grid {
    float range_min[3];  /* point_cloud_range[:3]  (0, 0, 0) */
    float range_max[3];  /* point_cloud_range[3:]  (in_width, in_height, in_voxel_size.z) */
    float voxel_size[3]; /* in_voxel_size.{x,y,z} */
    int32_t max_points;  /* max_num_points_per_voxel (M) */
    int32_t max_voxels;  /* max_num_voxels.{train|test} -- the caller picks by module mode */
    int32_t ny, nx;      /* scatter output_shape = [ny, nx] */
    int32_t flags;       /* 0, or P3P_GRID_DROP_OVERFLOW */
} p3p_grid;

/* Points whose cell hash is >= extents_x*extents_y*extents_z (they sit exactly on range_max: z == 100
 * -> z-cell 1, y == 224 -> y-cell 28) are ordinary runs by default (SURVEY Appendix A.1 / B.2); with this
 * flag they are dropped like out-of-range points (the other reading of Open3D's invalid_hash guard). */
#define P3P_GRID_DROP_OVERFLOW 1

/* Raw (un-folded) eval-mode parameters of the PillarFeatureNet, fp32 device pointers.
 * Names are the reference's state_dict keys under `voxel_encoder.pfn_layers.{0,1}.`. */
typedef struct p3p_pfn_params {
    const float* linear0_weight; /* (C0, 8)   pfn_layers.0.linear.weight, C0 = feat_channels[0] / 2 = 32 */
    const float* norm0_weight;   /* (C0)      pfn_layers.0.norm.weight */
    const float* norm0_bias;     /* (C0) */
    const float* norm0_mean;     /* (C0)      running_mean */
    const float* norm0_var;      /* (C0)      running_var */
    const float* linear1_weight; /* (C, 2*C0) pfn_layers.1.linear.weight */
    const float* norm1_weight;   /* (C) */
    const float* norm1_bias;     /* (C) */
    const float* norm1_mean;     /* (C) */
    const float* norm1_var;      /* (C) */
    float eps;                   /* BatchNorm1d eps (1e-3) */
    int32_t channels;            /* C = feat_channels[1] = patch_feature_dim (384) */
    int32_t center_alias;        /* 1: channels 0,1 hold the pillar-centre offsets (SURVEY App. A.3, E1) */
} p3p_pfn_params;

/* Optional integer outputs of p3p_voxelize (the bit-exact parity surface).  Any pointer may be
 * NULL.  All arrays are padded per tile to max_voxels rows; rows >= num_pillars[b] are untouched. */
typedef struct p3p_voxel_outputs {
    int32_t* point_hash;       /* (total_points) cell hash per point, invalid_hash (= number of keys) when out of range */
    int32_t* num_pillars;      /* (B) pillars per tile after the max_voxels cut and the x/y bound filter */
    int32_t* pillar_coords;    /* (B, max_voxels, 4) [b, z, y, x] in voxel order */
    int32_t* pillar_num_points;/* (B, max_voxels) min(count, M) */
    int32_t* pillar_point_idx; /* (B, max_voxels, M) tile-local point indices, ascending, -1 padded */
    float* pillar_points;      /* (B, max_voxels, M, 3) gathered xyz, zero padded (== `voxels`) */
    int32_t* cell_owner;       /* (B, ny*nx) voxel ordinal that owns each canvas cell (last writer), -1 if empty */
} p3p_voxel_outputs;

/* Raw parameters of a 3x3 convolution followed by an eval-mode BatchNorm2d, fp32 device pointers.  Names are the
 * reference's state_dict keys under `fusion_layer.{0,1}.` / `proj.{1,2}.` (nn.Sequential indices). */
typedef struct p3p_conv_params {
    const float* weight;      /* (Cout, Cin, 3, 3)  0.weight */
    const float* bias;        /* (Cout) or NULL     0.bias */
    const float* norm_weight; /* (Cout) or NULL (no BatchNorm)  1.weight */
    const float* norm_bias;   /* (Cout)             1.bias */
    const float* norm_mean;   /* (Cout)             1.running_mean */
    const float* norm_var;    /* (Cout)             1.running_var */
    float eps;                /* BatchNorm2d eps (1e-5) */
    int32_t in_channels;      /* Cin: a multiple of 64 */
    int32_t out_channels;     /* Cout */
} p3p_conv_params;

/* Per-tile constants of p3p_las_to_pixels (a device array of num_tiles entries). */
typedef struct p3p_las_tile {
    double scale[3];         /* las.header.scales */
    double offset[3];        /* las.header.offsets */
    double left, top;        /* img_info['top_left'] (ignored when origin_from_min) */
    double res;              /* img_info.get('res_x', 0.25) */
    double height, width;    /* img_info['height'], img_info['width'] (pixels) */
    int32_t origin_from_min; /* 1: the tile's own x / y minimum is the origin (predictor.py:126) */
    int32_t clip;            /* 1: clip x to [0, width], y to [0, height] (p3_coco.py:95-96) */
    int32_t d4;              /* replayed D4 element on x, y (p3_coco.py:114-160): P3P_D4_NONE (not applied) or E ... T */
    int32_t reserved;
    double center_x, center_y; /* in_width // 2, in_height // 2: centre of the D4 transform */
} p3p_las_tile;

/* P3P_D4_E is the applied identity: like the reference it still moves the points to the centre and back (two float32
 * roundings); P3P_D4_NONE leaves them untouched (transform not applied / not the training split). */
enum { P3P_D4_NONE = 0, P3P_D4_E = 1, P3P_D4_R90 = 2, P3P_D4_R180 = 3, P3P_D4_R270 = 4, P3P_D4_V = 5, P3P_D4_HVT = 6,
       P3P_D4_H = 7, P3P_D4_T = 8 };

const char* p3p_last_error(void);
int p3p_version(void);

/* Bytes of scratch the compute calls need for a batch of B tiles holding total_points points. */
size_t p3p_workspace_bytes(const p3p_grid* grid, int32_t num_tiles, int64_t total_points);

/* Bytes of the prepared-weights blob for C output channels. */
size_t p3p_pfn_blob_bytes(int32_t channels);

/* Fold BN into the linears and pack for `precision`; writes `blob` (device). */
int p3p_pfn_prepare(const p3p_pfn_params* params, int32_t precision, void* blob, size_t blob_bytes, void* stream);

/*
 * Voxelise a jagged batch.  points: (total_points, point_stride) fp32, xyz in lanes 0..2;
 * tile_offsets: (B + 1) int64 on the device (NestedTensor jagged offsets, or arange * N for dense).
 * Leaves the pillar table of the batch in `workspace` for p3p_pillar_features.
 */
int p3p_voxelize(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
                 int64_t total_points, const p3p_grid* grid, const p3p_voxel_outputs* out,
                 void* workspace, size_t workspace_bytes, void* stream);

/*
 * PillarFeatureNet over the pillar table left in `workspace` by p3p_voxelize (same stream, same
 * num_tiles / total_points): features (B, max_voxels, C) fp32, rows >= num_pillars[b] untouched.
 */
int p3p_pillar_features(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const void* blob,
                        int32_t channels, int32_t precision, float* features, void* workspace,
                        size_t workspace_bytes, void* stream);

/*
 * The fused hot path: voxelize -> PFN -> scatter, one call per batch.
 * out: NCHW (B, c_total, ny, nx) written at channels [c_offset, c_offset + C), or NLC rows (B, ny*nx, C) when
 * c_total == 0, (B, ny*nx, c_total) rows at channel c_offset otherwise; out_dtype fp32, bf16 or fp16.  Every cell of the LiDAR channels is written (empty cells = 0), so the
 * buffer needs no memset.  lidar_zero != 0 reproduces `x_lidar * 0.0` (LiDAR dropout) without running
 * the encoder.
 */
int p3p_encode(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
               int64_t total_points, const p3p_grid* grid, const void* blob, int32_t channels, int32_t precision,
               void* out, int32_t out_layout, int32_t out_dtype, int32_t c_total, int32_t c_offset,
               int32_t lidar_zero, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The LiDAR-only ViT input (SURVEY 8f-2): the fused hot path emitting the token sequence the transformer blocks
 * consume, i.e. what timm's `VisionTransformer._pos_embed(self.patch_embed(x))` returns in eval mode for the reference's
 * `vit_small_patch8_224` (one class token, no register tokens, `no_embed_class = False`; call site
 * pixelspointspolygons/models/pointpillars/pointpillars_vit.py:64,74):
 *   tokens[b, 0, :]        = cls_token + pos_embed[0, :]
 *   tokens[b, 1 + cell, :] = encoder(b, cell, :) + pos_embed[1 + cell, :]      (empty cells: pos_embed only)
 * tokens: (B, 1 + ny*nx, C) fp32; cls_token: (C) fp32; pos_embed: (1 + ny*nx, C) fp32, all on the device.
 */
int p3p_encode_tokens(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
                      int64_t total_points, const p3p_grid* grid, const void* blob, int32_t channels, int32_t precision,
                      const float* cls_token, const float* pos_embed, float* tokens, void* workspace,
                      size_t workspace_bytes, void* stream);

/*
 * Image patch embedding: Conv2d(in_chans, C, kernel=P, stride=P, bias) on (B, in_chans, H, W) fp32,
 * written into channels [c_offset, c_offset + C) of out: P3P_LAYOUT_NCHW (B, c_total, H/P, W/P) or P3P_LAYOUT_NLC
 * channels-last rows (B, H/P * W/P, c_total) -- with a 16-bit out_dtype the image half of the fusion convolution's input.
 * weight: (C, in_chans, P, P) fp32; bias: (C) fp32 or NULL.
 */
int p3p_patch_embed(const float* images, int32_t num_tiles, int32_t in_chans, int32_t height, int32_t width,
                    int32_t patch, const float* weight, const float* bias, int32_t channels, int32_t precision,
                    void* out, int32_t out_dtype, int32_t out_layout, int32_t c_total, int32_t c_offset, void* stream);

/*
 * The same with the weights prepared once per checkpoint instead of converted by every CTA of every call (the module of
 * early_fusion_vit.py:69-70 keeps its `proj` parameters for the whole run): p3p_patch_embed_prepare writes the 128-channel
 * tiles of `weight` as tensor-core operand images of `precision` (+ the bias) into blob (p3p_patch_embed_blob_bytes bytes,
 * device memory, 16-byte aligned); p3p_patch_embed_prepared runs the convolution from it -- bit-identical to
 * p3p_patch_embed.  weight / bias are still passed (they may be NULL for 8-px patches with a tensor-core precision): shapes
 * and precisions outside the tensor-core route (other patch sizes, P3P_PRECISION_FP32) read them.
 */
size_t p3p_patch_embed_blob_bytes(int32_t channels, int32_t in_chans, int32_t patch);
int p3p_patch_embed_prepare(const float* weight, const float* bias, int32_t channels, int32_t in_chans, int32_t patch,
                            int32_t precision, void* blob, size_t blob_bytes, void* stream);
int p3p_patch_embed_prepared(const float* images, int32_t num_tiles, int32_t in_chans, int32_t height, int32_t width,
                             int32_t patch, const void* blob, const float* weight, const float* bias, int32_t channels,
                             int32_t precision, void* out, int32_t out_dtype, int32_t out_layout, int32_t c_total, int32_t c_offset,
                             void* stream);

/*
 * The same convolution on the decoded image as a loader holds it before its normalisation: images (B, H, W, in_chans)
 * uint8, channels-last, 8-byte aligned, in_chans 1..4; pixel_lut (in_chans, 256) fp32 on the device, pixel_lut[c][u] the
 * value the loader's normalisation gives byte u of channel c (torchvision ToTensor: u / 255).  The result equals
 * p3p_patch_embed / p3p_patch_embed_prepared on the fp32 image (B, in_chans, H, W) with x[b][c][y][x] =
 * pixel_lut[c][images[b][y][x][c]], bit for bit: the same route, the same row group, the same operand rounding.  blob:
 * prepared weights (as for p3p_patch_embed_prepared) or NULL (then weight is required); the table is read by every call
 * (a CUDA graph that captured one sees later in-place updates of it).
 */
int p3p_patch_embed_u8(const uint8_t* images, const float* pixel_lut, int32_t num_tiles, int32_t in_chans, int32_t height,
                       int32_t width, int32_t patch, const void* blob, const float* weight, const float* bias, int32_t channels,
                       int32_t precision, void* out, int32_t out_dtype, int32_t out_layout, int32_t c_total, int32_t c_offset,
                       void* stream);

/*
 * LiDAR input front end (SURVEY 8a row a1 / 8f-3): raw LAS integer coordinates of a jagged batch -> the (total_points, 3)
 * fp32 pixel-space points p3p_encode consumes, bit-identical to the numpy / scikit-learn code of
 * P3Dataset.load_lidar_points (p3_coco.py:74-101; clip = 1) and Predictor.load_lidar_from_file (predictor.py:116-137;
 * origin_from_min = 1, clip = 0): x = (X*sx+ox - left)/res, y = height - (Y*sy+oy - top)/res, z = MinMaxScaler over the
 * tile to [0, z_hi], all in float64, then float32.  X, Y, Z: (total_points) int32; tile_offsets: (B + 1) int64;
 * minmax_ws: 4 * num_tiles int32 of scratch.  Everything on the device.
 */
int p3p_las_to_pixels(const int32_t* X, const int32_t* Y, const int32_t* Z, const int64_t* tile_offsets, int32_t num_tiles,
                      int64_t total_points, const p3p_las_tile* tiles, double z_hi, int32_t* minmax_ws, float* points,
                      void* stream);

/*
 * The same front end fed with the packed transfer format (6 bytes per point instead of 12, halving the host -> device
 * copy of a batch): per tile an int32 base (X0, Y0, Z0) and per point three uint16 deltas, X = X0 + dX etc.  -- what a
 * loader gets from `las.X - las.X.min()` when the tile spans < 65536 steps of the LAS scale (56 m at 1 mm .. 1 cm).
 * deltas: (total_points, 3) uint16; tile_base: (B, 3) int32.  Results are bit-identical to p3p_las_to_pixels on the same
 * integers.
 */
int p3p_las_packed_to_pixels(const uint16_t* deltas, const int32_t* tile_base, const int64_t* tile_offsets, int32_t num_tiles,
                             int64_t total_points, const p3p_las_tile* tiles, double z_hi, int32_t* minmax_ws, float* points,
                             void* stream);

/*
 * SURVEY 8f rank 1 -- the reference's `fusion_layer` (early_fusion_vit.py:75-79,123; early_fusion_vit_cnn.py:72-76,94):
 *     x = ReLU(BatchNorm2d(Conv2d(Cin, Cout, kernel_size=3, padding=1)(x)))        [ .flatten(2).transpose(1, 2) ]
 * as an implicit GEMM on the tensor cores.  The input is 16-bit channels-last, x: (B, H, W, Cin) fp16 (precision
 * P3P_PRECISION_FP16) or bf16 (P3P_PRECISION_BF16); p3p_encode / p3p_patch_embed write their halves of it directly
 * (out_layout P3P_LAYOUT_NLC with c_total = Cin and dtype P3P_DTYPE_F16 / BF16), p3p_nchw_to_nhwc16 converts an existing
 * fp32 NCHW tensor.  out: fp32, P3P_LAYOUT_NLC = token rows (B, H W, c_total) at channel c_offset (the flatten +
 * transpose of the reference is the store address), or P3P_LAYOUT_NCHW (B, c_total, H, W).
 * The same call with other sizes is the convolution of the `proj` tails (rank 5) behind p3p_upsample_bilinear_nhwc16.
 */
size_t p3p_conv3x3_blob_bytes(int32_t in_channels, int32_t out_channels);
int p3p_conv3x3_prepare(const p3p_conv_params* params, int32_t precision, void* blob, size_t blob_bytes, void* stream);
int p3p_conv3x3(const void* x, int32_t num_tiles, int32_t height, int32_t width, int32_t in_channels, const void* blob,
                int32_t out_channels, int32_t precision, int32_t relu, float* out, int32_t out_layout, int32_t c_total,
                int32_t c_offset, void* stream);

/*
 * The early-fusion ViT input in the same launch: p3p_conv3x3 (ReLU on) followed by what timm's
 * `VisionTransformer._pos_embed` does to the fusion layer's token rows in `EarlyFusionViT.forward`
 * (early_fusion_vit.py:123-124: `x = self.fusion_layer(x).flatten(2).transpose(1, 2)`, then `vit.forward_features(x)`
 * with `patch_embed = Identity`; one class token, no register tokens, `no_embed_class = False`):
 *   out[b, 0, :]       = cls_token + pos_embed[0, :]
 *   out[b, 1 + pos, :] = ReLU(BatchNorm2d(Conv2d(x)))[b, :, pos] + pos_embed[1 + pos, :]      pos = y W + x
 * out: (B, 1 + H W, Cout) fp32; cls_token: (Cout) fp32; pos_embed: (1 + H W, Cout) fp32, all on the device.  x, blob,
 * precision and the error codes as p3p_conv3x3; a null cls_token or pos_embed is P3P_ERR_INVALID_ARGUMENT.
 */
int p3p_conv3x3_vit_tokens(const void* x, int32_t num_tiles, int32_t height, int32_t width, int32_t in_channels, const void* blob,
                           int32_t out_channels, int32_t precision, const float* cls_token, const float* pos_embed, float* out,
                           void* stream);

/* fp32 NCHW (B, C, H, W) -> 16-bit channels-last (B, H, W, c_total) at channel offset c_offset. */
int p3p_nchw_to_nhwc16(const float* x, int32_t num_tiles, int32_t channels, int32_t height, int32_t width, int32_t precision,
                       void* out, int32_t c_total, int32_t c_offset, void* stream);

/*
 * nn.Upsample(size=(out_h, out_w), mode='bilinear', align_corners=False) of fp32 token rows x: (B, h w, C) with
 * src_batch_stride floats between tiles (the ViT output with its class token skipped; pointpillars_vit_cnn.py:31-36,
 * early_fusion_vit_cnn.py:97-102) into 16-bit channels-last out: (B, out_h, out_w, C), the input of p3p_conv3x3.
 */
int p3p_upsample_bilinear_nhwc16(const float* x, int32_t num_tiles, int32_t h, int32_t w, int32_t channels,
                                 int64_t src_batch_stride, int32_t out_h, int32_t out_w, int32_t precision, void* out, void* stream);

/*
 * PFN + scatter over the pillar table a p3p_voxelize call (same num_tiles / total_points, same stream) left in
 * `workspace`: the second half of p3p_encode, for callers that need the voxelizer's result for more than one pass
 * (the training step below).  Arguments as in p3p_encode.
 */
int p3p_encode_workspace(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const void* blob, int32_t channels,
                         int32_t precision, void* out, int32_t out_layout, int32_t out_dtype, int32_t c_total, int32_t c_offset,
                         void* workspace, size_t workspace_bytes, void* stream);

/*
 * SURVEY 8f rank 4 -- the training step of the PillarFeatureNet (`module.train()`): what autograd does through Open3D-ML's
 * PillarFeatureNet / PFNLayer x2 (call site pointpillars_o3d.py:93; DDP + SyncBatchNorm wrap
 * R:pixelspointspolygons/models/pix2poly/model_pix2poly.py:326-328), without any (V, M, *) tensor.  `params` carries the
 * RAW parameters (the norm*_mean / norm*_var pointers are ignored: the batch statistics live in `state`); `workspace` must
 * hold the pillar table of a p3p_voxelize call on the same batch and stay untouched until the backward has run.
 *
 * state: p3p_pfn_train_state_doubles(C, offsets) doubles on the device.  offsets[14] (in doubles) =
 *   { mom0, sums0, bn0, mom1, sums1, bn1, cen, back1, back1g, A1, kq, back0, back0g, A0 }.  The regions a multi-rank caller
 *   touches between the calls (SyncBatchNorm: one all-reduce(sum) each, SURVEY 8e):
 *     sums0  [65]      sum y0 (32), sum y0^2 (32), rows        after p3p_pfn_train_stats0
 *     sums1  [2C + 1]  sum y1 (C),  sum y1^2 (C),  rows        after p3p_pfn_train_stats1
 *     back1g [2C]      dbeta1, dgamma1: copy of back1 (this rank's sums), then all-reduced, before p3p_pfn_backward2
 *     back0g [64]      the same for layer 0 (copy of back0), before p3p_pfn_backward3
 *   A single-rank caller only does the two copies.
 *
 * forward:  p3p_pfn_train_stats0 -> [all-reduce sums0] -> p3p_pfn_train_stats1 -> [all-reduce sums1] ->
 *           p3p_pfn_train_forward (out: (B, ny nx, C) fp32 token rows, exact fp32; route: p3p_pfn_train_route_bytes bytes
 *           that carry the winning rows to the backward) and p3p_pfn_train_stats2 (batch mean / biased variance of both
 *           layers as fp32, for the running-statistics update; folded with p3p_pfn_prepare they also drive the inference
 *           kernels through p3p_encode_workspace when a tensor-core forward is preferred).
 * backward: p3p_pfn_backward1 (grad_out, out: (B, ny nx, C) fp32 rows, route as left by the forward) ->
 *           [back1g] -> p3p_pfn_backward2 -> [back0g] -> p3p_pfn_backward3 (gradients of the six parameters, fp32,
 *           this rank's share: DDP averages them as it does for the reference).
 * Covers every C <= 512 with every max_points <= 512.  Each entry refuses anything else with P3P_ERR_UNSUPPORTED and a
 * message naming the limit before it launches or writes anything (p3p_pfn_train_state_doubles returns 0 for such a C).
 * A batch without pillars is valid: zero output, zero gradients, batch mean and variance 0 with rows = 0.
 */
int64_t p3p_pfn_train_state_doubles(int32_t channels, int64_t* offsets);
size_t p3p_pfn_train_route_bytes(const p3p_grid* grid, int32_t num_tiles, int32_t channels);
int p3p_pfn_train_stats0(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                         double* state, void* workspace, size_t workspace_bytes, void* stream);
int p3p_pfn_train_stats1(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                         double* state, void* workspace, size_t workspace_bytes, void* stream);
int p3p_pfn_train_stats2(const p3p_pfn_params* params, double* state, float* mean0, float* var0, float* mean1, float* var1,
                         void* stream);
int p3p_pfn_train_forward(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                          double* state, float* out, void* route, void* workspace, size_t workspace_bytes, void* stream);
int p3p_pfn_backward1(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params, double* state,
                      const float* grad_out, const float* out, void* route, void* workspace, size_t workspace_bytes, void* stream);
int p3p_pfn_backward2(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params, double* state,
                      const void* route, void* workspace, size_t workspace_bytes, void* stream);
int p3p_pfn_backward3(const p3p_pfn_params* params, const double* state, float* d_linear0, float* d_norm0_weight,
                      float* d_norm0_bias, float* d_linear1, float* d_norm1_weight, float* d_norm1_bias, void* stream);

/*
 * Measurement hooks (bench.py's roofline leg; no reference counterpart).  Between begin and end every
 * p3p_encode call made by this thread records CUDA events around its two kernels on the caller's stream.
 * p3p_profile_end synchronises those events and returns, per recorded call, the milliseconds of the
 * voxelize kernel (incl. its counter memset) and of the PFN kernel (arrays of `capacity` floats, may be NULL).
 */
int p3p_profile_begin(int32_t max_records);
int p3p_profile_end(float* ms_voxelize, float* ms_pfn, int32_t capacity, int32_t* num_records);

#ifdef __cplusplus
}
#endif
#endif /* P3P_H_ */
