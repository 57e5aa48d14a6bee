// pfn.cu -- PillarFeatureNet (decorate + Linear/BN/ReLU/max x2) fused with the BEV scatter (sm_100a).
//
// Replaces `self.voxel_encoder(...)` + `self.middle_encoder(...)` of the reference
// (R:pixelspointspolygons/models/pointpillars/pointpillars_o3d.py:93-95; Open3D-ML PillarFeatureNet,
// PFNLayer, PointPillarsScatter; SURVEY 8a rows a6-a8, Appendix A.3-A.5) and, for the fusion encoders, the
// LiDAR half of `torch.cat((x_image, x_lidar), 1)` (R:.../fusion_layers/early_fusion_vit.py:121).
//
// Eval-mode closed form (Appendix A.4), a = gamma / sqrt(var + eps), b = beta - mean * a folded into the weights:
//   h_p   = relu(W0' d_p + b0)                      per kept point p (d_p: 8 decorated channels)
//   h_pad = relu(b0)                                every padded slot (present iff n < M)
//   hmax  = max over the M slots of h
//   o_p   = relu(W1a' h_p + W1b' hmax + b1),  out = max over the M slots of o
//         = relu(max_p(W1a' h_p) + W1b' hmax + b1)  (relu and "+ const" are monotone; the BN scale is already
//                                                    inside W1a', so its sign does not matter)
//
// pfn_tc_kernel (M <= 512 as 1 / 2 / 4 / 8 blocks of 64 rows per pillar, C <= 384): persistent warp-specialised pipeline,
// described at the kernel.  The decorated (V, M, 8) tensor and every (V, M, *) intermediate of the reference never exist
// in HBM.
//
// pfn_simt_kernel: exact fp32 FMA, literal 8-channel formulation, any M and C -- the GPU-side cross-check of the
// tensor-core path, the P3P_PRECISION_FP32 route, and the route for configurations the tensor-core kernel does not cover
// (M > 512, C > 384).  The training step (batch statistics, backward) lives in pfn_train.cu.
#include <cuda_fp16.h>

#include "p3p_internal.cuh"

namespace p3p {

// Optional pipeline timeline (build with -DP3P_TIMELINE): lane 0 of the MMA warp, of every front-end warp and of the
// first warp of every epilogue group stamps clock64 at its pipeline events; tools/pfn_timeline.py reads them back.
#ifdef P3P_TIMELINE
constexpr int kTlCtas = 4, kTlRoles = 12, kTlIters = 96, kTlStamps = 4;
__device__ long long g_pfn_tl[kTlCtas][kTlRoles][kTlIters][kTlStamps];
__device__ __forceinline__ void ptl(int role, long long it, int k) {
    if ((threadIdx.x & 31) == 0 && blockIdx.x < kTlCtas && it < kTlIters) g_pfn_tl[blockIdx.x][role][it][k] = clock64();
}
#define PTL(role, it, k) ptl(role, it, k)
extern "C" int p3p_debug_pfn_timeline(long long* host) {
    return (int)cudaMemcpyFromSymbol(host, g_pfn_tl, sizeof(g_pfn_tl));
}
#else
#define PTL(role, it, k)
#endif

void make_blob_layout(int C, BlobLayout* out) {
    BlobLayout l;
    l.C = C;
    l.Cpad = (C + 127) / 128 * 128;
    l.MT = l.Cpad / 128;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 1023) / 1024 * 1024;
        return o;
    };
    l.off_header = take(64);
    l.off_front = take(10 * 32 * 4);
    l.off_w0 = take(32 * 8 * 4);
    l.off_b0 = take(32 * 4);
    l.off_w1 = take((size_t)l.Cpad * 64 * 4);
    l.off_b1 = take((size_t)l.Cpad * 4);
    l.off_a1 = take((size_t)l.Cpad * 128);  // sized for tf32 rows (128 B); bf16 uses half
    l.off_a2 = take((size_t)l.Cpad * 128);
    l.total_bytes = off;
    *out = l;
}

namespace {

// ------------------------------------------------------------------------------------------------
// weight preparation
// ------------------------------------------------------------------------------------------------
__global__ void pfn_prepare_kernel(p3p_pfn_params p, int precision, char* blob, BlobLayout bl) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nthreads = gridDim.x * blockDim.x;
    int* header = reinterpret_cast<int*>(blob + bl.off_header);
    float* front = reinterpret_cast<float*>(blob + bl.off_front);
    float* w0 = reinterpret_cast<float*>(blob + bl.off_w0);
    float* b0 = reinterpret_cast<float*>(blob + bl.off_b0);
    float* w1 = reinterpret_cast<float*>(blob + bl.off_w1);
    float* b1 = reinterpret_cast<float*>(blob + bl.off_b1);
    if (tid == 0) {
        header[0] = kBlobMagic; header[1] = precision; header[2] = bl.C; header[3] = bl.Cpad; header[4] = p.center_alias;
    }
    for (int k = tid; k < kC0; k += nthreads) {
        const float a = p.norm0_weight[k] / sqrtf(p.norm0_var[k] + p.eps);
        const float sh = p.norm0_bias[k] - p.norm0_mean[k] * a;
        float w[8];
        for (int i = 0; i < 8; ++i) {
            w[i] = a * p.linear0_weight[k * 8 + i];
            w0[k * 8 + i] = w[i];
        }
        b0[k] = sh;
        // affine form: channels [c0, c1, z, x-mx, y-my, z-mz, x-cx, y-cy]; c0,c1 = (x-cx, y-cy) if alias else (x, y)
        front[0 * 32 + k] = w[0] + w[3] + w[6];          // Ux
        front[1 * 32 + k] = w[1] + w[4] + w[7];          // Uy
        front[2 * 32 + k] = w[2] + w[5];                 // Uz
        front[3 * 32 + k] = p.center_alias ? 0.f : w[0]; // Kcx (multiplies centre_x)
        front[4 * 32 + k] = p.center_alias ? 0.f : w[1]; // Kcy
        front[5 * 32 + k] = w[3];                        // Wmx (multiplies mean_x - centre_x)
        front[6 * 32 + k] = w[4];                        // Wmy
        front[7 * 32 + k] = w[5];                        // Wmz (multiplies mean_z)
        front[8 * 32 + k] = sh;                          // b0
        front[9 * 32 + k] = fmaxf(sh, 0.f);              // h_pad
        if (precision == P3P_PRECISION_TF32) {
            // kind::tf32 reads the upper 19 bits of each fp32 operand (truncation).  Layer 0 is positively homogeneous
            // (relu of an affine map), so scaling all of it by (1 + 2^-12) makes that truncation a round-to-nearest
            // of the unscaled h -- no conversion instruction per value in the kernel.
            const float up = 1.0f + 0x1p-12f;
            for (int r = 0; r < 10; ++r) front[r * 32 + k] *= up;
        }
    }
    const bool tf32 = (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16);
    for (int c = tid; c < bl.Cpad; c += nthreads) {
        float a = 0.f, sh = 0.f;
        if (c < bl.C) {
            a = p.norm1_weight[c] / sqrtf(p.norm1_var[c] + p.eps);
            sh = p.norm1_bias[c] - p.norm1_mean[c] * a;
        }
        b1[c] = sh;
        const int t = c >> 7, r = c & 127;
        for (int j = 0; j < 64; ++j) {
            const float v = (c < bl.C) ? a * p.linear1_weight[c * 64 + j] : 0.f;
            w1[c * 64 + j] = v;
            const int k = j & 31;
            char* tile = blob + (j < 32 ? bl.off_a1 : bl.off_a2);
            if (tf32) {
                const size_t o = (size_t)t * 16384 + (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 +
                                 (size_t)(((k >> 2) ^ (r & 7)) * 16) + (size_t)(k & 3) * 4;
                *reinterpret_cast<uint32_t*>(tile + o) = to_tf32(v);
            } else {
                const size_t o = (size_t)t * 8192 + (size_t)(r >> 3) * 512 + (size_t)(r & 7) * 64 +
                                 (size_t)(((k >> 3) ^ ((r >> 1) & 3)) * 16) + (size_t)(k & 7) * 2;
                *reinterpret_cast<unsigned short*>(tile + o) = (precision == P3P_PRECISION_FP16)
                                                                   ? __half_as_ushort(__float2half_rn(v))
                                                                   : (unsigned short)(pack_bf16(v, 0.f) & 0xFFFF);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// output addressing shared by both kernels
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_scalar(const PfnArgs& a, int64_t idx, float v) {
    if (a.out_dtype == P3P_DTYPE_F32) {
        static_cast<float*>(a.out)[idx] = v;
    } else {
        static_cast<unsigned short*>(a.out)[idx] = to_16bit(v, a.out_dtype);
    }
}
__device__ __forceinline__ int64_t out_index(const PfnArgs& a, int64_t item, int b, int cell, int c) {
    if (a.item_mode == kItemsCanvas && a.out_layout == P3P_LAYOUT_NCHW)
        return ((int64_t)b * a.c_total + a.c_offset + c) * a.items_per_tile + cell;
    return item * a.row_stride + a.row_offset + c;
}
// one output value of item (b, cell): plain layouts, or the token sequence (row 1 + cell of the tile, + pos_embed)
__device__ __forceinline__ void store_item(const PfnArgs& a, int64_t item, int b, int cell, int c, float v) {
    if (a.token_rows) {
        static_cast<float*>(a.out)[((int64_t)b * a.token_rows + 1 + cell) * a.bl.C + c] = v + a.pos_embed[(int64_t)(1 + cell) * a.bl.C + c];
        return;
    }
    store_scalar(a, out_index(a, item, b, cell, c), v);
}

// ------------------------------------------------------------------------------------------------
// exact fp32 kernel (literal formulation)
// ------------------------------------------------------------------------------------------------
constexpr int kSimtMaxThreads = 512;
constexpr int kHStride = 36;  // floats per H row: 16-byte aligned and bank-conflict free for float4 row stores

// One CTA per work item at a time, thread = output channel (blockDim = C rounded up to a warp, C <= 512): the channel's 64
// folded layer-1 weights stay in registers for every item of the CTA, the pillar's layer-0 rows sit in shared memory.
// kHoist = false (C > 512): threads loop over channels and re-read their weights per item.
template <bool kHoist>
__global__ void __launch_bounds__(kSimtMaxThreads) pfn_simt_kernel(PfnArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    float* H = smem_f;                                  // [(M + 1)][kHStride]
    float* w0s = H + (size_t)(a.g.M + 1) * kHStride;    // [32][8]
    float* b0s = w0s + 256;                             // [32]
    int* red = reinterpret_cast<int*>(b0s + 32);        // [16 warps][6] fixed-point partial sums
    int* hmax_bits = red + 96;                          // [32]

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nthreads = blockDim.x, nwarps = nthreads >> 5;
    const float* w0g = reinterpret_cast<const float*>(a.blob + a.bl.off_w0);
    const float* b0g = reinterpret_cast<const float*>(a.blob + a.bl.off_b0);
    const float* w1g = reinterpret_cast<const float*>(a.blob + a.bl.off_w1);
    const float* b1g = reinterpret_cast<const float*>(a.blob + a.bl.off_b1);
    const int alias = reinterpret_cast<const int*>(a.blob + a.bl.off_header)[4];
    for (int i = tid; i < 256; i += nthreads) w0s[i] = w0g[i];
    if (tid < 32) b0s[tid] = b0g[tid];
    const int C = a.bl.C, M = a.g.M;
    float wa[32], wb[32], b1c = 0.f;
    if (kHoist) {
        const int c = tid < C ? tid : 0;
        b1c = b1g[c];
#pragma unroll
        for (int k = 0; k < 32; ++k) { wa[k] = w1g[(size_t)c * 64 + k]; wb[k] = w1g[(size_t)c * 64 + 32 + k]; }
    }
    __syncthreads();

    for (int64_t item = blockIdx.x; item < a.num_items; item += gridDim.x) {
        const Item it = fetch_item(a, item);
        if (!it.valid) {
            if (a.item_mode == kItemsCanvas)
                for (int c = tid; c < C; c += nthreads) store_item(a, item, it.b, it.cell, c, 0.f);
            continue;
        }
        const float4* slot = item_slots(a, it);
        const int n = it.n;
        // cluster mean over the kept points (padded slots are zeros in the reference's sum), on the fixed-point grid
        int sl[3] = {0, 0, 0}, sh[3] = {0, 0, 0};
        for (int r = tid; r < n; r += nthreads) {
            const float4 p = slot[r];
            int lo, hi;
            fix_split(p.x, a.g.fix_scale, lo, hi); sl[0] += lo; sh[0] += hi;
            fix_split(p.y, a.g.fix_scale, lo, hi); sl[1] += lo; sh[1] += hi;
            fix_split(p.z, a.g.fix_scale, lo, hi); sl[2] += lo; sh[2] += hi;
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            sl[i] = __reduce_add_sync(0xffffffffu, sl[i]);
            sh[i] = __reduce_add_sync(0xffffffffu, sh[i]);
            if (lane == 0) { red[w * 6 + i] = sl[i]; red[w * 6 + 3 + i] = sh[i]; }
        }
        if (tid < 32) hmax_bits[tid] = 0;
        __syncthreads();
        int tl[3] = {0, 0, 0}, th[3] = {0, 0, 0};
        for (int ww = 0; ww < nwarps; ++ww) {
#pragma unroll
            for (int i = 0; i < 3; ++i) { tl[i] += red[ww * 6 + i]; th[i] += red[ww * 6 + 3 + i]; }
        }
        const float fn = (float)n;
        const float mx = fix_mean(tl[0], th[0], a.g.fix_inv, fn);
        const float my = fix_mean(tl[1], th[1], a.g.fix_inv, fn);
        const float mz = fix_mean(tl[2], th[2], a.g.fix_inv, fn);

        float hm[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) hm[k] = 0.f;
        bool any_row = false;
        for (int r = tid; r < n; r += nthreads) {
            any_row = true;
            const float4 p = slot[r];
            float d[8];
            const float xc = p.x - it.ctr_x, yc = p.y - it.ctr_y;
            d[0] = alias ? xc : p.x; d[1] = alias ? yc : p.y; d[2] = p.z;
            d[3] = p.x - mx; d[4] = p.y - my; d[5] = p.z - mz;
            d[6] = xc; d[7] = yc;
            float* hrow = H + (size_t)r * kHStride;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                float acc = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) acc = __fmaf_rn(w0s[k * 8 + i], d[i], acc);
                const float h = fmaxf(acc + b0s[k], 0.f);
                hrow[k] = h;
                hm[k] = fmaxf(hm[k], h);
            }
        }
        if (__any_sync(0xffffffffu, any_row)) {  // (warp-uniform) warps without a row have nothing to contribute
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const float v = warp_max_f32(hm[k]);
                if (lane == 0) atomicMax(&hmax_bits[k], __float_as_int(v));  // h >= 0: int order == float order
            }
        }
        if (n < M && tid < 32) {  // one representative padded slot: relu(BN(0))
            const float hp = fmaxf(b0s[tid], 0.f);
            H[(size_t)n * kHStride + tid] = hp;
            atomicMax(&hmax_bits[tid], __float_as_int(hp));
        }
        __syncthreads();
        const int rows = n + (n < M ? 1 : 0);
        if (kHoist) {
            if (tid < C) {
                float g = b1c;
#pragma unroll
                for (int k = 0; k < 32; ++k) g = __fmaf_rn(wb[k], __int_as_float(hmax_bits[k]), g);
                float best = -INFINITY;
                for (int r = 0; r < rows; ++r) {
                    const float4* hr = reinterpret_cast<const float4*>(H + (size_t)r * kHStride);
                    float acc = 0.f;
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 h = hr[k4];
                        acc = __fmaf_rn(wa[k4 * 4 + 0], h.x, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 1], h.y, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 2], h.z, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 3], h.w, acc);
                    }
                    best = fmaxf(best, acc);
                }
                store_item(a, item, it.b, it.cell, tid, fmaxf(best + g, 0.f));
            }
        } else {
            for (int c = tid; c < C; c += nthreads) {
                float g = b1g[c];
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    wa[k] = w1g[(size_t)c * 64 + k];
                    g = __fmaf_rn(w1g[(size_t)c * 64 + 32 + k], __int_as_float(hmax_bits[k]), g);
                }
                float best = -INFINITY;
                for (int r = 0; r < rows; ++r) {
                    const float4* hr = reinterpret_cast<const float4*>(H + (size_t)r * kHStride);
                    float acc = 0.f;
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 h = hr[k4];
                        acc = __fmaf_rn(wa[k4 * 4 + 0], h.x, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 1], h.y, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 2], h.z, acc);
                        acc = __fmaf_rn(wa[k4 * 4 + 3], h.w, acc);
                    }
                    best = fmaxf(best, acc);
                }
                store_item(a, item, it.b, it.cell, c, fmaxf(best + g, 0.f));
            }
        }
        __syncthreads();
    }
}

// class-token rows of the token sequence: tokens[b, 0, :] = cls_token + pos_embed[0, :]
__global__ void cls_rows_kernel(PfnArgs a, const float* __restrict__ cls_token) {
    const int C = a.bl.C;
    const int64_t total = (int64_t)a.B * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / C;
        const int c = (int)(i - b * C);
        static_cast<float*>(a.out)[b * a.token_rows * C + c] = cls_token[c] + a.pos_embed[c];
    }
}

__global__ void zero_lidar_kernel(PfnArgs a) {
    const int C = a.bl.C;
    const int64_t total = a.num_items * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t idx;
        if (a.out_layout == P3P_LAYOUT_NCHW) {
            const int64_t per_tile = (int64_t)C * a.items_per_tile;
            const int64_t b = i / per_tile, rem = i - b * per_tile;
            idx = (b * a.c_total + a.c_offset) * a.items_per_tile + rem;
        } else {
            const int64_t item = i / C;
            idx = item * a.row_stride + a.row_offset + (i - item * C);
        }
        store_scalar(a, idx, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------
// tensor-core kernel
// ------------------------------------------------------------------------------------------------
constexpr int kNF = 8;                         // front-end warps: warp w takes item w of every unit
constexpr int kMmaWarps = 4;                   // warp group 0: warp m < 3 issues the MMAs of channel tile m (warp 0 also owns the TMEM allocation), warp 3 idles
constexpr int kEpiWarp0 = kMmaWarps + kNF;     // then kNF front-end warps, then the epilogue warps
constexpr int kEpiGroups = 3;                  // epilogue groups of 4 warps (one warp per TMEM lane quarter)
constexpr int kTcThreads = 32 * (kEpiWarp0 + 4 * kEpiGroups);

constexpr int kRegMma = 40, kRegFront = 104, kRegEpi = 72;  // registers per thread after setmaxnreg (launch: 80)
// setmaxnreg redistributes the CTA's OWN launch allocation (24 warps x 80 registers), not the SM's spare registers: a split
// that exceeds it leaves the last warps spinning in the allocation forever
static_assert(4 * kRegMma + 8 * kRegFront + 12 * kRegEpi <= 24 * 80, "register pool of the launch exceeded");
constexpr int kUnit = 8;                       // items per unit = 4 pillar pairs, consecutive canvas cells
constexpr int kPairsPerUnit = kUnit / 2;
constexpr int kTiles = 3;                      // 128-channel MMA tiles (C <= 384)
constexpr int kAccCols = 64;                   // TMEM columns of one accumulator stage: one pillar (64 operand rows)
constexpr int kAccStages = 2;                  // accumulator stages per channel tile: the issuer refills one while the epilogue drains the other
constexpr int kGCol0 = kTiles * kAccStages * kAccCols;  // W1b' hmax of a unit: 2 slots (unit parity) x 3 tiles x 16 columns from 384 on
constexpr int kGSlotCols = kTiles * 16;
constexpr int kValidRing = 64;               // pairs of validity flags in flight between front end and epilogue (>= kNS + ring slack)
constexpr int kStageRows = 128;                // operand rows of a pair: 2 x 64 slots

template <int kPrec>
struct TcCfg {
    static constexpr bool kTf32 = (kPrec == P3P_PRECISION_TF32);
    static constexpr int kFmt = kTf32 ? 2 : (kPrec == P3P_PRECISION_BF16 ? 1 : 0);  // UMMA operand format code
    static constexpr int RB = kTf32 ? 128 : 64;           // bytes of one K = 32 operand row
    static constexpr int kATile = 128 * RB;               // 128 channels
    static constexpr int kHStage = kStageRows * RB;       // 2 pillars x 64 rows
    static constexpr int kGStage = 16 * RB;               // hmax rows of the 8 items of a unit (padded to 16)
    static constexpr uint32_t kLayout = kTf32 ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
    static constexpr uint32_t kSBO = 8 * RB;
    static constexpr int kKSteps = kTf32 ? 4 : 2;         // UMMA_K = 8 (tf32) / 16 (16-bit): 32 bytes per step
    static constexpr int kNS = kTf32 ? 4 : 8;             // B-operand stages: pillar pairs in flight
    static constexpr size_t kSmemOperands = (size_t)6 * kATile + (size_t)kNS * kHStage + 2 * (size_t)kGStage;
    static constexpr size_t kSmemFloats = 10 * 32 + 384 + kNF * 128 * 4;
    static constexpr size_t kSmemBytes = kSmemOperands + kSmemFloats * 4 + (2 * kNS + 2 * kTiles * kAccStages + 4 * kTiles + 2 + 2) * 8 + 16 + 2 * kNF * 4 + 2 * kValidRing + 4 * kEpiGroups * kUnit * 32 * 4 + 2 * kNF * 4 * 4 + 2 * kNF * 32 * 4;
};


// two fp32 -> packed 16-bit pair with relu fused into the conversion (lo = first channel)
template <int kPrec>
__device__ __forceinline__ uint32_t pack_relu16(float lo, float hi) {
    uint32_t r;
    if constexpr (kPrec == P3P_PRECISION_BF16)
        asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else
        asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
template <int kPrec>
__device__ __forceinline__ uint32_t max16x2(uint32_t a, uint32_t b) {
    uint32_t r;
    if constexpr (kPrec == P3P_PRECISION_BF16)
        asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    else
        asm("max.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// 16-byte global -> shared copy, zero-filled when src_bytes == 0
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
template <int kRegs>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs)); }
template <int kRegs>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs)); }
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// running (tile, position) of an item index that advances by a fixed stride: divisions at start-up only
struct ItemWalk {
    int b, r, ipt, db, dr;
    __device__ __forceinline__ void init(int item, int delta, int items_per_tile) {
        ipt = items_per_tile;
        b = item / ipt; r = item - b * ipt;
        db = delta / ipt; dr = delta - db * ipt;
    }
    __device__ __forceinline__ void step() {
        b += db; r += dr;
        if (r >= ipt) { r -= ipt; ++b; }
    }
};

__device__ __forceinline__ void tmem_ld8_wait(uint32_t taddr, float (&v)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ float max16(const float (&v)[16]) {
    float r[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) r[i] = fmax3(v[3 * i], v[3 * i + 1], v[3 * i + 2]);
    return fmax3(fmax3(r[0], r[1], r[2]), fmaxf(r[3], r[4]), v[15]);
}
// the same with a running maximum folded in: 17 values, still 8 three-input maxima
__device__ __forceinline__ float max16_with(float prev, const float (&v)[16]) {
    const float r0 = fmax3(prev, v[0], v[1]), r1 = fmax3(v[2], v[3], v[4]), r2 = fmax3(v[5], v[6], v[7]);
    const float r3 = fmax3(v[8], v[9], v[10]), r4 = fmax3(v[11], v[12], v[13]);
    return fmax3(fmax3(r0, r1, r2), fmax3(r3, r4, v[14]), v[15]);
}
// pfn_tc_kernel (C <= 384; M <= 64 per 64-row block, larger M as 2 / 4 / 8 blocks in mode 0): per CTA a persistent pipeline
//   8 front-end warps  : warp w takes item w of every unit (8 consecutive items); layer 0 in its affine form
//                        W0' d_p + b0 = Ux x' + Uy y' + Uz z + kappa(pillar)   (x' = x - centre_x, ...)
//                        -> 3 FMA per (point, channel); 16-byte row chunks written (tf32 / 16-bit) straight into the
//                        swizzled K-major B-operand stage of the pair, hmax into the stage's two extra rows
//   3 MMA warps        : warp m, per pair: D[128 ch x 128 pts] = W1a'[tile m] H^T into accumulator stage m; per unit
//                        (8 items): D[128 ch x 16] = W1b'[tile m] hmax^T into the stage's 16 spare columns
//   3 x 4 epilogue warps: group g reads accumulator stage g: tcgen05.ld, max over each
//                        pillar's 64 columns with 3-input max, + W1b' hmax + b1, relu, store of the two cells.
// kMode: 0 = any item source / layout / dtype (run-time branches); 1 = canvas items, whole units inside one tile, fp32 rows
// of C channels (B, ny nx, C); 2 = the same into the fp32 NCHW (concat) buffer; 3 = the same as token rows 1 + cell of a
// (B, 1 + ny nx, C) sequence with pos_embed added.  Modes 1-3 are the shipped encoder configurations with every run-time
// branch of the steady-state loops resolved at compile time.
template <int kPrec, int kMode>
__global__ void __launch_bounds__(kTcThreads, 1) pfn_tc_kernel(PfnArgs a) {
    using Cfg = TcCfg<kPrec>;
    constexpr bool kTf32 = Cfg::kTf32;
    constexpr int kNS = Cfg::kNS;
    // The kernel has no static shared memory, so the dynamic block starts at shared-memory offset 0 of the CTA window and
    // the declared alignment holds (checked below): every shared address below is a compile-time offset.
    extern __shared__ __align__(1024) unsigned char smem_dyn[];
    unsigned char* base = smem_dyn;
    unsigned char* sA1 = base;
    unsigned char* sA2 = sA1 + 3 * Cfg::kATile;
    unsigned char* sH = sA2 + 3 * Cfg::kATile;                          // [kNS][128 rows]
    unsigned char* sG = sH + kNS * Cfg::kHStage;                        // [2 unit slots][16 rows]: hmax rows of a unit's 8 items
    float* sFront = reinterpret_cast<float*>(sG + 2 * Cfg::kGStage);    // [10][32]
    float* sB1 = sFront + 10 * 32;                                      // [384]
    float4* sPts = reinterpret_cast<float4*>(sB1 + 384);                // [kNF][2 sets][64] points of the pillar in work / of the next one
    uint64_t* bars = reinterpret_cast<uint64_t*>(sPts + kNF * 128);
    uint64_t* h_full = bars;                  // [kNS] front end -> MMA (2 arrivals: the two warps of a pair)
    uint64_t* h_empty = bars + kNS;           // [kNS] MMA -> front end (one tcgen05.commit per channel tile)
    uint64_t* t_full = bars + 2 * kNS;                  // [3 tiles][2 stages] MMA warp m -> epilogue group m (tcgen05.commit), per pillar
    uint64_t* t_empty = t_full + kTiles * kAccStages;   // [3][2] epilogue group m -> MMA warp m (128 arrivals)
    uint64_t* gt_full = t_empty + kTiles * kAccStages;  // [3 tiles][2 slots] MMA warp m -> epilogue group m, per unit (W1b' hmax accumulator)
    uint64_t* gt_empty = gt_full + 2 * kTiles;          // [3][2] epilogue group m -> MMA warp m (128 arrivals)
    uint64_t* g_empty = gt_empty + 2 * kTiles;          // [2] MMA warps -> front end: hmax rows of the unit slot consumed (MT commits)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(g_empty + 2);
    int* sDesc = reinterpret_cast<int*>(tmem_slot + 2);                 // [kNF][2] descriptor word of the item decoded next
    unsigned char* sValid = reinterpret_cast<unsigned char*>(sDesc + 2 * kNF);  // [kValidRing pairs][2]: the item holds a pillar
    float* sRmax = reinterpret_cast<float*>(sValid + 2 * kValidRing);           // [12 epilogue warps][kUnit][32]: pillar maxima of the unit in work
    int* sBlkSum = reinterpret_cast<int*>(sRmax + 4 * kEpiGroups * kUnit * 32);  // [2 unit parities][kNF][4] fixed-point sums of a block
    uint32_t* sBlkMax = reinterpret_cast<uint32_t*>(sBlkSum + 2 * kNF * 4);          // [2][kNF][32] hmax of a block (32 words: fp32, or 16 packed)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int MT = a.bl.MT;
    const int total_items = (int)a.num_items;
    // M > 64 (density ablation, general mode only): a pillar = 2 / 4 / 8 consecutive 64-row blocks of a unit; its cluster
    // mean and hmax are merged across the blocks' front-end warps, its maximum across the blocks in the epilogue
    const int bs = (kMode == 0) ? a.blk_shift : 0;  // log2(blocks per pillar)
    const int num_units = ((total_items << bs) + kUnit - 1) / kUnit;
    const int my_units = (num_units > (int)blockIdx.x) ? (num_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int my_pairs = my_units * kPairsPerUnit;  // pairs this CTA processes, in order p = 0, 1, ...
    const bool canvas = (kMode != 0) || (a.item_mode == kItemsCanvas);

    // ---- one-time setup --------------------------------------------------------------------------
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();  // the swizzled operand tiles need 1024-byte alignment
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 32) {
        for (int i = 0; i < kNS; ++i) { mbar_init(&h_full[i], 2); mbar_init(&h_empty[i], (uint32_t)MT); }
        for (int i = 0; i < kTiles * kAccStages; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 128); }
        for (int i = 0; i < 2 * kTiles; ++i) { mbar_init(&gt_full[i], 1); mbar_init(&gt_empty[i], 128); }
        mbar_init(&g_empty[0], (uint32_t)MT); mbar_init(&g_empty[1], (uint32_t)MT);
        fence_mbar_init();
    }
    {
        const uint4* g1 = reinterpret_cast<const uint4*>(a.blob + a.bl.off_a1);
        const uint4* g2 = reinterpret_cast<const uint4*>(a.blob + a.bl.off_a2);
        const int nvec = MT * Cfg::kATile / 16;
        for (int i = tid; i < nvec; i += kTcThreads) {
            reinterpret_cast<uint4*>(sA1)[i] = g1[i];
            reinterpret_cast<uint4*>(sA2)[i] = g2[i];
        }
        // rows 8..15 of the hmax blocks feed accumulator columns nobody reads; zero the blocks once all the same
        for (int i = tid; i < 2 * Cfg::kGStage / 16; i += kTcThreads) reinterpret_cast<uint4*>(sG)[i] = make_uint4(0, 0, 0, 0);
        const float* fg = reinterpret_cast<const float*>(a.blob + a.bl.off_front);
        const float* b1g = reinterpret_cast<const float*>(a.blob + a.bl.off_b1);
        for (int i = tid; i < 10 * 32; i += kTcThreads) sFront[i] = fg[i];
        for (int i = tid; i < 384; i += kTcThreads) sB1[i] = (i < a.bl.Cpad) ? b1g[i] : 0.f;
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above reads only the prepared weights; the voxelizer's tables and slots are read from here on
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // Register budget per role (warp groups of 4 warps): the launch allots 80 registers per thread; the issuers and the
    // epilogue hand registers back, the front end (long independent FMA chains) takes them.  Measured splits
    // (MMA / front / epilogue -> fp16, tf32 kernel time), per-pair W1b'hmax MMA: 40/112/72 -> 43.3, 68.9 us; 40/120/64 ->
    // 43.9, 52.4 us; 40/136/56 -> 44.6, 53.1 us; 24/104/80 -> 78.6, 55.2 us (the issuers spill below 32); no reallocation
    // -> 47.1, 56.4 us.  With the per-unit W1b'hmax MMA (the epilogue holds a unit's 8 maxima): 40/120/64 -> 45.0, 52.2 us;
    // 40/112/72 -> 39.6, 50.9 us; 40/104/72 -> 38.6, 49.0 us; 40/96/80 -> 66.9, 85.7 us (the front end spills below 104).
    if (warp < kMmaWarps) {
        setmaxnreg_dec<kRegMma>();
        // =========================== MMA issuers: warp m owns channel tile m and accumulator stage m ===========================
        // The whole warp walks the loop (warp-uniform control flow keeps descriptors in uniform registers); one elected
        // lane issues the tcgen05 instructions and their commits.  One issuing warp per tile keeps the per-pair chain of
        // barrier waits (about 100 cycles each, even when already satisfied) short.
        const int m = warp;
        if (m < MT) {
            const bool leader = elect_one();
            const uint32_t idesc_main = make_idesc(Cfg::kFmt, 128, kAccCols);
            const uint32_t idesc_g = make_idesc(Cfg::kFmt, 128, 16);
            const uint32_t desc_hi = (Cfg::kSBO >> 4) | (1u << 14) | (Cfg::kLayout << 29);
            const uint32_t a1_lo = ((smem_u32(sA1) + (uint32_t)(m * Cfg::kATile)) >> 4) | (1u << 16);
            const uint32_t a2_lo = ((smem_u32(sA2) + (uint32_t)(m * Cfg::kATile)) >> 4) | (1u << 16);
            const uint32_t h_lo = (smem_u32(sH) >> 4) | (1u << 16), g_lo = (smem_u32(sG) >> 4) | (1u << 16);
            const uint32_t d_tile = tmem_base + (uint32_t)(m * kAccStages * kAccCols);
            const uint32_t d_g = tmem_base + (uint32_t)(kGCol0 + m * 16);  // + kGSlotCols * (unit parity)
            uint64_t* tf = t_full + m * kAccStages;
            uint64_t* te = t_empty + m * kAccStages;
            int st = 0;
            uint32_t use = 0;
            for (int p = 0; p < my_pairs; ++p) {
                mbar_wait(&h_full[st], use & 1);
                if (m == 0) PTL(0, p, 0);
                const uint32_t hs_lo = h_lo + (uint32_t)st * (Cfg::kHStage >> 4);
                // the pair's two pillars go to the tile's two accumulator stages: while the epilogue drains stage 1 of pair
                // p - 1, stage 0 is already being refilled with pillar A of pair p
#pragma unroll
                for (int s = 0; s < kAccStages; ++s) {
                    mbar_wait(&te[s], ((uint32_t)p & 1u) ^ 1u);
                    if (m == 0 && s == 0) PTL(0, p, 1);
                    tc_fence_after();
                    if (leader) {
                        const uint32_t b_lo = hs_lo + (uint32_t)(s * ((64 * Cfg::RB) >> 4));  // rows 64 s .. 64 s + 63 of the stage
#pragma unroll
                        for (int k = 0; k < Cfg::kKSteps; ++k)
                            tc_mma<kTf32>(d_tile + (uint32_t)(s * kAccCols), ((uint64_t)desc_hi << 32) | (a1_lo + (uint32_t)(k * 2)),
                                          ((uint64_t)desc_hi << 32) | (b_lo + (uint32_t)(k * 2)), idesc_main, k > 0);
                        tc_commit(&tf[s]);
                    }
                    __syncwarp();
                }
                if (leader) tc_commit(&h_empty[st]);
                __syncwarp();
                if (m == 0) PTL(0, p, 2);
                if (++st == kNS) { st = 0; ++use; }
                // ---- end of a unit (all 8 hmax rows are written: its 4 pairs have arrived): W1b' hmax of the 8 items
                //      with one N = 16 MMA chain into the tile's 16 spare accumulator columns -----------------------------
                if ((p & (kPairsPerUnit - 1)) == kPairsPerUnit - 1) {
                    const uint32_t j = (uint32_t)p / kPairsPerUnit, slot = j & 1u;
                    mbar_wait(&gt_empty[m * 2 + slot], ((j >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    if (leader) {
                        const uint32_t gs_lo = g_lo + slot * (Cfg::kGStage >> 4);
#pragma unroll
                        for (int k = 0; k < Cfg::kKSteps; ++k)
                            tc_mma<kTf32>(d_g + slot * kGSlotCols, ((uint64_t)desc_hi << 32) | (a2_lo + (uint32_t)(k * 2)),
                                          ((uint64_t)desc_hi << 32) | (gs_lo + (uint32_t)(k * 2)), idesc_g, k > 0);
                        tc_commit(&gt_full[m * 2 + slot]);
                        tc_commit(&g_empty[slot]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp < kEpiWarp0) {
        // =========================== front end: warp fw takes item fw of every unit ===========================
        // lane = (channel octet o, point pt): 8 independent combos per lane, combo i = slot pt + 8 i of the pillar x the
        // lane's 8 channels (one 16-byte chunk of a 16-bit operand row, two chunks of a tf32 row).  The pillar's points
        // arrive by cp.async (zero-filled beyond n) into a per-warp double buffer one item ahead; the descriptor word is
        // loaded two items ahead and decoded one iteration later; the channel constants of layer 0 sit in registers.
        setmaxnreg_inc<kRegFront>();
        const int fw = warp - kMmaWarps, half = fw & 1, pr = fw >> 1;
        const int o = lane & 3, pt = lane >> 2;
        float2 ux[4], uy[4], uz[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            ux[i] = *reinterpret_cast<const float2*>(sFront + 0 * 32 + 8 * o + 2 * i);
            uy[i] = *reinterpret_cast<const float2*>(sFront + 1 * 32 + 8 * o + 2 * i);
            uz[i] = *reinterpret_cast<const float2*>(sFront + 2 * 32 + 8 * o + 2 * i);
        }
        const float* kc = sFront + 8 * o;  // row 9 (relu(b0) of a padded slot) of the lane's 8 channels
        // rows 3..8 of channel `lane`: the per-pillar constant kappa is computed one channel per lane
        const float k_cx = sFront[3 * 32 + lane], k_cy = sFront[4 * 32 + lane], k_mx = sFront[5 * 32 + lane];
        const float k_my = sFront[6 * 32 + lane], k_mz = sFront[7 * 32 + lane], k_b0 = sFront[8 * 32 + lane];
        float4* pbuf = sPts + fw * 128;    // [2 sets][64]
        const uint32_t pbuf_sa = smem_u32(pbuf);
        // byte offset of the lane's first slot inside a stage: row (half * 64 + pt), the lane's chunk(s) under the swizzle
        uint32_t row_off[2];
        if constexpr (kTf32) {
            row_off[0] = (uint32_t)(half * 64 + pt) * Cfg::RB + (uint32_t)(((2 * o) ^ pt) * 16);
            row_off[1] = (uint32_t)(half * 64 + pt) * Cfg::RB + (uint32_t)(((2 * o + 1) ^ pt) * 16);
        } else {
            row_off[0] = (uint32_t)(half * 64 + pt) * Cfg::RB + (uint32_t)((o ^ ((pt >> 1) & 3)) * 16);
            row_off[1] = 0;
        }
        // hmax row fw of the unit's block of 16 rows, the lane's chunk(s) under the swizzle
        const uint32_t g_off0 = (uint32_t)fw * Cfg::RB + (uint32_t)(kTf32 ? (((2 * o) ^ (fw & 7)) * 16) : ((o ^ ((fw >> 1) & 3)) * 16));
        const uint32_t g_off1 = (uint32_t)fw * Cfg::RB + (uint32_t)(((2 * o + 1) ^ (fw & 7)) * 16);
        const float inv_nx = 1.0f / (float)a.g.nx;
        const int kblk = fw & ((1 << bs) - 1), row0 = kblk * 64;  // this warp's block of its pillar: slots [row0, row0 + 64)
        auto item_of = [&](int j) -> int {
            const int it = (((int)blockIdx.x + j * (int)gridDim.x) * kUnit + fw) >> bs;
            return (j < my_units && it < total_items) ? it : total_items;
        };
        // rows of this warp's block that hold points, and whether the block takes part: it holds points, or it is the first
        // empty block of a pillar with n < M whose blocks are all full (the padded slot of the reference lives there)
        auto block_rows = [&](const Item& it) -> int {
            const int r = it.n - row0;
            return r < 0 ? 0 : (r > 64 ? 64 : r);
        };
        auto block_valid = [&](const Item& it) -> bool {
            return it.valid && (bs == 0 || it.n > row0 || (it.n == row0 && it.n < a.g.M));
        };
        // descriptor word of item j (canvas: cell_desc; list: resolved when decoded) travels through shared memory by
        // cp.async like the points, so no register waits on a global load
        int* my_desc = sDesc + 2 * fw;
        const uint32_t my_desc_sa = smem_u32(my_desc);
        auto prefetch_desc = [&](int j) {
            const int item = item_of(j);
            if (lane == 0) {
                if (canvas && item < total_items) cp_async4(my_desc_sa + 4u * (uint32_t)(j & 1), a.ws.cell_desc + item);
                else my_desc[j & 1] = -1;
            }
        };
        ItemWalk wk;  // position of the item decoded next
        wk.init(item_of(0) < total_items ? item_of(0) : 0, ((int)gridDim.x * kUnit) >> bs, a.items_per_tile);
        auto decode = [&](int j, int d) -> Item {
            Item it;
            if (!canvas) {
                it = fetch_item(a, item_of(j));
            } else {
                it.valid = d >= 0 ? 1 : 0;
                it.b = wk.b; it.cell = wk.r;
                it.key = d & 0xFFFF; it.n = d >> 16;
                const int cy = __float2int_rz(((float)wk.r + 0.5f) * inv_nx), cx = wk.r - cy * a.g.nx;
                it.ctr_x = __fmaf_rn((float)cx, a.g.vx, a.g.x_off);
                it.ctr_y = __fmaf_rn((float)cy, a.g.vy, a.g.y_off);
            }
            wk.step();
            return it;
        };
        auto prefetch_points = [&](const Item& it, int set) {
            if (block_valid(it)) {
                const float4* sl = item_slots(a, it) + row0;
                const int nr = block_rows(it);
                const uint32_t dst = pbuf_sa + (uint32_t)set * 1024u + (uint32_t)lane * 16u;
                cp_async16(dst, sl + lane, lane < nr ? 16u : 0u);
                cp_async16(dst + 512u, sl + lane + 32, lane + 32 < nr ? 16u : 0u);
            }
        };
        prefetch_desc(0);
        cp_async_wait_all();
        __syncwarp();
        Item it_cur = decode(0, my_desc[0]);
        __syncwarp();
        prefetch_points(it_cur, 0);
        prefetch_desc(1);
        for (int j = 0; j < my_units; ++j) {
            const Item it = it_cur;
            cp_async_wait_all();
            __syncwarp();  // points of item j and descriptor of item j + 1 visible to every lane; the other buffers are free
            it_cur = decode(j + 1, my_desc[(j + 1) & 1]);
            __syncwarp();
            prefetch_points(it_cur, (j + 1) & 1);
            prefetch_desc(j + 2);

            const int p = j * kPairsPerUnit + pr, st = p % kNS;
            const uint32_t use = (uint32_t)(p / kNS);
            PTL(1 + fw, j, 0);
            mbar_wait(&h_empty[st], (use & 1u) ^ 1u);
            mbar_wait(&g_empty[j & 1], (((uint32_t)j >> 1) & 1u) ^ 1u);  // the unit slot's hmax rows of two units ago are consumed
            PTL(1 + fw, j, 1);
            const uint32_t gslot_sa = smem_u32(sG) + (uint32_t)(j & 1) * Cfg::kGStage;
            const bool bvalid = block_valid(it);
            const float4* P = pbuf + (j & 1) * 64;
            uint32_t hm[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};  // M > 64: this block's hmax (8 fp32 channels, or 8 packed in 4 words)
            // cluster mean on the fixed-point grid (exact integer sums: independent of the order of the slots); rows beyond
            // the block's points are zero-filled by the copy.  |q| * M slots < 2^31 (fix2_scale is sized for M).
            int sx = 0, sy = 0, sz = 0;
            if (bvalid) {
                const float4 s0 = P[lane], s1 = P[lane + 32];
                const float fs = a.g.fix2_scale;
                sx = __reduce_add_sync(0xffffffffu, __float2int_rn(s0.x * fs) + __float2int_rn(s1.x * fs));
                sy = __reduce_add_sync(0xffffffffu, __float2int_rn(s0.y * fs) + __float2int_rn(s1.y * fs));
                sz = __reduce_add_sync(0xffffffffu, __float2int_rn(s0.z * fs) + __float2int_rn(s1.z * fs));
            }
            if (bs) {  // the pillar's sums = the sums of its blocks (the blocks' warps meet at a named barrier)
                int* mine = sBlkSum + ((j & 1) * kNF + fw) * 4;
                if (lane == 0) { mine[0] = sx; mine[1] = sy; mine[2] = sz; }
                asm volatile("bar.sync %0, %1;" ::"r"(1 + (fw >> bs)), "r"(32 << bs) : "memory");
                const int* first = sBlkSum + ((j & 1) * kNF + (fw - kblk)) * 4;
                sx = sy = sz = 0;
                for (int k = 0; k < (1 << bs); ++k) { sx += first[4 * k]; sy += first[4 * k + 1]; sz += first[4 * k + 2]; }
            }
            if (bvalid) {
                const int n = block_rows(it);   // rows of this block that hold points
                const int n_all = it.n;         // points of the pillar
                float mpx, mpy, mz;
                {
                    const float wn = __fdividef(a.g.fix2_inv, (float)n_all);
                    mpx = (float)sx * wn - it.ctr_x;
                    mpy = (float)sy * wn - it.ctr_y;
                    mz = (float)sz * wn;
                }
                float qx[8], qy[8], qz[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 q = P[pt + 8 * i];
                    qx[i] = q.x - it.ctr_x; qy[i] = q.y - it.ctr_y; qz[i] = q.z;
                }
                // per-pillar constant of channel `lane` (one channel per lane), then the lane's 8 channels by shuffle
                float2 kap[4];
                {
                    float kl = __fmaf_rn(k_cx, it.ctr_x, k_b0);
                    kl = __fmaf_rn(k_cy, it.ctr_y, kl);
                    kl = __fmaf_rn(k_mx, -mpx, kl);
                    kl = __fmaf_rn(k_my, -mpy, kl);
                    kl = __fmaf_rn(k_mz, -mz, kl);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        kap[i] = make_float2(__shfl_sync(0xffffffffu, kl, 8 * o + 2 * i), __shfl_sync(0xffffffffu, kl, 8 * o + 2 * i + 1));
                }
                const uint32_t stage_sa = smem_u32(sH) + (uint32_t)st * Cfg::kHStage;
                if constexpr (kTf32) {
                    // rows beyond the pillar's n points: relu(BN(0)) of a padded slot while n < M; when the pillar is
                    // full at M < 64 the reference has no padded slot, the spare rows repeat slot 0 (the max ignores them)
                    float hp[8], mx8[8];
                    if (n_all < a.g.M || n == 64) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) hp[c] = kc[9 * 32 + c];
                    } else {
                        const float4 q0 = P[0];
                        const float x0 = q0.x - it.ctr_x, y0 = q0.y - it.ctr_y, z0 = q0.z;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float2 v = ffma2(ux[c], make_float2(x0, x0), ffma2(uy[c], make_float2(y0, y0), ffma2(uz[c], make_float2(z0, z0), kap[c])));
                            hp[2 * c] = fmaxf(v.x, 0.f); hp[2 * c + 1] = fmaxf(v.y, 0.f);
                        }
                    }
#pragma unroll
                    for (int c = 0; c < 8; ++c) mx8[c] = (n < 64) ? hp[c] : 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float h[8];
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float2 v = ffma2(ux[c], make_float2(qx[i], qx[i]), ffma2(uy[c], make_float2(qy[i], qy[i]), ffma2(uz[c], make_float2(qz[i], qz[i]), kap[c])));
                            h[2 * c] = fmaxf(v.x, 0.f); h[2 * c + 1] = fmaxf(v.y, 0.f);
                        }
                        if (pt + 8 * i >= n) {  // padded slots carry relu(BN(0))
#pragma unroll
                            for (int c = 0; c < 8; ++c) h[c] = hp[c];
                        }
#pragma unroll
                        for (int c = 0; c < 8; ++c) mx8[c] = fmaxf(mx8[c], h[c]);
                        // operands are already scaled by (1 + 2^-12): the MMA's truncation rounds them to nearest tf32
                        sts128(stage_sa + row_off[0] + (uint32_t)i * (8u * Cfg::RB), __float_as_uint(h[0]), __float_as_uint(h[1]), __float_as_uint(h[2]), __float_as_uint(h[3]));
                        sts128(stage_sa + row_off[1] + (uint32_t)i * (8u * Cfg::RB), __float_as_uint(h[4]), __float_as_uint(h[5]), __float_as_uint(h[6]), __float_as_uint(h[7]));
                    }
#pragma unroll
                    for (int off = 4; off < 32; off <<= 1) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) mx8[c] = fmaxf(mx8[c], __shfl_xor_sync(0xffffffffu, mx8[c], off));
                    }
                    if (bs) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) hm[c] = __float_as_uint(mx8[c]);
                    } else if (pt == 0) {
                        sts128(gslot_sa + g_off0, __float_as_uint(mx8[0]), __float_as_uint(mx8[1]), __float_as_uint(mx8[2]), __float_as_uint(mx8[3]));
                        sts128(gslot_sa + g_off1, __float_as_uint(mx8[4]), __float_as_uint(mx8[5]), __float_as_uint(mx8[6]), __float_as_uint(mx8[7]));
                    }
                } else {
                    uint32_t mm[4] = {0u, 0u, 0u, 0u};
                    if (n == 64) {  // (warp-uniform) full pillar: no padded slots
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            uint32_t h[4];
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const float2 v = ffma2(ux[c], make_float2(qx[i], qx[i]), ffma2(uy[c], make_float2(qy[i], qy[i]), ffma2(uz[c], make_float2(qz[i], qz[i]), kap[c])));
                                h[c] = pack_relu16<kPrec>(v.x, v.y);
                                mm[c] = max16x2<kPrec>(mm[c], h[c]);
                            }
                            sts128(stage_sa + row_off[0] + (uint32_t)i * (8u * Cfg::RB), h[0], h[1], h[2], h[3]);
                        }
                    } else {
                        // rows beyond the pillar's n points: relu(BN(0)) of a padded slot while n < M; when the pillar
                        // is full at M < 64 the reference has no padded slot, the spare rows repeat slot 0
                        uint32_t hp[4];
                        if (n_all < a.g.M) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) hp[c] = pack_relu16<kPrec>(kc[9 * 32 + 2 * c], kc[9 * 32 + 2 * c + 1]);
                        } else {
                            const float4 q0 = P[0];
                            const float x0 = q0.x - it.ctr_x, y0 = q0.y - it.ctr_y, z0 = q0.z;
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const float2 v = ffma2(ux[c], make_float2(x0, x0), ffma2(uy[c], make_float2(y0, y0), ffma2(uz[c], make_float2(z0, z0), kap[c])));
                                hp[c] = pack_relu16<kPrec>(v.x, v.y);
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            uint32_t h[4];
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const float2 v = ffma2(ux[c], make_float2(qx[i], qx[i]), ffma2(uy[c], make_float2(qy[i], qy[i]), ffma2(uz[c], make_float2(qz[i], qz[i]), kap[c])));
                                h[c] = pack_relu16<kPrec>(v.x, v.y);
                                if (pt + 8 * i >= n) h[c] = hp[c];  // padded slots carry relu(BN(0))
                                mm[c] = max16x2<kPrec>(mm[c], h[c]);
                            }
                            sts128(stage_sa + row_off[0] + (uint32_t)i * (8u * Cfg::RB), h[0], h[1], h[2], h[3]);
                        }
                    }
#pragma unroll
                    for (int off = 4; off < 32; off <<= 1) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) mm[c] = max16x2<kPrec>(mm[c], __shfl_xor_sync(0xffffffffu, mm[c], off));
                    }
                    if (bs) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) hm[c] = mm[c];
                    } else if (pt == 0) {
                        sts128(gslot_sa + g_off0, mm[0], mm[1], mm[2], mm[3]);
                    }
                }
            }
            if (bs) {
                // hmax of the pillar = max over its blocks (h >= 0: an absent block contributes zeros); every block's warp
                // writes the merged row as ITS hmax row of the unit, so the W1b' hmax MMA needs no notion of pillars
                constexpr int kW = kTf32 ? 8 : 4;  // words per lane: 8 fp32 channels, or 8 channels packed in 4
                uint32_t* mine = sBlkMax + ((j & 1) * kNF + fw) * 32 + kW * o;
                if (pt == 0) {
#pragma unroll
                    for (int c = 0; c < kW; ++c) mine[c] = hm[c];
                }
                asm volatile("bar.sync %0, %1;" ::"r"(1 + (fw >> bs)), "r"(32 << bs) : "memory");
                if (pt == 0) {
                    const uint32_t* first = sBlkMax + ((j & 1) * kNF + (fw - kblk)) * 32 + kW * o;
                    for (int k = 0; k < (1 << bs); ++k) {
#pragma unroll
                        for (int c = 0; c < kW; ++c) {
                            const uint32_t v = first[32 * k + c];
                            if constexpr (kTf32) hm[c] = __float_as_uint(fmaxf(__uint_as_float(hm[c]), __uint_as_float(v)));
                            else hm[c] = max16x2<kPrec>(hm[c], v);
                        }
                    }
                    sts128(gslot_sa + g_off0, hm[0], hm[1], hm[2], hm[3]);
                    if constexpr (kTf32) sts128(gslot_sa + g_off1, hm[4], hm[5], hm[6], hm[7]);
                }
            }
            if (lane == 0) sValid[(p & (kValidRing - 1)) * 2 + half] = (unsigned char)bvalid;
            fence_async_smem();
            __syncwarp();
            PTL(1 + fw, j, 2);
            if (lane == 0) mbar_arrive(&h_full[st]);
        }
    } else {
        // =========================== epilogue: group g owns channel tile g ===========================
        setmaxnreg_dec<kRegEpi>();
        const int g = (warp - kEpiWarp0) >> 2;
        const int quad = warp & 3;  // TMEM lanes this warp may read: 32 * (warp id % 4)
        const bool nchw = (kMode == 2) || (kMode == 0 && canvas && (a.out_layout == P3P_LAYOUT_NCHW));
        const bool f32 = (kMode == 2) || (kMode == 3) || (a.out_dtype == P3P_DTYPE_F32);  // (mode 1: rows of either width)
        const int C = a.bl.C, ipt = a.items_per_tile;
        // fast path: whole units inside one tile, every item exists -> no per-item bounds, two-cell vector stores
        const bool fast = (kMode != 0) || (bs == 0 && canvas && (total_items % kUnit == 0) && (ipt % kUnit == 0) && a.token_rows == 0);
        const bool tokens = (kMode == 3);
        const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
        const int cl = quad * 32 + lane;  // channel inside a 128-channel tile
        float b1v[3];
#pragma unroll
        for (int mm = 0; mm < 3; ++mm) b1v[mm] = sB1[mm * 128 + cl];
        ItemWalk wu;  // position of the first item of the unit in work
        wu.init((((int)blockIdx.x * kUnit) >> bs) < total_items ? (((int)blockIdx.x * kUnit) >> bs) : 0, ((int)gridDim.x * kUnit) >> bs, ipt);
        int unit_item0 = ((int)blockIdx.x * kUnit) >> bs;  // first pillar of the unit
        const int m = g;  // group g reads accumulator stage g = channel tile g
        const float bb = (m == 0) ? b1v[0] : ((m == 1) ? b1v[1] : b1v[2]);
        const int c = m * 128 + cl;
        const uint32_t taddr = tlane + (uint32_t)(g * kAccStages * kAccCols);
        const uint32_t gaddr = tlane + (uint32_t)(kGCol0 + g * 16);
        const uint32_t tf_sa = opaque(smem_u32(t_full + g * kAccStages));   // stage s: + 8 s
        const uint32_t te_sa = opaque(smem_u32(t_empty + g * kAccStages));
        const uint32_t gtf_sa = opaque(smem_u32(gt_full + 2 * g)), gte_sa = opaque(smem_u32(gt_empty + 2 * g));  // slot: + 8
        int jn = 0;
        // Pillar q of the CTA sits in accumulator stage q & 1 of the tile; its barrier phase is (q >> 1) & 1.  The probe of
        // the NEXT pillar's barrier is issued before the arithmetic on the current one, so that in the steady state (the
        // issuer runs ahead) no wait is exposed.
        uint32_t ready = 0;
        float va[16], vb[16];
        const uint32_t rmax_sa = opaque(smem_u32(sRmax + (warp - kEpiWarp0) * (kUnit * 32) + lane));  // [kUnit][32 lanes] strip of this warp (thread-private words)
        const uint32_t valid_sa = opaque(smem_u32(sValid));
        const uint32_t taddr_o = opaque(taddr);
        // rows layout: this thread's channel of the unit's first cell; advanced by one pointer addition per unit
        const int64_t rs = a.row_stride;
        const int64_t rows_first = (int64_t)blockIdx.x * kUnit * rs + a.row_offset + c;
        float* rows_dst = static_cast<float*>(a.out) + rows_first;
        unsigned short* rows_dst16 = static_cast<unsigned short*>(a.out) + rows_first;
        const int64_t rows_step = (int64_t)gridDim.x * kUnit * rs;
        // ---- W1b' hmax of the unit's 8 items (one MMA per unit), bias, relu, the 8 cells --------------------------------
        auto unit_tail = [&](int j, int ub, int ur, int item0) {
            float rmax[kUnit];
#pragma unroll
            for (int i = 0; i < kUnit; ++i) rmax[i] = lds_f32(rmax_sa + (uint32_t)(i * 128));
            // ---- W1b' hmax of the unit's 8 items (one MMA per unit), bias, relu, the 8 cells ---------------------------
            float gv[8];
            mbar_wait_sa(gtf_sa + 8u * ((uint32_t)j & 1u), ((uint32_t)j >> 1) & 1u);
            tc_fence_after();
            tmem_ld8_wait(gaddr + (uint32_t)((j & 1) * kGSlotCols), gv);
            tc_fence_before();
            mbar_arrive_sa(gte_sa + 8u * ((uint32_t)j & 1u));
            // which items hold a pillar: written by the front end before the pairs' operands were released
            const uint2 vv = lds_u32x2(valid_sa + (uint32_t)(((j * kPairsPerUnit) & (kValidRing - 1)) * 2));
            float ob[kUnit];
#pragma unroll
            for (int i = 0; i < kUnit; ++i) {
                const unsigned word = i < 4 ? vv.x : vv.y;
                const bool v = ((word >> (8 * (i & 3))) & 0xFFu) != 0;
                ob[i] = v ? fmaxf(rmax[i] + (gv[i] + bb), 0.f) : 0.f;
            }
            if (c < C) {
                if (tokens) {
                    // token sequence: rows 1 + cell of the tile, positional embedding added on the way out
                    const int64_t row = (int64_t)ub * a.token_rows + 1 + ur;
                    float* dst = static_cast<float*>(a.out) + row * C + c;
                    const float* pe = a.pos_embed + (int64_t)(1 + ur) * C + c;
#pragma unroll
                    for (int i = 0; i < kUnit; ++i) dst[(int64_t)i * C] = ob[i] + __ldg(pe + (int64_t)i * C);
                } else if (fast) {
                    if (nchw) {
                        const int64_t i0 = ((int64_t)ub * a.c_total + a.c_offset + c) * ipt + ur;
                        if (f32) {
                            float4* dst = reinterpret_cast<float4*>(static_cast<float*>(a.out) + i0);
                            dst[0] = make_float4(ob[0], ob[1], ob[2], ob[3]);
                            dst[1] = make_float4(ob[4], ob[5], ob[6], ob[7]);
                        } else {
                            const int dt = a.out_dtype;
                            *reinterpret_cast<uint4*>(static_cast<unsigned short*>(a.out) + i0) =
                                make_uint4((uint32_t)to_16bit(ob[0], dt) | ((uint32_t)to_16bit(ob[1], dt) << 16), (uint32_t)to_16bit(ob[2], dt) | ((uint32_t)to_16bit(ob[3], dt) << 16),
                                           (uint32_t)to_16bit(ob[4], dt) | ((uint32_t)to_16bit(ob[5], dt) << 16), (uint32_t)to_16bit(ob[6], dt) | ((uint32_t)to_16bit(ob[7], dt) << 16));
                        }
                    } else if (f32) {
                        // (B, ny nx, C) rows: a warp writes 32 consecutive channels of each of the unit's 8 cells
                        float* dst = rows_dst;
#pragma unroll
                        for (int i = 0; i < kUnit; ++i) { *dst = ob[i]; dst += rs; }
                    } else {
                        // 16-bit rows (the channels-last input of the fusion convolution)
                        unsigned short* dst = rows_dst16;
#pragma unroll
                        for (int i = 0; i < kUnit; ++i) { *dst = to_16bit(ob[i], a.out_dtype); dst += rs; }
                    }
                } else {
                    if (bs) {
                        // M > 64: the pillar's value = max over its blocks that took part (same W1b' hmax term in each)
                        const int bpp = 1 << bs;
#pragma unroll
                        for (int i = 0; i < kUnit; ++i) {
                            const unsigned word = i < 4 ? vv.x : vv.y;
                            const bool v = ((word >> (8 * (i & 3))) & 0xFFu) != 0;
                            ob[i] = v ? rmax[i] + (gv[i] + bb) : -INFINITY;
                        }
#pragma unroll
                        for (int i = 0; i < kUnit; ++i) {
                            if ((i & (bpp - 1)) == 0) {
                                float mval = ob[i];
#pragma unroll
                                for (int k = 1; k < kUnit; ++k)
                                    if (k < bpp && i + k < kUnit) mval = fmaxf(mval, ob[i + k]);
                                ob[i >> bs] = mval == -INFINITY ? -INFINITY : fmaxf(mval, 0.f);  // (i >> bs <= i: no hazard)
                            }
                        }
                    }
                    int bi = ub, ri = ur;
#pragma unroll
                    for (int i = 0; i < kUnit; ++i) {
                        if (bs && i >= (kUnit >> bs)) break;
                        const int item = item0 + i;
                        const unsigned word = i < 4 ? vv.x : vv.y;
                        bool v = ((word >> (8 * (i & 3))) & 0xFFu) != 0;
                        if (bs) { v = ob[i] != -INFINITY; if (!v) ob[i] = 0.f; }
                        // list rows past num_pillars stay untouched, canvas cells are always written
                        if (item < total_items && (v || canvas)) {
                            if (a.token_rows) {  // token sequence: row 1 + cell of the tile, + pos_embed
                                static_cast<float*>(a.out)[((int64_t)bi * a.token_rows + 1 + ri) * C + c] =
                                    ob[i] + a.pos_embed[(int64_t)(1 + ri) * C + c];
                            } else {
                                const int64_t idx = nchw ? ((int64_t)bi * a.c_total + a.c_offset + c) * ipt + ri : (int64_t)item * rs + a.row_offset + c;
                                store_scalar(a, idx, ob[i]);
                            }
                        }
                        if (++ri >= ipt) { ri = 0; ++bi; }
                    }
                }
            }
            rows_dst += rows_step;
            rows_dst16 += rows_step;
            if (quad == 0) PTL(9 + g, 8 * j + 7, 3);
        };
        const int my_units_g = (g < MT) ? my_units : 0;
        for (int j = 0; j < my_units_g; ++j) {
            const int ub = wu.b, ur = wu.r;  // tile / position of the unit's first item
            const int item0 = unit_item0;
            wu.step();
            unit_item0 += ((int)gridDim.x * kUnit) >> bs;
            // ---- the unit's 8 pillars: max over each pillar's 64 accumulator columns ---------------------------------
            // (the loop over the pairs is unrolled: barrier parities, strip offsets and probe conditions become constants of
            // the body; the pillar maxima wait for the unit's W1b' hmax term in a per-warp shared-memory strip, not in
            // registers).  Four loads of 16 columns per pillar through two register buffers: the arithmetic on one buffer
            // overlaps the load into the other.
#pragma unroll
            for (int pr = 0; pr < kPairsPerUnit; ++pr) {
#pragma unroll
                for (int s = 0; s < kAccStages; ++s, ++jn) {
                    const uint32_t tph = (uint32_t)pr & 1u;  // jn = 8 j + 2 pr + s: (jn >> 1) & 1 is a constant of the unrolled body
                    if (quad == 0) PTL(9 + g, jn, 0);
                    if (!ready) mbar_wait_sa(tf_sa + 8u * s, tph);
                    tc_fence_after();
                    tmem_ld16_issue(taddr_o + (uint32_t)(s * kAccCols), va);
                    if (quad == 0) PTL(9 + g, jn, 1);
                    tmem_ld_wait16(va);
                    tmem_ld16_issue(taddr_o + (uint32_t)(s * kAccCols + 16), vb);
                    // (inside a unit the next pillar always exists; behind its last pillar only if another unit follows)
                    ready = (2 * pr + s + 1 < kUnit || j + 1 < my_units_g) ? mbar_test_sa(tf_sa + 8u * (s ^ 1), (uint32_t)((2 * pr + s + 1) >> 1) & 1u) : 0u;
                    const float r0 = max16(va);
                    tmem_ld_wait16(vb);
                    tmem_ld16_issue(taddr_o + (uint32_t)(s * kAccCols + 32), va);
                    const float r1 = max16_with(r0, vb);
                    tmem_ld_wait16(va);
                    tmem_ld16_issue(taddr_o + (uint32_t)(s * kAccCols + 48), vb);
                    const float r2 = max16_with(r1, va);
                    tmem_ld_wait16(vb);
                    tc_fence_before();
                    mbar_arrive_sa(te_sa + 8u * s);
                    sts_f32(rmax_sa + (uint32_t)((2 * pr + s) * 128), max16_with(r2, vb));
                    if (quad == 0) PTL(9 + g, jn, 2);
                }
            }
            unit_tail(j, ub, ur, item0);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace

int launch_pfn_prepare(const p3p_pfn_params* p, int precision, char* blob, const BlobLayout& bl, cudaStream_t st) {
    pfn_prepare_kernel<<<4, 128, 0, st>>>(*p, precision, blob, bl);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_pfn_simt(const PfnArgs& a, cudaStream_t st) {
    if (a.num_items <= 0) return P3P_OK;
    if (a.num_items > 0x7fffffff - 64) return fail(P3P_ERR_UNSUPPORTED, "%lld work items exceed the 32-bit item index", (long long)a.num_items);
    const size_t smem = ((size_t)(a.g.M + 1) * kHStride + 256 + 32 + 96 + 32) * sizeof(float);
    // (the attribute belongs to the current device's context: set per launch, it is cheap)
    P3P_CUDA_CHECK(cudaFuncSetAttribute(pfn_simt_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    P3P_CUDA_CHECK(cudaFuncSetAttribute(pfn_simt_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    const int sms = device_sm_count();
    const bool hoist = a.bl.C <= kSimtMaxThreads;
    const int threads = hoist ? (a.bl.C + 31) / 32 * 32 : kSimtMaxThreads;
    int64_t grid = (int64_t)sms * (hoist ? (threads <= 256 ? 4 : 2) : 2);
    if (grid > a.num_items) grid = a.num_items;
    if (hoist)
        pfn_simt_kernel<true><<<(unsigned)grid, threads, smem, st>>>(a);
    else
        pfn_simt_kernel<false><<<(unsigned)grid, threads, smem, st>>>(a);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_cls_rows(const PfnArgs& a, const float* cls_token, cudaStream_t st) {
    if (a.B <= 0) return P3P_OK;
    const int64_t total = (int64_t)a.B * a.bl.C;
    cls_rows_kernel<<<(unsigned)((total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024), 256, 0, st>>>(a, cls_token);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_zero_lidar(const PfnArgs& a, cudaStream_t st) {
    if (a.num_items <= 0) return P3P_OK;
    zero_lidar_kernel<<<device_sm_count() * 4, 256, 0, st>>>(a);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_pfn_tc(const PfnArgs& a_in, int precision, cudaStream_t st) {
    if (a_in.num_items <= 0) return P3P_OK;
    if (a_in.num_items > 0x7fffffff - 64) return fail(P3P_ERR_UNSUPPORTED, "%lld work items exceed the 32-bit item index", (long long)a_in.num_items);
    PfnArgs a = a_in;
    a.blk_shift = 0;
    while ((64 << a.blk_shift) < a.g.M) ++a.blk_shift;  // blocks per pillar: 1, 2, 4, 8
    if ((a.num_items << a.blk_shift) > 0x7fffffff - 64) return fail(P3P_ERR_UNSUPPORTED, "too many row blocks for the 32-bit item index");
    const int64_t units = ((a.num_items << a.blk_shift) + kUnit - 1) / kUnit;
    int64_t grid = device_sm_count();
    if (grid > units) grid = units;
    int mode = 0;
    if (a.blk_shift == 0 && a.item_mode == kItemsCanvas && a.num_items % kUnit == 0 && a.items_per_tile % kUnit == 0) {
        if (a.token_rows) mode = a.out_dtype == P3P_DTYPE_F32 ? 3 : 0;
        else if (a.out_layout == P3P_LAYOUT_NCHW) mode = a.out_dtype == P3P_DTYPE_F32 ? 2 : 0;
        else mode = 1;  // rows, fp32 or 16-bit
    }
    // Programmatic dependent launch: the CTAs start (TMEM allocation, barriers, weights -> shared memory) while the
    // voxelizer's last chunks drain, and wait for its results with griddepcontrol.wait before their first read.
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kTcThreads);
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
#define P3P_LAUNCH_TC(PREC, MODE)                      \
    do {                                               \
        cfg.dynamicSmemBytes = TcCfg<PREC>::kSmemBytes; \
        P3P_CUDA_CHECK(cudaFuncSetAttribute(pfn_tc_kernel<PREC, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                            (int)TcCfg<PREC>::kSmemBytes)); /* per device context: set per launch */ \
        P3P_CUDA_CHECK(cudaLaunchKernelEx(&cfg, pfn_tc_kernel<PREC, MODE>, a)); \
    } while (0)
#define P3P_LAUNCH_TC_MODES(PREC)                         \
    do {                                                  \
        if (mode == 1) P3P_LAUNCH_TC(PREC, 1);            \
        else if (mode == 2) P3P_LAUNCH_TC(PREC, 2);       \
        else if (mode == 3) P3P_LAUNCH_TC(PREC, 3);       \
        else P3P_LAUNCH_TC(PREC, 0);                      \
    } while (0)
    if (precision == P3P_PRECISION_TF32) P3P_LAUNCH_TC_MODES(P3P_PRECISION_TF32);
    else if (precision == P3P_PRECISION_BF16) P3P_LAUNCH_TC_MODES(P3P_PRECISION_BF16);
    else P3P_LAUNCH_TC_MODES(P3P_PRECISION_FP16);
#undef P3P_LAUNCH_TC_MODES
#undef P3P_LAUNCH_TC
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

}  // namespace p3p
