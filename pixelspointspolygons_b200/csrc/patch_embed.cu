// patch_embed.cu -- image patch embedding written into the early-fusion concat buffer (sm_100a).
//
// Replaces `x_image = self.image_embed(x_image)` of the fusion encoders
// (R:pixelspointspolygons/models/fusion_layers/early_fusion_vit.py:69-70,99 and early_fusion_vit_cnn.py:67-68,90;
// timm PatchEmbed with flatten=False: Conv2d(in_chans, C, kernel=P, stride=P, bias), output NCHW; SURVEY 8a row a9)
// and the image half of `torch.cat((x_image, x_lidar), dim=1)` (early_fusion_vit.py:121, row a11): the result goes
// straight to channels [c_offset, c_offset + C) of the (B, c_total, H/P, W/P) buffer, so the concat copy never runs.
//
// A stride-P PxP convolution is one GEMM per tile, out[ch][cell] = sum_k W[ch][k] X[k][cell] + bias[ch] with
// k = (c, py, px) -- the natural memory order of the (C, in_chans, P, P) weight -- and X[k][cell] the pixel
// (c, cy*P + py, cx*P + px).  With P = 8 one (c, py) row of a patch is 8 consecutive fp32 pixels = 32 bytes = exactly
// one UMMA K step (8 tf32 / 16 bf16 -> 32 bytes), so the im2col matrix is never built: every 32-byte pixel run is
// copied (coalesced along the image row) to its place in the swizzled K-major B operand in shared memory.
//
// patch_embed_tc_kernel: CTA = (row group of R cell rows, 128-channel tile, image).  D[128 ch x R*nx cells] lives in
//   TMEM; tcgen05.mma kind::tf32 (fp32 contract) or kind::f16 on bf16 operands (bf16 contract), fp32 accumulate;
//   epilogue: tcgen05.ld, + bias, NCHW rows of R*nx contiguous values per channel.
// patch_embed_simt_kernel: exact fp32 FMA for any P / shape -- the GPU-side cross-check and the fp32 route.
//
// Both kernels take the image in one of two formats, a compile-time parameter (kIn):
//   kInF32:  (B, in_chans, H, W) fp32 NCHW, already normalised by the loader;
//   kInU8:   (B, H, W, in_chans) uint8 channels-last -- the decoded image as the loader holds it before its Normalize /
//            ToTensor -- with a pixel table lut (in_chans, 256) fp32: pixel value = lut[c][byte].  Every per-channel pointwise
//            normalisation is such a table, so the conversion is exact whatever arithmetic the loader used.  The table is
//            copied to a static shared array (4 KB), outside the dynamic shared-memory budget: both formats take the same
//            route with the same row group, and the u8 image moves a quarter of the fp32 bytes.
#include "p3p_internal.cuh"

namespace p3p {
namespace {

constexpr int kInF32 = 0, kInU8 = 1;  // image formats (see the file comment)
constexpr int kMaxU8Chans = 4;      // channels of a u8 image: one 8-byte load per channel per 8-pixel span

__device__ __forceinline__ void store_out(void* out, int out_dtype, int64_t idx, float v) {
    if (out_dtype == P3P_DTYPE_F32)
        static_cast<float*>(out)[idx] = v;
    else
        static_cast<unsigned short*>(out)[idx] = to_16bit(v, out_dtype);
}

// ------------------------------------------------------------------------------------------------
// exact fp32 kernel: one CTA per (cell, image); the patch sits in shared memory, one thread per channel
// ------------------------------------------------------------------------------------------------
// kInU8: img is NULL; img8 (B, H, W, in_chans) and lut (in_chans, 256) are read instead
template <int kIn>
__global__ void __launch_bounds__(128)
patch_embed_simt_kernel(const float* __restrict__ img, int in_chans, int H, int W, int P, const float* __restrict__ weight,
                        const float* __restrict__ bias, int C, void* out, int out_dtype, int out_layout, int c_total, int c_offset,
                        const unsigned char* __restrict__ img8, const float* __restrict__ lut) {
    extern __shared__ float patch[];  // [in_chans * P * P]
    const int nx = W / P, ny = H / P;
    const int cell = blockIdx.x, b = blockIdx.y;
    const int cy = cell / nx, cx = cell - cy * nx;
    const int K = in_chans * P * P;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const int c = k / (P * P), r = k - c * P * P, py = r / P, px = r - py * P;
        if constexpr (kIn == kInU8)
            patch[k] = __ldg(lut + c * 256 + img8[(((int64_t)b * H + cy * P + py) * W + cx * P + px) * in_chans + c]);
        else
            patch[k] = img[(((int64_t)b * in_chans + c) * H + cy * P + py) * W + cx * P + px];
    }
    __syncthreads();
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
        const float* w = weight + (int64_t)ch * K;
        float acc = 0.f;
        for (int k = 0; k < K; ++k) acc = __fmaf_rn(w[k], patch[k], acc);
        if (bias) acc += bias[ch];
        const int64_t idx = out_layout == P3P_LAYOUT_NLC ? ((int64_t)b * (ny * nx) + cell) * c_total + c_offset + ch
                                                         : ((int64_t)b * c_total + c_offset + ch) * (ny * nx) + cell;
        store_out(out, out_dtype, idx, acc);
    }
}

// ------------------------------------------------------------------------------------------------
// tensor-core kernel (P == 8)
// ------------------------------------------------------------------------------------------------
constexpr int kPeThreads = 256;

struct PeArgs {
    const float* img;
    const float* weight;
    const float* bias;
    const unsigned char* blob;  // prepared weights (p3p_patch_embed_prepare): the tiles' operand images, or NULL
    void* out;
    int in_chans, H, W, C, nx, ny;
    int rows;       // cell rows per CTA
    int N;          // rows * nx: MMA N (multiple of 16, <= 128)
    int out_dtype, out_layout, c_total, c_offset;
    const unsigned char* img8;  // kInU8: (B, H, W, in_chans) uint8 (img is NULL) ...
    const float* lut;           // ... and its pixel table (in_chans, 256)
};

// Operand rows are K-major and split into 128-byte chunks (SWIZZLE_128B atoms, 8 rows x 128 B); chunk q of a tile
// with `nrows` rows starts at q * nrows * 128.  One 32-byte pixel run (c, py) of 8 fp32 values becomes
//   tf32: 2 x 16-byte units  (chunk = k8 / 4, units (k8 % 4) * 2 + {0, 1}),   k8 = c * 8 + py
//   bf16: 1 x 16-byte unit   (chunk = k8 / 8, unit k8 % 8)
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

template <int kPrec>
__device__ __forceinline__ void put_run(unsigned char* tile, int nrows, int row, int k8, const float4& lo, const float4& hi) {
    if constexpr (kPrec == P3P_PRECISION_TF32) {
        unsigned char* base = tile + (size_t)(k8 >> 2) * nrows * 128 + (size_t)row * 128;
        const int u = (k8 & 3) * 2;
        const uint4 a = make_uint4(to_tf32(lo.x), to_tf32(lo.y), to_tf32(lo.z), to_tf32(lo.w));
        const uint4 b = make_uint4(to_tf32(hi.x), to_tf32(hi.y), to_tf32(hi.z), to_tf32(hi.w));
        *reinterpret_cast<uint4*>(base + (((u + 0) ^ (row & 7)) * 16)) = a;
        *reinterpret_cast<uint4*>(base + (((u + 1) ^ (row & 7)) * 16)) = b;
    } else {
        unsigned char* base = tile + (size_t)(k8 >> 3) * nrows * 128 + (size_t)row * 128;
        const int u = k8 & 7;
        const uint4 a = (kPrec == P3P_PRECISION_BF16)
                            ? make_uint4(pack_bf16(lo.x, lo.y), pack_bf16(lo.z, lo.w), pack_bf16(hi.x, hi.y), pack_bf16(hi.z, hi.w))
                            : make_uint4(pack_f16(lo.x, lo.y), pack_f16(lo.z, lo.w), pack_f16(hi.x, hi.y), pack_f16(hi.z, hi.w));
        *reinterpret_cast<uint4*>(base + ((u ^ (row & 7)) * 16)) = a;
    }
}

// One span of a u8 image: 8 pixels x kIC bytes (pixel-major, as the image stores them) of pixel row py of a cell, loaded as
// kIC 8-byte words.  Byte c of every pixel goes through the channel's table to the fp32 run (c, py), which put_run converts
// and stores exactly as it does an fp32 image's run.  (kIC is a template parameter so that every byte position is a constant:
// the bytes are picked out of registers, no local-memory array.)
template <int kPrec, int kIC>
__device__ __forceinline__ void put_span_u8(unsigned char* tile, int nrows, int row, int py, const uint2 (&w)[kMaxU8Chans],
                                            const float* lut) {
#pragma unroll
    for (int c = 0; c < kIC; ++c) {
        float v[8];
#pragma unroll
        for (int p = 0; p < 8; ++p) {
            const int j = p * kIC + c;  // byte of the span
            const uint32_t word = (j & 4) ? w[j >> 3].y : w[j >> 3].x;
            v[p] = lut[c * 256 + ((word >> ((j & 3) * 8)) & 0xffu)];
        }
        put_run<kPrec>(tile, nrows, row, c * 8 + py, make_float4(v[0], v[1], v[2], v[3]), make_float4(v[4], v[5], v[6], v[7]));
    }
}

// CTA = (row group of R cell rows, image): the B operand (the pixel runs of the row group, the only HBM read) is built ONCE
// and multiplied with every 128-channel tile of the weights -- kTilesResident tiles at a time (all three of C = 384 with
// 16-bit operands; one with tf32, whose tiles are twice as large), each tile an MMA chain into its own TMEM columns with its
// own commit barrier, so that the epilogue of tile m runs under the MMAs of tile m + 1.  (r01: one CTA per (row group,
// channel tile, image) re-read the image slab three times and idled through load -> MMA -> epilogue; 28 us at B = 16.)
template <int kPrec, int kIn>
__global__ void __launch_bounds__(kPeThreads, 1) patch_embed_tc_kernel(PeArgs a) {
    constexpr bool kTf32 = (kPrec == P3P_PRECISION_TF32);
    constexpr int kTilesResident = kTf32 ? 1 : 3;
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t raw = smem_u32(smem_dyn);
    unsigned char* base = smem_dyn + ((1024u - (raw & 1023u)) & 1023u);
    const int K8 = a.in_chans * 8;                    // 32-byte pixel runs per operand row
    const int NQ = kTf32 ? K8 / 4 : K8 / 8;           // 128-byte chunks per operand row
    const int Npad = (a.N + 7) / 8 * 8;               // (N is a multiple of 16 already)
    const size_t a_tile_bytes = (size_t)NQ * 128 * 128;
    unsigned char* sA = base;                                   // [kTilesResident][NQ][128 rows][128 B]
    unsigned char* sB = sA + kTilesResident * a_tile_bytes;     // [NQ][Npad rows][128 B]
    __shared__ uint64_t bar[kTilesResident];
    __shared__ uint64_t abar;  // prepared weights: the tiles' bulk copies have landed
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rg = blockIdx.x, b = blockIdx.y;
    const int cy0 = rg * a.rows;
    const int MT = (a.C + 127) / 128;

    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 32) {
        for (int i = 0; i < kTilesResident; ++i) mbar_init(&bar[i], 1);
        mbar_init(&abar, 1);
        fence_mbar_init();
    }
    const bool prepared = a.blob != nullptr;
    float* lut_s = nullptr;  // kInU8: the pixel table in static shared memory (not in the dynamic operand budget)
    if constexpr (kIn == kInU8) {
        __shared__ float lut_tab[kMaxU8Chans * 256];
        lut_s = lut_tab;
        for (int i = tid; i < a.in_chans * 256; i += kPeThreads) lut_s[i] = __ldg(a.lut + i);
    }
    // (the barrier is initialised before the copies that complete on it are issued; the table is in place before the
    // pixel spans are built)
    if (kIn == kInU8 || prepared) __syncthreads();
    // 32-byte runs -> operand rows.  A: 128 channels x K weights of tile mt, natural (C, in_chans, 8, 8) order == K-major
    // rows; B: the pixel runs of `rows` cell rows: image rows (c, cy0*8 + y), nx runs each.  kDepth runs (2 x float4 each) per
    // thread in flight.
    const int runs_a = 128 * K8;
    const int runs_b = a.in_chans * a.rows * 8 * a.nx;
    const float* src_b = a.img + (size_t)b * a.in_chans * a.H * a.W;
    auto load_runs = [&](int mt0, int ntiles, bool with_b) {
        constexpr int kDepth = 6;
        const int runs = ntiles * runs_a + (with_b ? runs_b : 0);
        for (int i0 = tid; i0 < runs; i0 += kPeThreads * kDepth) {
            float4 lo[kDepth], hi[kDepth];
            int row[kDepth], k8v[kDepth], dst[kDepth];  // dst: -1 nothing, 0..2 A tile, 3 B
#pragma unroll
            for (int d = 0; d < kDepth; ++d) {
                const int i = i0 + d * kPeThreads;
                lo[d] = make_float4(0.f, 0.f, 0.f, 0.f); hi[d] = lo[d];
                row[d] = 0; k8v[d] = 0; dst[d] = -1;
                if (i < ntiles * runs_a) {
                    const int t = i / runs_a, j = i - t * runs_a;
                    const int r = j / K8, k8 = j - r * K8;
                    const int ch = (mt0 + t) * 128 + r;
                    row[d] = r; k8v[d] = k8; dst[d] = t;
                    if (ch < a.C) {
                        const float4* src = reinterpret_cast<const float4*>(a.weight + ((size_t)ch * K8 + k8) * 8);
                        lo[d] = __ldg(src);
                        hi[d] = __ldg(src + 1);
                    }
                } else if (i < runs) {
                    const int ib = i - ntiles * runs_a;
                    const int ir = ib / a.nx, cx = ib - ir * a.nx;
                    const int c = ir / (a.rows * 8), yl = ir - c * (a.rows * 8);
                    const int cyl = yl >> 3, py = yl & 7;
                    const float4* src = reinterpret_cast<const float4*>(src_b + ((size_t)c * a.H + cy0 * 8 + yl) * a.W + cx * 8);
                    lo[d] = __ldg(src);
                    hi[d] = __ldg(src + 1);
                    row[d] = cyl * a.nx + cx; k8v[d] = c * 8 + py; dst[d] = 3;
                }
            }
#pragma unroll
            for (int d = 0; d < kDepth; ++d) {
                if (dst[d] < 0) continue;
                if (dst[d] < 3)
                    put_run<kPrec>(sA + (size_t)dst[d] * a_tile_bytes, 128, row[d], k8v[d], lo[d], hi[d]);
                else
                    put_run<kPrec>(sB, Npad, row[d], k8v[d], lo[d], hi[d]);
            }
        }
    };
    // u8 image: the B operand from the spans of `rows` cell rows -- image rows cy0*8 + y, nx spans of 8 pixels x in_chans
    // bytes each, consecutive threads on consecutive spans of a row (coalesced), kDepthU8 spans per thread in flight
    auto load_spans_u8 = [&]() {
        if constexpr (kIn == kInU8) {
            constexpr int kDepthU8 = 4;
            const int spans = a.rows * 8 * a.nx;
            const int span_bytes = 8 * a.in_chans;
            const unsigned char* src8 = a.img8 + ((size_t)b * a.H + (size_t)cy0 * 8) * a.W * a.in_chans;
            for (int i0 = tid; i0 < spans; i0 += kPeThreads * kDepthU8) {
                uint2 w[kDepthU8][kMaxU8Chans];
#pragma unroll
                for (int d = 0; d < kDepthU8; ++d) {
                    const int i = i0 + d * kPeThreads;
                    const int yl = i / a.nx, cx = i - yl * a.nx;
                    const uint2* src = reinterpret_cast<const uint2*>(src8 + (size_t)yl * a.W * a.in_chans + (size_t)cx * span_bytes);
#pragma unroll
                    for (int c = 0; c < kMaxU8Chans; ++c) w[d][c] = (i < spans && c < a.in_chans) ? __ldg(src + c) : make_uint2(0u, 0u);
                }
#pragma unroll
                for (int d = 0; d < kDepthU8; ++d) {
                    const int i = i0 + d * kPeThreads;
                    if (i >= spans) break;
                    const int yl = i / a.nx, cx = i - yl * a.nx;
                    const int row = (yl >> 3) * a.nx + cx, py = yl & 7;
                    switch (a.in_chans) {
                        case 1: put_span_u8<kPrec, 1>(sB, Npad, row, py, w[d], lut_s); break;
                        case 2: put_span_u8<kPrec, 2>(sB, Npad, row, py, w[d], lut_s); break;
                        case 3: put_span_u8<kPrec, 3>(sB, Npad, row, py, w[d], lut_s); break;
                        default: put_span_u8<kPrec, 4>(sB, Npad, row, py, w[d], lut_s); break;
                    }
                }
            }
        }
    };
    const int quad = warp & 3, hi_half = warp >> 2;
    // The fp32 NCHW epilogue stages its transposes in a weight tile's space, 8 warps x 32 x 17 floats.  A 16-bit tile of one
    // input channel is 16 KB, smaller than that: past its end lie the next tile, still under its MMAs, or the image operand,
    // which a further round reads again.  Such tiles store their 16 cells per thread directly.
    const bool stage_nchw = a.out_layout == P3P_LAYOUT_NCHW && a.out_dtype == P3P_DTYPE_F32 &&
                            a_tile_bytes >= (size_t)kPeThreads * 17 * sizeof(float);
    const int nblk = a.N / 16, split = (nblk + 1) / 2;
    const int blk0 = hi_half ? split : 0, blk1 = hi_half ? nblk : split;
    uint32_t tmem_base = 0;
    int round = 0;
    for (int mt0 = 0; mt0 < MT; mt0 += kTilesResident, ++round) {
        const int ntiles = (MT - mt0 < kTilesResident) ? MT - mt0 : kTilesResident;
        // A further round (tf32: one resident tile) refills the weight tile's space, which the previous round's epilogue uses
        // as its transpose staging: every warp must be through with it first.  (Found by running the suite under
        // compute-sanitizer, whose timing let warp 0's bulk copy land under the other warps' staged values.)
        if (round > 0) __syncthreads();
        if (prepared) {
            // the tiles are stored as their shared-memory operand images: one bulk copy per tile (TMA, no register
            // traffic) next to the threads' work on the pixel runs
            if (tid == 0) {
                mbar_expect_tx(&abar, (uint32_t)(ntiles * a_tile_bytes));
                for (int t = 0; t < ntiles; ++t)
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sA + (size_t)t * a_tile_bytes)),
                                 "l"(a.blob + (size_t)(mt0 + t) * a_tile_bytes), "r"((uint32_t)a_tile_bytes), "r"(smem_u32(&abar)) : "memory");
            }
            if constexpr (kIn == kInU8) {
                if (mt0 == 0) load_spans_u8();
            } else {
                load_runs(mt0, 0, mt0 == 0);
            }
        } else {
            load_runs(mt0, ntiles, kIn == kInF32 && mt0 == 0);
            if constexpr (kIn == kInU8) {
                if (mt0 == 0) load_spans_u8();
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();  // operands written; the previous round's epilogue has drained its TMEM columns
        tc_fence_after();
        if (prepared && warp == 0) mbar_wait(&abar, (uint32_t)round & 1u);
        tmem_base = tmem_slot;
        if (warp == 0) {
            if (elect_one()) {
                const uint32_t idesc = make_idesc(kTf32 ? 2 : (kPrec == P3P_PRECISION_BF16 ? 1 : 0), 128, a.N);
                const uint32_t desc_hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024 B, SWIZZLE_128B
                const uint32_t b_lo = (smem_u32(sB) >> 4) | (1u << 16);
                for (int t = 0; t < ntiles; ++t) {
                    const uint32_t a_lo = (smem_u32(sA + (size_t)t * a_tile_bytes) >> 4) | (1u << 16);
                    for (int q = 0; q < NQ; ++q) {
#pragma unroll
                        for (int s = 0; s < 4; ++s) {
                            const uint32_t ao = (uint32_t)((q * 128 * 128 + s * 32) >> 4), bo = (uint32_t)((q * Npad * 128 + s * 32) >> 4);
                            tc_mma<kTf32>(tmem_base + (uint32_t)(t * 128), ((uint64_t)desc_hi << 32) | (a_lo + ao),
                                          ((uint64_t)desc_hi << 32) | (b_lo + bo), idesc, (q | s) != 0);
                        }
                    }
                    tc_commit(&bar[t]);
                }
            }
            __syncwarp();
        }
        // ---- epilogue: thread = channel (TMEM lane), warps 0-3 take the first 16-column blocks, warps 4-7 the rest ----------
        for (int t = 0; t < ntiles; ++t) {
            mbar_wait(&bar[t], (uint32_t)round & 1u);
            tc_fence_after();
            const int ch = (mt0 + t) * 128 + quad * 32 + lane;
            const float bv = (a.bias && ch < a.C) ? a.bias[ch] : 0.f;
            const int64_t row0 = ((int64_t)b * a.c_total + a.c_offset + ch) * ((int64_t)a.ny * a.nx) + (int64_t)cy0 * a.nx;
            for (int blk = blk0; blk < blk1; ++blk) {
                float v[16];
                tmem_ld16_wait(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(t * 128 + blk * 16), v);
                if (stage_nchw) {
                    // The thread holds 16 consecutive cells (64 bytes) of ITS channel: stored as they are, one instruction
                    // touches 32 cache lines.  Through a per-warp transpose in shared memory (the weight tile's space: its
                    // MMAs are done) a quarter-warp writes the 64 bytes of one channel, 8 channels = 8 lines per instruction.
                    float* stg = reinterpret_cast<float*>(sA + (size_t)t * a_tile_bytes) + warp * (32 * 17);
#pragma unroll
                    for (int i = 0; i < 16; ++i) stg[lane * 17 + i] = v[i] + bv;
                    __syncwarp();
                    const int cq = lane & 3, c8 = lane >> 2;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int cl = 8 * j + c8;  // channel of the warp's 32
                        const float* src = stg + cl * 17 + 4 * cq;
                        const float4 o = make_float4(src[0], src[1], src[2], src[3]);
                        const int chj = (mt0 + t) * 128 + quad * 32 + cl;
                        if (chj < a.C)
                            *reinterpret_cast<float4*>(static_cast<float*>(a.out) + ((int64_t)b * a.c_total + a.c_offset + chj) * ((int64_t)a.ny * a.nx) +
                                                       (int64_t)cy0 * a.nx + blk * 16 + 4 * cq) = o;
                    }
                    __syncwarp();
                } else if (ch < a.C) {
                    if (a.out_layout == P3P_LAYOUT_NLC) {
                        // channels-last rows (B, ny nx, c_total): a warp writes 32 consecutive channels of one cell per store
                        const int64_t r0 = ((int64_t)b * a.ny * a.nx + (int64_t)cy0 * a.nx + blk * 16) * a.c_total + a.c_offset + ch;
#pragma unroll
                        for (int i = 0; i < 16; ++i) store_out(a.out, a.out_dtype, r0 + (int64_t)i * a.c_total, v[i] + bv);
                    } else if (a.out_dtype == P3P_DTYPE_F32) {
                        float* dst = static_cast<float*>(a.out) + row0 + blk * 16;
#pragma unroll
                        for (int i = 0; i < 16; ++i) dst[i] = v[i] + bv;
                    } else {
                        unsigned short* dst = static_cast<unsigned short*>(a.out) + row0 + blk * 16;
#pragma unroll
                        for (int i = 0; i < 16; ++i) dst[i] = to_16bit(v[i] + bv, a.out_dtype);
                    }
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// Weights -> the 128-channel tiles' shared-memory operand images (what load_runs writes, once instead of per CTA and call),
// followed by the bias padded to whole tiles.  One thread per 32-byte run.
template <int kPrec>
__global__ void __launch_bounds__(256)
patch_embed_prepare_kernel(const float* __restrict__ weight, const float* __restrict__ bias, int C, int in_chans, unsigned char* blob) {
    constexpr bool kTf32 = (kPrec == P3P_PRECISION_TF32);
    const int K8 = in_chans * 8, MT = (C + 127) / 128;
    const size_t a_tile_bytes = (size_t)128 * K8 * (kTf32 ? 32 : 16);
    const int64_t runs = (int64_t)MT * 128 * K8;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < runs; i += (int64_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i / K8), k8 = (int)(i - (int64_t)ch * K8);
        float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
        if (ch < C) {
            const float4* src = reinterpret_cast<const float4*>(weight + ((size_t)ch * K8 + k8) * 8);
            lo = __ldg(src);
            hi = __ldg(src + 1);
        }
        put_run<kPrec>(blob + (size_t)(ch >> 7) * a_tile_bytes, 128, ch & 127, k8, lo, hi);
    }
    float* bdst = reinterpret_cast<float*>(blob + (size_t)MT * a_tile_bytes);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < MT * 128; i += gridDim.x * blockDim.x)
        bdst[i] = (bias && i < C) ? bias[i] : 0.f;
}

}  // namespace

size_t patch_embed_blob_bytes(int C, int in_chans, int P) {
    const size_t MT = ((size_t)C + 127) / 128;
    return MT * 128 * (size_t)in_chans * P * P * 4 + MT * 128 * sizeof(float);  // (tf32 tiles: the 16-bit ones are half of it)
}

int launch_patch_embed_prepare(const float* weight, const float* bias, int C, int in_chans, int P, int precision, void* blob, cudaStream_t st) {
    if (P != 8 || precision == P3P_PRECISION_FP32) return P3P_OK;  // the exact route reads the raw weights
    const int64_t runs = (int64_t)((C + 127) / 128) * 128 * in_chans * 8;
    const unsigned grid = (unsigned)((runs + 255) / 256 < 1184 ? (runs + 255) / 256 : 1184);
    unsigned char* bl = static_cast<unsigned char*>(blob);
    if (precision == P3P_PRECISION_TF32)
        patch_embed_prepare_kernel<P3P_PRECISION_TF32><<<grid, 256, 0, st>>>(weight, bias, C, in_chans, bl);
    else if (precision == P3P_PRECISION_BF16)
        patch_embed_prepare_kernel<P3P_PRECISION_BF16><<<grid, 256, 0, st>>>(weight, bias, C, in_chans, bl);
    else
        patch_embed_prepare_kernel<P3P_PRECISION_FP16><<<grid, 256, 0, st>>>(weight, bias, C, in_chans, bl);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

// blob: the prepared weights of `precision` (p3p_patch_embed_prepare) or NULL (raw weights converted by every CTA).
// images_u8 (B, H, W, in_chans) uint8 + pixel_lut (in_chans, 256), when given, replace the fp32 NCHW images; the route and
// the row group do not depend on the image format.
int launch_patch_embed(const float* images, int B, int in_chans, int H, int W, int P, const float* weight, const float* bias,
                       const void* blob, int C, int precision, void* out, int out_dtype, int out_layout, int c_total, int c_offset,
                       cudaStream_t st, const uint8_t* images_u8, const float* pixel_lut) {
    if (B <= 0) return P3P_OK;
    const bool u8 = images_u8 != nullptr;
    const int nx = W / P, ny = H / P;
    const bool tf32 = (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16);
    // tensor-core route: 8x8 patches; a row group of `rows` cell rows with rows * nx a multiple of 16 and <= 128 that
    // divides ny; operands (128 + N rows of K values) within the shared-memory budget; 16-byte aligned output rows
    int rows = 0;
    if (precision != P3P_PRECISION_FP32 && P == 8 && (W % 8) == 0) {
        for (int r = ny; r >= 1; --r) {
            const int n = r * nx;
            if (ny % r == 0 && n <= 128 && n % 16 == 0) { rows = r; break; }
        }
    }
    const size_t esize = tf32 ? 4 : 2;
    const size_t K = (size_t)in_chans * 64;
    const size_t smem = 1024 + ((tf32 ? 1 : 3) * 128 + (size_t)rows * nx) * K * esize;  // resident weight tiles + the row group
    const bool k_ok = tf32 ? (K % 32 == 0) : (K % 64 == 0);
    if (rows > 0 && k_ok && smem <= 200 * 1024 && ((size_t)ny * nx * (out_dtype == P3P_DTYPE_F32 ? 4 : 2)) % 16 == 0) {
        PeArgs a;
        a.img = images; a.weight = weight; a.bias = bias; a.out = out;
        a.img8 = images_u8; a.lut = pixel_lut;
        a.blob = static_cast<const unsigned char*>(blob);
        if (blob)  // the bias (padded to whole tiles, zeros without one) follows the tiles
            a.bias = reinterpret_cast<const float*>(a.blob + (size_t)((C + 127) / 128) * 128 * K * esize);
        a.in_chans = in_chans; a.H = H; a.W = W; a.C = C; a.nx = nx; a.ny = ny;
        a.rows = rows; a.N = rows * nx;
        a.out_dtype = out_dtype; a.out_layout = out_layout; a.c_total = c_total; a.c_offset = c_offset;
        dim3 grid((unsigned)(ny / rows), (unsigned)B);
        // (the attribute belongs to the current device's context: set per launch, it is cheap)
        auto launch = [&](auto kernel) -> int {
            P3P_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            kernel<<<grid, kPeThreads, smem, st>>>(a);
            P3P_CUDA_CHECK(cudaGetLastError());
            return P3P_OK;
        };
        if (tf32)
            return u8 ? launch(patch_embed_tc_kernel<P3P_PRECISION_TF32, kInU8>) : launch(patch_embed_tc_kernel<P3P_PRECISION_TF32, kInF32>);
        if (precision == P3P_PRECISION_BF16)
            return u8 ? launch(patch_embed_tc_kernel<P3P_PRECISION_BF16, kInU8>) : launch(patch_embed_tc_kernel<P3P_PRECISION_BF16, kInF32>);
        return u8 ? launch(patch_embed_tc_kernel<P3P_PRECISION_FP16, kInU8>) : launch(patch_embed_tc_kernel<P3P_PRECISION_FP16, kInF32>);
    }
    if (!weight) return fail(P3P_ERR_UNSUPPORTED, "this shape / precision takes the exact route, which needs the raw weights");
    const size_t smem_simt = (size_t)in_chans * P * P * sizeof(float);
    if (smem_simt > 48 * 1024) return fail(P3P_ERR_UNSUPPORTED, "patch of %d x %d x %d values exceeds the shared-memory budget", in_chans, P, P);
    dim3 grid((unsigned)(ny * nx), (unsigned)B);
    if (u8)
        patch_embed_simt_kernel<kInU8><<<grid, 128, smem_simt, st>>>(nullptr, in_chans, H, W, P, weight, bias, C, out, out_dtype, out_layout,
                                                                   c_total, c_offset, images_u8, pixel_lut);
    else
        patch_embed_simt_kernel<kInF32><<<grid, 128, smem_simt, st>>>(images, in_chans, H, W, P, weight, bias, C, out, out_dtype, out_layout,
                                                                    c_total, c_offset, nullptr, nullptr);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

}  // namespace p3p
