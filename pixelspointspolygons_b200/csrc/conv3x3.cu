// conv3x3.cu -- 3x3 / pad 1 convolution + folded BatchNorm2d + ReLU as an implicit GEMM on tcgen05, operands by TMA (sm_100a).
//
// Replaces the reference's `fusion_layer` (SURVEY 8f rank 1):
//     nn.Sequential(nn.Conv2d(2 C, C, kernel_size=3, padding=1), nn.BatchNorm2d(C), nn.ReLU(inplace=True))
//     x = self.fusion_layer(x).flatten(2).transpose(1, 2)
// (R:pixelspointspolygons/models/fusion_layers/early_fusion_vit.py:75-79,123; early_fusion_vit_cnn.py:72-76,94) and, with
// other sizes, the convolution of the `proj` tails (early_fusion_vit_cnn.py:78-83, pointpillars_vit_cnn.py:20-25; SURVEY 8f
// rank 5) behind a bilinear upsampling.
//
// Data layout.  The input is channels-last 16-bit: X (B, H, W, Cin) fp16 / bf16 -- for the fusion layer the two producers
// (patch embedding, PFN epilogue) write their halves of it directly, so the fp32 NCHW concat tensor of the reference
// never exists.  Weights are prepared once: BN scale folded in, 16-bit, K-major rows Wp (Cout_pad, 9 Cin) with
// K = tap * Cin + ci; the BN shift and the conv bias become one fp32 vector.
//
// Kernel.  CTA = (image, strip of `rows` image rows) x all output channels: D[co, pos] with M = 128 channels per MMA tile
// (up to 3 tiles side by side in TMEM, one issuing warp each), N = rows * W positions (a multiple of 16, <= 256).  K loop = 9 taps x Cin / 64
// blocks of 64 channels (128-byte rows, SWIZZLE_128B): per block one 4-D TMA box (64 ch, W, rows, 1) of X shifted by the
// tap -- the padding is the TMA's out-of-bounds zero fill, there is no im2col and no halo code -- and one 2-D box
// (64, 128) of Wp per channel tile.  Warp 0 produces (TMA + mbarrier expect_tx), warps 1-3 issue tcgen05.mma (one channel tile each) and
// release the stages with tcgen05.commit, warps 4-7 drain TMEM: + shift, ReLU, store as token rows (B, H W, Cout) -- the
// `.flatten(2).transpose(1, 2)` of the reference is the store address -- or NCHW.
//
// ViT-token epilogue (template flag kVitTokens; the NLC / NCHW instantiation is compiled without it): the output is the
// ViT's input sequence (B, 1 + H W, Cout), what timm's `_pos_embed` makes of the token rows (early_fusion_vit.py:123-124):
// position pos of image b goes to row b (1 + H W) + 1 + pos as relu(acc + shift) + pos_embed[1 + pos] -- BN, ReLU, then the
// fp32 add, the reference's order -- and the epilogue warps of the CTA holding strip 0 of an image write its row 0,
// cls_token + pos_embed[0], while the MMAs run.  pos_embed is read as the rows are stored: 32 consecutive channels of one
// position per warp access.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstring>

#include "p3p_internal.cuh"

namespace p3p {

namespace {

constexpr int kConvThreads = 256;  // warp 0: TMA producer, warps 1-3: one MMA issuer per channel tile, warps 4-7: epilogue
constexpr int kKBlockBytes = 128;        // one operand row of a K block: 64 16-bit channels
constexpr int kKBlock = 64;
constexpr int kWTileBytes = 128 * kKBlockBytes;  // 128 output channels x 64 k

struct ConvArgs {
    int B, H, W, Cin, Cout;
    int rows, N;           // image rows per strip, positions per strip = rows * W
    int strips;            // strips per image
    int co_tiles;          // 128-channel MMA tiles
    int acc_stride;        // TMEM columns between the accumulators of two channel tiles (128 or 256)
    int stages;            // operand stages in shared memory
    int stage_bytes;       // co_tiles * kWTileBytes + N rounded up to 8 rows * 128
    int fmt;               // UMMA format code: 0 = fp16, 1 = bf16
    int relu;
    const float* shift;    // (Cout) folded BN shift + conv bias
    float* out;
    int out_layout;        // P3P_LAYOUT_NLC: (B, H W, c_total) rows at c_offset; P3P_LAYOUT_NCHW: (B, c_total, H, W)
    int c_total, c_offset;
    const float* cls_token;  // (Cout)                  ViT-token epilogue only
    const float* pos_embed;  // ((1 + H W), Cout)       ViT-token epilogue only
};

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

template <bool kVitTokens>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w, ConvArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_dyn[];  // no static shared memory below: the block starts at offset 0
    constexpr int kMaxStages = 8;
    unsigned char* stage0 = smem_dyn;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_dyn + (size_t)a.stages * a.stage_bytes);
    uint64_t* full = bars;                   // [stages] TMA -> MMA (expect_tx)
    uint64_t* empty = bars + kMaxStages;     // [stages] MMA -> TMA (tcgen05.commit)
    uint64_t* acc_full = empty + kMaxStages; // MMA -> epilogue
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int strip = blockIdx.x % a.strips, b = blockIdx.x / a.strips;
    const int y0 = strip * a.rows;
    const int kblocks = a.Cin / kKBlock;
    const int iters = 9 * kblocks;

    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();  // the swizzled operand tiles need 1024-byte alignment
    if (warp == 4) tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        for (int i = 0; i < a.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], (uint32_t)a.co_tiles); }
        mbar_init(acc_full, (uint32_t)a.co_tiles);
        fence_mbar_init();
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w) : "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // (programmatic dependent launch: everything above overlaps the tail of the producers of X)
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            const uint32_t bytes = (uint32_t)(a.co_tiles * kWTileBytes + a.N * kKBlockBytes);
            int st = 0;
            uint32_t use = 0;
            for (int it = 0; it < iters; ++it) {
                const int tap = it / kblocks, kb = it - tap * kblocks;
                const int dy = tap / 3, dx = tap - dy * 3;
                mbar_wait(&empty[st], (use & 1u) ^ 1u);
                mbar_expect_tx(&full[st], bytes);
                const uint32_t dst = smem_u32(stage0 + (size_t)st * a.stage_bytes);
                // activations: channels [64 kb, +64) of the strip's positions shifted by the tap; rows / columns outside
                // the image arrive as zeros (the convolution's padding)
                tma_load_4d(dst + (uint32_t)(a.co_tiles * kWTileBytes), &tm_x, &full[st], kb * kKBlock, dx - 1, y0 + dy - 1, b);
                for (int t = 0; t < a.co_tiles; ++t)
                    tma_load_2d(dst + (uint32_t)(t * kWTileBytes), &tm_w, &full[st], tap * a.Cin + kb * kKBlock, t * 128);
                if (++st == a.stages) { st = 0; ++use; }
            }
        }
        __syncwarp();
    } else if (warp < 4) {
        // =========================== MMA issuers: warp 1 + t owns channel tile t ===========================
        // One elected thread per tile runs the whole loop (no per-iteration warp reconvergence): three issuing threads keep
        // the tensor pipe's queue full, each stage is released when all of them have committed.
        const int t = warp - 1;
        if (t < a.co_tiles && elect_one()) {
            const uint32_t idesc = make_idesc(a.fmt, 128, a.N);
            const uint64_t desc_hi = (uint64_t)((1024u >> 4) | (1u << 14) | (2u << 29)) << 32;  // SBO = 1024 B, SWIZZLE_128B
            const uint32_t d_tmem = tmem_base + (uint32_t)(t * a.acc_stride);
            const uint32_t w_off = (uint32_t)((t * kWTileBytes) >> 4), x_off = (uint32_t)((a.co_tiles * kWTileBytes) >> 4);
            const uint32_t stage16 = (uint32_t)(a.stage_bytes >> 4);
            const uint32_t s0_lo = (smem_u32(stage0) >> 4) | (1u << 16);
            int st = 0;
            uint32_t use = 0, s_lo = s0_lo;
            for (int it = 0; it < iters; ++it) {
                mbar_wait(&full[st], use & 1u);
                tc_fence_after();
                const uint64_t wd = desc_hi | (uint64_t)(s_lo + w_off), xd = desc_hi | (uint64_t)(s_lo + x_off);
                tc_mma<false>(d_tmem, wd, xd, idesc, it != 0);
                tc_mma<false>(d_tmem, wd + 2, xd + 2, idesc, 1);
                tc_mma<false>(d_tmem, wd + 4, xd + 4, idesc, 1);
                tc_mma<false>(d_tmem, wd + 6, xd + 6, idesc, 1);
                tc_commit(&empty[st]);
                s_lo += stage16;
                if (++st == a.stages) { st = 0; ++use; s_lo = s0_lo; }
            }
            tc_commit(acc_full);
        }
        __syncwarp();
    } else {
        // =========================== epilogue: thread = output channel (TMEM lane), columns = positions ===================
        const int quad = warp & 3;
        if constexpr (kVitTokens) {
            // the class-token row of this image, while the MMAs run
            if (strip == 0) {
                float* row0 = a.out + (int64_t)b * (a.H * a.W + 1) * a.Cout;
                for (int c = tid - 4 * 32; c < a.Cout; c += 4 * 32) row0[c] = a.cls_token[c] + a.pos_embed[c];
            }
        }
        mbar_wait(acc_full, 0);
        tc_fence_after();
        const int HW = a.H * a.W;
        const int pos0 = y0 * a.W;
        for (int t = 0; t < a.co_tiles; ++t) {
            const int co = t * 128 + quad * 32 + lane;
            const float sh = co < a.Cout ? a.shift[co] : 0.f;
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(t * a.acc_stride);
            for (int j0 = 0; j0 < a.N; j0 += 16) {
                float v[16];
                tmem_ld16_wait(taddr + (uint32_t)j0, v);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    v[i] += sh;
                    if (a.relu) v[i] = fmaxf(v[i], 0.f);
                }
                if (co < a.Cout) {
                    if constexpr (kVitTokens) {
                        // token row 1 + pos of image b, + pos_embed[1 + pos]: the same coalesced pattern on both sides
                        const int64_t r0 = 1 + pos0 + j0;
                        float* dst = a.out + ((int64_t)b * (HW + 1) + r0) * a.Cout + co;
                        const float* pe = a.pos_embed + r0 * a.Cout + co;
                        float p[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) p[i] = pos0 + j0 + i < HW ? __ldg(pe + (int64_t)i * a.Cout) : 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (pos0 + j0 + i < HW) dst[(int64_t)i * a.Cout] = v[i] + p[i];
                    } else if (a.out_layout == P3P_LAYOUT_NLC) {
                        // token rows: a warp writes 32 consecutive channels of one position per store
                        float* dst = a.out + ((int64_t)b * HW + pos0 + j0) * a.c_total + a.c_offset + co;
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (pos0 + j0 + i < HW) dst[(int64_t)i * a.c_total] = v[i];
                    } else {
                        float* dst = a.out + ((int64_t)b * a.c_total + a.c_offset + co) * HW + pos0 + j0;
                        if (pos0 + j0 + 16 <= HW && (((int64_t)HW) & 3) == 0) {
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                reinterpret_cast<float4*>(dst)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i)
                                if (pos0 + j0 + i < HW) dst[i] = v[i];
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// weight preparation: fold BatchNorm2d (eval) into the convolution, pack 16-bit K-major
// ------------------------------------------------------------------------------------------------
__global__ void conv3x3_prepare_kernel(p3p_conv_params p, int fmt, unsigned short* wp, float* shift, int cout_pad) {
    const int K = 9 * p.in_channels;
    const int64_t total = (int64_t)cout_pad * K;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int co = (int)(i / K), k = (int)(i - (int64_t)co * K);
        const int tap = k / p.in_channels, ci = k - tap * p.in_channels;
        float v = 0.f;
        if (co < p.out_channels) {
            const float a = p.norm_weight ? p.norm_weight[co] / sqrtf(p.norm_var[co] + p.eps) : 1.f;
            v = a * p.weight[((int64_t)co * p.in_channels + ci) * 9 + tap];  // (Cout, Cin, 3, 3): tap = ky * 3 + kx
        }
        wp[i] = fmt == 1 ? (unsigned short)(pack_bf16(v, 0.f) & 0xFFFF) : __half_as_ushort(__float2half_rn(v));
    }
    for (int co = blockIdx.x * blockDim.x + threadIdx.x; co < cout_pad; co += gridDim.x * blockDim.x) {
        float sh = 0.f;
        if (co < p.out_channels) {
            const float bias = p.bias ? p.bias[co] : 0.f;
            if (p.norm_weight) {
                const float a = p.norm_weight[co] / sqrtf(p.norm_var[co] + p.eps);
                sh = a * (bias - p.norm_mean[co]) + p.norm_bias[co];
            } else {
                sh = bias;
            }
        }
        shift[co] = sh;
    }
}

// fp32 NCHW (B, C, H, W) -> 16-bit channels-last (B, H, W, c_total) at channel offset c_offset (32 x 32 tiles through
// shared memory: coalesced on both sides)
__global__ void nchw_to_nhwc16_kernel(const float* __restrict__ x, int C, int HW, int fmt, unsigned short* __restrict__ out, int c_total,
                                      int c_offset) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;  // (32, 8)
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, p = p0 + tx;
        tile[r][tx] = (c < C && p < HW) ? x[((int64_t)b * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int p = p0 + r, c = c0 + tx;
        if (p < HW && c < C) {
            const float v = tile[tx][r];
            out[((int64_t)b * HW + p) * c_total + c_offset + c] =
                fmt == 1 ? (unsigned short)(pack_bf16(v, 0.f) & 0xFFFF) : __half_as_ushort(__float2half_rn(v));
        }
    }
}

// Bilinear upsampling (nn.Upsample(size, mode='bilinear', align_corners=False)) of fp32 token rows (B, h w, C) -- the ViT
// output after the class token is dropped, i.e. `x.permute(0, 2, 1).view(B, C, h, w)` read in place -- into 16-bit
// channels-last (B, H, W, C).  Source index = (dst + 0.5) * scale - 0.5 clamped at 0, as ATen's upsample_bilinear2d.
__global__ void upsample_bilinear_nhwc16_kernel(const float* __restrict__ x, int h, int w, int C, int64_t src_batch_stride, int H, int W,
                                                int fmt, unsigned short* __restrict__ out) {
    const int b = blockIdx.z, oy = blockIdx.y;
    const float sy = (float)h / (float)H, sx = (float)w / (float)W;
    float fy = ((float)oy + 0.5f) * sy - 0.5f;
    fy = fy < 0.f ? 0.f : fy;
    const int y0 = (int)fy, y1 = y0 + (y0 < h - 1 ? 1 : 0);
    const float ly = fy - (float)y0, hy = 1.f - ly;
    const float* src = x + (int64_t)b * src_batch_stride;
    const int64_t total = (int64_t)W * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ox = (int)(i / C), c = (int)(i - (int64_t)ox * C);
        float fx = ((float)ox + 0.5f) * sx - 0.5f;
        fx = fx < 0.f ? 0.f : fx;
        const int x0 = (int)fx, x1 = x0 + (x0 < w - 1 ? 1 : 0);
        const float lx = fx - (float)x0, hx = 1.f - lx;
        const float v00 = src[((int64_t)y0 * w + x0) * C + c], v01 = src[((int64_t)y0 * w + x1) * C + c];
        const float v10 = src[((int64_t)y1 * w + x0) * C + c], v11 = src[((int64_t)y1 * w + x1) * C + c];
        const float v = hy * (hx * v00 + lx * v01) + ly * (hx * v10 + lx * v11);
        out[(((int64_t)b * H + oy) * W + ox) * C + c] =
            fmt == 1 ? (unsigned short)(pack_bf16(v, 0.f) & 0xFFFF) : __half_as_ushort(__float2half_rn(v));
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace

size_t conv3x3_blob_bytes(int Cin, int Cout) {
    const size_t cout_pad = ((size_t)Cout + 127) / 128 * 128;
    return cout_pad * 9 * (size_t)Cin * 2 + cout_pad * 4;
}

int launch_conv3x3_prepare(const p3p_conv_params* p, int precision, void* blob, cudaStream_t st) {
    const int cout_pad = (p->out_channels + 127) / 128 * 128;
    unsigned short* wp = static_cast<unsigned short*>(blob);
    float* shift = reinterpret_cast<float*>(static_cast<char*>(blob) + (size_t)cout_pad * 9 * p->in_channels * 2);
    conv3x3_prepare_kernel<<<256, 256, 0, st>>>(*p, precision == P3P_PRECISION_BF16 ? 1 : 0, wp, shift, cout_pad);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_nchw_to_nhwc16(const float* x, int B, int C, int H, int W, int precision, void* out, int c_total, int c_offset, cudaStream_t st) {
    if (B <= 0) return P3P_OK;
    const int HW = H * W;
    dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
    nchw_to_nhwc16_kernel<<<grid, dim3(32, 8), 0, st>>>(x, C, HW, precision == P3P_PRECISION_BF16 ? 1 : 0, static_cast<unsigned short*>(out),
                                                         c_total, c_offset);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_upsample_bilinear_nhwc16(const float* x, int B, int h, int w, int C, int64_t src_batch_stride, int H, int W, int precision,
                                    void* out, cudaStream_t st) {
    if (B <= 0) return P3P_OK;
    const int64_t per_row = (int64_t)W * C;
    int bx = (int)((per_row + 255) / 256);
    if (bx > 64) bx = 64;
    dim3 grid((unsigned)bx, (unsigned)H, (unsigned)B);
    upsample_bilinear_nhwc16_kernel<<<grid, 256, 0, st>>>(x, h, w, C, src_batch_stride, H, W, precision == P3P_PRECISION_BF16 ? 1 : 0,
                                                          static_cast<unsigned short*>(out));
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

namespace {

// cls_token / pos_embed non-null: the ViT-token epilogue (out: (B, 1 + H W, Cout); out_layout, c_total, c_offset unused)
int launch_conv3x3_any(const void* x, int B, int H, int W, int Cin, const void* blob, int Cout, int precision, int relu, float* out,
                       int out_layout, int c_total, int c_offset, const float* cls_token, const float* pos_embed, cudaStream_t st) {
    if (B <= 0) return P3P_OK;
    if (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16)
        return fail(P3P_ERR_UNSUPPORTED, "conv3x3 runs on 16-bit operands (precision bf16 or fp16), got %d", precision);
    if (Cin % kKBlock != 0) return fail(P3P_ERR_UNSUPPORTED, "conv3x3 needs in_channels a multiple of %d, got %d", kKBlock, Cin);
    const int co_tiles = (Cout + 127) / 128;
    if (co_tiles > 3) return fail(P3P_ERR_UNSUPPORTED, "conv3x3 supports up to 384 output channels (one issuing warp per 128), got %d", Cout);
    // strip height: rows * W a multiple of 16, <= 256, co_tiles accumulators of rows * W columns inside the 512 TMEM columns,
    // box dimensions <= 256; the tallest strip wins (weight tiles are re-read per strip)
    if (W > 256) return fail(P3P_ERR_UNSUPPORTED, "conv3x3 supports widths up to 256, got %d", W);
    int rows = 0;
    for (int r = 1; r <= H && r * W <= 256; ++r)
        if ((r * W) % 16 == 0 && co_tiles * (r * W <= 128 ? 128 : 256) <= 512) rows = r;
    if (rows == 0) return fail(P3P_ERR_UNSUPPORTED, "conv3x3: no strip of whole rows of width %d is a multiple of 16 positions within TMEM (%d channel tiles)", W, co_tiles);
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(P3P_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout;
    a.rows = rows; a.N = rows * W; a.strips = (H + rows - 1) / rows; a.co_tiles = co_tiles;
    a.acc_stride = a.N <= 128 ? 128 : 256;
    a.stage_bytes = co_tiles * kWTileBytes + (a.N * kKBlockBytes + 1023) / 1024 * 1024;
    a.stages = (int)((200 * 1024) / a.stage_bytes);
    if (a.stages > 8) a.stages = 8;
    if (a.stages < 2) return fail(P3P_ERR_UNSUPPORTED, "conv3x3: operand stage of %d bytes does not fit shared memory twice", a.stage_bytes);
    a.fmt = precision == P3P_PRECISION_BF16 ? 1 : 0;
    a.relu = relu;
    const int cout_pad = co_tiles * 128;
    a.shift = reinterpret_cast<const float*>(static_cast<const char*>(blob) + (size_t)cout_pad * 9 * Cin * 2);
    a.out = out; a.out_layout = out_layout; a.c_total = c_total; a.c_offset = c_offset;
    a.cls_token = cls_token; a.pos_embed = pos_embed;

    CUtensorMap tm_x, tm_w;
    const CUtensorMapDataType dt = precision == P3P_PRECISION_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    {
        const cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        const cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cin * 2 * W, (cuuint64_t)Cin * 2 * W * H};
        const cuuint32_t box[4] = {(cuuint32_t)kKBlock, (cuuint32_t)W, (cuuint32_t)rows, 1};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult r = enc(&tm_x, dt, 4, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(P3P_ERR_CUDA, "cuTensorMapEncodeTiled (activations) failed: %d", (int)r);
    }
    {
        const cuuint64_t dims[2] = {(cuuint64_t)9 * Cin, (cuuint64_t)cout_pad};
        const cuuint64_t strides[1] = {(cuuint64_t)9 * Cin * 2};
        const cuuint32_t box[2] = {(cuuint32_t)kKBlock, 128};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = enc(&tm_w, dt, 2, const_cast<void*>(blob), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(P3P_ERR_CUDA, "cuTensorMapEncodeTiled (weights) failed: %d", (int)r);
    }
    const size_t smem = (size_t)a.stages * a.stage_bytes + (2 * 8 + 1) * 8 + 16;
    auto* kernel = pos_embed ? conv3x3_tc_kernel<true> : conv3x3_tc_kernel<false>;
    P3P_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * a.strips));
    cfg.blockDim = dim3(kConvThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    P3P_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, tm_x, tm_w, a));
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

}  // namespace

int launch_conv3x3(const void* x, int B, int H, int W, int Cin, const void* blob, int Cout, int precision, int relu, float* out,
                   int out_layout, int c_total, int c_offset, cudaStream_t st) {
    return launch_conv3x3_any(x, B, H, W, Cin, blob, Cout, precision, relu, out, out_layout, c_total, c_offset, nullptr, nullptr, st);
}

int launch_conv3x3_vit_tokens(const void* x, int B, int H, int W, int Cin, const void* blob, int Cout, int precision,
                              const float* cls_token, const float* pos_embed, float* out, cudaStream_t st) {
    return launch_conv3x3_any(x, B, H, W, Cin, blob, Cout, precision, 1, out, P3P_LAYOUT_NLC, Cout, 0, cls_token, pos_embed, st);
}

}  // namespace p3p
