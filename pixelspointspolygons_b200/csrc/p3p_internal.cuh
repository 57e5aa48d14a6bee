// p3p_internal.cuh -- shared declarations of libp3p.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "p3p.h"

namespace p3p {

// ----------------------------------------------------------------------------------------------
// error plumbing (capi.cu owns the thread-local message)
// ----------------------------------------------------------------------------------------------
int fail(int code, const char* fmt, ...);
#define P3P_CUDA_CHECK(expr)                                                                   \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess)                                                                 \
            return ::p3p::fail(P3P_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                               __FILE__, __LINE__);                                            \
    } while (0)

// ----------------------------------------------------------------------------------------------
// grid constants, derived on the host with the same fp32 operations as Open3D's VoxelizeCPU
// (SURVEY Appendix A.1 / A.2) and passed to every kernel by value
// ----------------------------------------------------------------------------------------------
constexpr int kFlagDropOverflow = P3P_GRID_DROP_OVERFLOW;  // DESIGN.md uncertainty ledger U1
constexpr int kMaxKeys = 6144;        // smem histogram budget of the ranking kernels
// voxelizer shape: a chunk holds threads * points-per-lane points and the whole batch should be ONE wave of CTAs (capi.cu
// sizes the chunks for that).  The CTA shape does not matter (DESIGN 4.1: 512 x 2 x 12 and 384 x 2 x 16 measured no faster).
constexpr int kVoxThreads = 256;                                // threads per CTA
constexpr int kVoxCtasPerSm = 3;                                // CTAs per SM
constexpr int kChunkGranule = 4 * kVoxThreads;                  // every lane owns whole groups of 4 points
constexpr int kMaxChunkPoints = kVoxThreads * 16;               // points per ranking chunk held in registers (16 per lane)
constexpr int kC0 = 32;               // feat_channels[0] / 2: width of PFN layer 0

struct GridDev {
    float mn[3], mx[3], inv[3];
    int ext[3];        // int32(ceil((max - min) * inv))
    int nv[3];         // int32((max - min) / voxel_size): x/y bound of the pillar filter
    int stride1, stride2;
    int num_cells;     // ext0 * ext1 * ext2 (upstream's batch_hash)
    int num_keys;      // largest reachable hash + 1
    int M, Vmax, ny, nx;
    int flags;
    float vx, vy, x_off, y_off;  // PillarFeatureNet: vx, vy, vx/2 + min_x, vy/2 + min_y
    float fix_scale, fix_inv;    // fixed-point grid of the cluster-mean sums (2^k, 2^-k): order-independent, exact
    float fix2_scale, fix2_inv;  // coarser grid whose sum over M slots fits one int32 (tensor-core kernel); 0: not available
};

int make_grid(const p3p_grid* g, GridDev* out);

// ----------------------------------------------------------------------------------------------
// workspace carve-up (all offsets 256-byte aligned)
// ----------------------------------------------------------------------------------------------
struct WsLayout {
    int B;
    int chunk_points;      // S: points per ranking chunk (multiple of kChunkGranule, <= kMaxChunkPoints)
    int max_chunks;        // upper bound of the number of chunks over the batch (= grid of the voxelize kernel)
    int key_stride;        // chunk_hist row stride (elements)
    size_t off_sync;       // uint32 ticket, flags[max_chunks], tile_done[B], tile_sat[B], then uint8 edge[B][num_keys]
    size_t sync_bytes;     //   (one block, zeroed at the start of every call)
    size_t off_edge;       // uint8 [B][num_keys]: the run of this key holds a point on the x / y max face (cell == extent),
                           //   i.e. its coordinates are not decodable from the key (hash aliasing, SURVEY A.1)
    size_t off_chunk_hist; // uint16 [max_chunks][key_stride]
    size_t off_totals;     // int32  [B][num_keys]   uncapped points per key
    size_t off_slots;      // float4 [B][num_keys][M] (x, y, z, bits(tile-local index)): the min(count, M) lowest-index
                           //   points of the key, in no particular order
    size_t off_pil_key;    // int32  [B][Vmax]       key of pillar r (voxel order, after both filters)
    size_t off_pil_n;      // int32  [B][Vmax]       min(count, M)
    size_t off_pil_coord;  // int32  [B][Vmax]       cx | cy << 10 | cz << 20
    size_t off_num_pil;    // int32  [B]
    size_t off_tile_hi;    // int32  [B]             bit 0: keys beyond the regular cells in use; bit 1: owner table written without a plan
    size_t off_owner;      // int32  [B][ny*nx]      voxel ordinal owning the canvas cell, -1 = empty
    size_t off_cell_desc;  // int32  [B][ny*nx]      key | n << 16 of the owning pillar, -1 = empty
    size_t off_train_list; // int4   [B][Vmax]       training kernels: the batch's pillars, compacted (pfn_train.cu)
    size_t off_train_count;// int32  [4]             their number
    size_t total_bytes;
};

int make_ws_layout(const GridDev& g, int B, int64_t total_points, WsLayout* out);
constexpr size_t kVoxelizeMaxSmem = 200 * 1024;  // dynamic shared memory the voxelize kernel may opt in to
size_t voxelize_smem_bytes(const GridDev& g);

struct WsPtrs {
    unsigned* sync;
    int max_chunks;
    int key_stride;  // row stride of chunk_hist in elements (num_keys rounded up to 8)
    uint16_t* chunk_hist;
    uint8_t* edge;
    int32_t* totals;
    float4* slots;
    int32_t* pil_key;
    int32_t* pil_n;
    int32_t* pil_coord;
    int32_t* num_pil;
    int32_t* tile_hi;
    int32_t* owner;
    int32_t* cell_desc;
    int4* train_list;
    int32_t* train_count;
};

inline WsPtrs ws_ptrs(void* base, const WsLayout& l) {
    char* b = static_cast<char*>(base);
    WsPtrs p;
    p.sync = reinterpret_cast<unsigned*>(b + l.off_sync);
    p.max_chunks = l.max_chunks;
    p.key_stride = l.key_stride;
    p.chunk_hist = reinterpret_cast<uint16_t*>(b + l.off_chunk_hist);
    p.edge = reinterpret_cast<uint8_t*>(b + l.off_edge);
    p.totals = reinterpret_cast<int32_t*>(b + l.off_totals);
    p.slots = reinterpret_cast<float4*>(b + l.off_slots);
    p.pil_key = reinterpret_cast<int32_t*>(b + l.off_pil_key);
    p.pil_n = reinterpret_cast<int32_t*>(b + l.off_pil_n);
    p.pil_coord = reinterpret_cast<int32_t*>(b + l.off_pil_coord);
    p.num_pil = reinterpret_cast<int32_t*>(b + l.off_num_pil);
    p.tile_hi = reinterpret_cast<int32_t*>(b + l.off_tile_hi);
    p.owner = reinterpret_cast<int32_t*>(b + l.off_owner);
    p.cell_desc = reinterpret_cast<int32_t*>(b + l.off_cell_desc);
    p.train_list = reinterpret_cast<int4*>(b + l.off_train_list);
    p.train_count = reinterpret_cast<int32_t*>(b + l.off_train_count);
    return p;
}

// ----------------------------------------------------------------------------------------------
// prepared-weights blob (written by pfn_prepare_kernel, read by the PFN kernels)
// ----------------------------------------------------------------------------------------------
struct BlobLayout {
    int C, Cpad, MT;      // channels, padded to 128, number of 128-channel MMA tiles
    size_t off_header;    // int32[16]: magic, precision, C, Cpad, center_alias
    size_t off_front;     // float[10][32]: Ux,Uy,Uz, Kcx,Kcy, Wmx,Wmy,Wmz, b0, hpad   (affine form of layer 0)
    size_t off_w0;        // float[32][8]  a0 * W0           (literal form, fp32 kernel)
    size_t off_b0;        // float[32]
    size_t off_w1;        // float[Cpad][64] a1 * W1         (literal form, fp32 kernel)
    size_t off_b1;        // float[Cpad]
    size_t off_a1;        // MMA A operand of W1[:, :32] (K-major, swizzled), MT tiles of 128 rows
    size_t off_a2;        // MMA A operand of W1[:, 32:]
    size_t total_bytes;
};
constexpr int kBlobMagic = 0x50335031;  // "P3P1"

void make_blob_layout(int C, BlobLayout* out);

// item sources of the PFN kernels
constexpr int kItemsCanvas = 0;  // item = b * (ny*nx) + cell, resolved through the owner table
constexpr int kItemsList = 1;    // item = b * Vmax + r, r < num_pil[b]

struct PfnArgs {
    GridDev g;
    WsPtrs ws;
    const char* blob;
    BlobLayout bl;
    int B;
    int item_mode;
    int64_t num_items;
    int items_per_tile;
    // output addressing: NLC / list: out[item * C + c]; NCHW: out[((b * c_total + c_offset + c) * HW) + cell]
    void* out;
    int out_layout;  // P3P_LAYOUT_*
    int out_dtype;   // P3P_DTYPE_*
    int c_total, c_offset;
    int blk_shift;               // tensor-core kernel, M > 64: log2 of the 64-row blocks per pillar (0: one block)
    int row_stride, row_offset;  // rows layouts: out[item * row_stride + row_offset + c] (row_stride = C when the rows are dense)
    // token sequence output (p3p_encode_tokens): rows of C channels, 1 + items_per_tile rows per tile, row 0 = class
    // token; pos_embed (1 + items_per_tile, C) is added to every row.  token_rows == 0: off
    const float* pos_embed;
    int token_rows;
};

// launchers (host) ---------------------------------------------------------------------------------
int launch_voxelize(const float* pts, int stride, const int64_t* offsets, int B, int64_t total, const GridDev& g,
                    const WsLayout& l, const WsPtrs& ws, int32_t* point_hash, int need_plan, cudaStream_t st);
int launch_export(const GridDev& g, int B, const WsPtrs& ws, const p3p_voxel_outputs* out, cudaStream_t st);
int launch_pfn_prepare(const p3p_pfn_params* p, int precision, char* blob, const BlobLayout& bl, cudaStream_t st);
int launch_pfn_simt(const PfnArgs& a, cudaStream_t st);
int launch_pfn_tc(const PfnArgs& a, int precision, cudaStream_t st);
int launch_zero_lidar(const PfnArgs& a, cudaStream_t st);
int launch_cls_rows(const PfnArgs& a, const float* cls_token, cudaStream_t st);
size_t patch_embed_blob_bytes(int C, int in_chans, int P);
int launch_patch_embed_prepare(const float* weight, const float* bias, int C, int in_chans, int P, int precision, void* blob, cudaStream_t st);
int launch_patch_embed(const float* images, int B, int in_chans, int H, int W, int P, const float* weight, const float* bias,
                       const void* blob, int C, int precision, void* out, int out_dtype, int out_layout, int c_total, int c_offset,
                       cudaStream_t st, const uint8_t* images_u8 = nullptr, const float* pixel_lut = nullptr);
int launch_las_to_pixels(const int32_t* X, const int32_t* Y, const int32_t* Z, const uint16_t* deltas, const int32_t* base,
                         const int64_t* offsets, int B, int64_t total, const p3p_las_tile* tiles, double z_hi, int32_t* mm, float* out,
                         cudaStream_t st);
size_t conv3x3_blob_bytes(int Cin, int Cout);
int launch_conv3x3_prepare(const p3p_conv_params* p, int precision, void* blob, cudaStream_t st);
int launch_conv3x3(const void* x, int B, int H, int W, int Cin, const void* blob, int Cout, int precision, int relu, float* out,
                   int out_layout, int c_total, int c_offset, cudaStream_t st);
int launch_conv3x3_vit_tokens(const void* x, int B, int H, int W, int Cin, const void* blob, int Cout, int precision,
                              const float* cls_token, const float* pos_embed, float* out, cudaStream_t st);
int launch_nchw_to_nhwc16(const float* x, int B, int C, int H, int W, int precision, void* out, int c_total, int c_offset, cudaStream_t st);
int launch_upsample_bilinear_nhwc16(const float* x, int B, int h, int w, int C, int64_t src_batch_stride, int H, int W, int precision,
                                    void* out, cudaStream_t st);
int device_sm_count();
size_t device_smem_optin();  // shared memory one CTA may opt in to, static + dynamic (cudaDevAttrMaxSharedMemoryPerBlockOptin)

// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// cell hash of one point, or -1 (Open3D VoxelizeCPU HashFn; fp32 subtract then multiply, truncation)
// `edge` is set when the point sits on the x or y max face (cell index == extent): only such points make a hash
// ambiguous (cx == ext_x aliases (0, cy + 1); cy == ext_y aliases (cx, 0, cz + 1)).
template <bool kCheckOverflow = true>
__device__ __forceinline__ int point_key(const GridDev& g, float x, float y, float z, bool& edge) {
    // branch-free: the cell indices of an invalid point (NaN, out of range) are garbage and masked below
    const bool valid = (x >= g.mn[0]) & (x <= g.mx[0]) & (y >= g.mn[1]) & (y <= g.mx[1]) & (z >= g.mn[2]) & (z <= g.mx[2]);
    const int cx = __float2int_rz(__fmul_rn(__fsub_rn(x, g.mn[0]), g.inv[0]));
    const int cy = __float2int_rz(__fmul_rn(__fsub_rn(y, g.mn[1]), g.inv[1]));
    const int cz = __float2int_rz(__fmul_rn(__fsub_rn(z, g.mn[2]), g.inv[2]));
    const int h = cx + cy * g.stride1 + cz * g.stride2;
    bool ok = valid;
    if (kCheckOverflow) ok = ok & !((g.flags & kFlagDropOverflow) && h >= g.num_cells);
    edge = ok & ((cx >= g.ext[0]) | (cy >= g.ext[1]));
    return ok ? h : -1;
}

__device__ __forceinline__ void point_cell(const GridDev& g, float x, float y, float z, int& cx, int& cy, int& cz) {
    cx = __float2int_rz(__fmul_rn(__fsub_rn(x, g.mn[0]), g.inv[0]));
    cy = __float2int_rz(__fmul_rn(__fsub_rn(y, g.mn[1]), g.inv[1]));
    cz = __float2int_rz(__fmul_rn(__fsub_rn(z, g.mn[2]), g.inv[2]));
}

// One pillar as seen by the PFN kernels.
struct Item {
    int valid;            // 0: empty canvas cell / padding row of the list
    int b;                // tile
    int n;                // min(count, M)
    int key;              // slot row of the pillar
    float ctr_x, ctr_y;   // pillar centre: cx * vx + x_off, cy * vy + y_off
    int cell;             // canvas cell (cy * nx + cx)
};

__device__ __forceinline__ const float4* item_slots(const PfnArgs& a, const Item& it) {
    return a.ws.slots + ((int64_t)it.b * a.g.num_keys + it.key) * a.g.M;
}

// One dependent-load level: canvas items read cell_desc, list items read the pillar table.
__device__ __forceinline__ Item fetch_item(const PfnArgs& a, int64_t item) {
    Item it;
    it.valid = 0; it.n = 0; it.key = 0; it.ctr_x = 0.f; it.ctr_y = 0.f; it.cell = 0; it.b = 0;
    if (item >= a.num_items) return it;
    const int b = (int)item / a.items_per_tile;  // (the launchers bound num_items to 31 bits: one 32-bit division)
    const int r = (int)item - b * a.items_per_tile;
    it.b = b;
    int cx, cy;
    if (a.item_mode == kItemsCanvas) {
        const int d = __ldg(a.ws.cell_desc + item);
        it.cell = r;
        if (d < 0) return it;
        it.key = d & 0xFFFF;
        it.n = d >> 16;
        cy = r / a.g.nx;
        cx = r - cy * a.g.nx;
    } else {
        if (r >= a.ws.num_pil[b]) return it;
        const int64_t pi = (int64_t)b * a.g.Vmax + r;
        it.key = a.ws.pil_key[pi];
        it.n = a.ws.pil_n[pi];
        const int pc = a.ws.pil_coord[pi];
        cx = pc & 1023;
        cy = (pc >> 10) & 1023;
        it.cell = cy * a.g.nx + cx;
    }
    it.valid = 1;
    it.ctr_x = __fmaf_rn((float)cx, a.g.vx, a.g.x_off);
    it.ctr_y = __fmaf_rn((float)cy, a.g.vy, a.g.y_off);
    return it;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{.reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0];}" ::"r"(smem_u32(bar)) : "memory");
}
// plain shared-memory accesses by 32-bit shared address (no generic-pointer arithmetic in the hot loops)
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ uint2 lds_u32x2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
// the same on a precomputed 32-bit shared address (kept in a register: `opaque` stops the compiler from re-deriving it
// from the thread index at every use)
__device__ __forceinline__ uint32_t opaque(uint32_t x) {
    asm volatile("" : "+r"(x));
    return x;
}
__device__ __forceinline__ void mbar_arrive_sa(uint32_t bar) {
    asm volatile("{.reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0];}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_sa(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{.reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p;}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_sa(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait_sa(bar, parity)) {
    }
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) { return mbar_try_wait_sa(smem_u32(bar), parity); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_sa(smem_u32(bar), parity); }
// arrive and expect `bytes` of async-copy transactions (TMA / bulk copies completing on the barrier)
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_test_sa(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{.reg .pred p; mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p;}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 --------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// arrive on an mbarrier when all tcgen05 ops previously issued by this thread have completed
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
template <bool kTf32>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    if constexpr (kTf32) {
        asm volatile(
            "{.reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;}" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
            : "memory");
    } else {
        asm volatile(
            "{.reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;}" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
            : "memory");
    }
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{.reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p;}" : "=r"(pred));
    return pred != 0;
}
// K-major smem operand descriptor (cute::UMMA::SmemDescriptor, version 1): 8-row groups `sbo` bytes apart
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type) {
    const uint32_t lo = ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
    const uint32_t hi = (sbo_bytes >> 4) | (1u << 14) | (layout_type << 29);
    return ((uint64_t)hi << 32) | lo;
}
// cute::UMMA::InstrDescriptor: dense, fp32 accumulate, both operands K-major
__device__ __forceinline__ uint32_t make_idesc(int fmt_code, int m, int n) {
    const uint32_t fmt = (uint32_t)fmt_code;  // F16F32Format: F16 = 0, BF16 = 1, TF32 = 2
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// tcgen05.ld + tcgen05.wait::ld in ONE asm statement: the destination registers are only defined once the wait has
// retired, so no consumer can be scheduled between the load and the wait.
__device__ __forceinline__ void tmem_ld16_wait(uint32_t taddr, float (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
          "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
        : "r"(taddr)
        : "memory");
}
// Split form for software pipelining inside a warp: issue a load, then later wait for every outstanding load of the
// thread.  The wait lists the registers of the load(s) it completes as in/out operands so that no consumer can be
// scheduled above it; ptxas tracks tcgen05.ld with a scoreboard, so arithmetic on registers of an EARLIER, already
// awaited load overlaps with a load that is still in flight.
#define P3P_R16(v)                                                                                                        \
    "+f"(v[0]),"+f"(v[1]),"+f"(v[2]),"+f"(v[3]),"+f"(v[4]),"+f"(v[5]),"+f"(v[6]),"+f"(v[7]),"+f"(v[8]),"+f"(v[9]),"+f"(v[10]),   \
    "+f"(v[11]),"+f"(v[12]),"+f"(v[13]),"+f"(v[14]),"+f"(v[15])
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, float (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=f"(v[0]),"=f"(v[1]),"=f"(v[2]),"=f"(v[3]),"=f"(v[4]),"=f"(v[5]),"=f"(v[6]),"=f"(v[7]),"=f"(v[8]),"=f"(v[9]),"=f"(v[10]),"=f"(v[11]),"=f"(v[12]),"=f"(v[13]),"=f"(v[14]),"=f"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(float (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" : P3P_R16(v) : : "memory");
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float warp_max_f32(float v) {
    float r;
    asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ uint32_t to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ unsigned short to_16bit(float v, int dtype) {  // P3P_DTYPE_BF16 / P3P_DTYPE_F16
    unsigned short r;
    if (dtype == P3P_DTYPE_F16)
        asm("cvt.rn.f16.f32 %0, %1;" : "=h"(r) : "f"(v));
    else
        asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// packed fp32 FMA (FFMA2): two lanes per instruction
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(d)
        : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)),
          "l"(*reinterpret_cast<unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}
// Cluster-mean sums on a fixed-point grid: q = rn(v * 2^k), |q| < 2^30, summed exactly as two 16-bit halves
// (<= 1024 terms each) -- independent of the order of the slots, hence bitwise reproducible.
__device__ __forceinline__ void fix_split(float v, float scale, int& lo, int& hi) {
    const int q = __float2int_rn(v * scale);
    lo = q & 0xFFFF;
    hi = q >> 16;
}
__device__ __forceinline__ float fix_mean(int sum_lo, int sum_hi, float inv_scale, float n) {
    return __fdiv_rn(__fmaf_rn((float)sum_hi, 65536.0f, (float)sum_lo) * inv_scale, n);
}

#endif  // __CUDACC__

}  // namespace p3p
