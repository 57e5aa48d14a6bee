// capi.cu -- extern "C" entry points of libp3p.so (declared in include/p3p.h).
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "p3p_internal.cuh"

namespace p3p {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int device_sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            sms = n;
        else
            sms = 148;  // B200; keeps p3p_workspace_bytes usable on a box without a GPU
        (void)cudaGetLastError();
    }
    return sms;
}

size_t device_smem_optin() {
    static size_t bytes = 0;
    if (bytes == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess && n > 0)
            bytes = (size_t)n;
        else
            bytes = 227 * 1024;  // sm_100 (the only target of this library); keeps the shape checks usable without a GPU
        (void)cudaGetLastError();
    }
    return bytes;
}

// Same fp32 operation sequence as Open3D VoxelizeCPU / PointPillarsVoxelization (SURVEY A.1, A.2).
int make_grid(const p3p_grid* g, GridDev* out) {
    if (!g) return fail(P3P_ERR_INVALID_ARGUMENT, "grid is null");
    GridDev d;
    memset(&d, 0, sizeof(d));
    for (int i = 0; i < 3; ++i) {
        if (!(g->voxel_size[i] > 0.f) || !(g->range_max[i] > g->range_min[i]))
            return fail(P3P_ERR_INVALID_ARGUMENT, "grid axis %d: voxel_size must be > 0 and range_max > range_min", i);
        d.mn[i] = g->range_min[i];
        d.mx[i] = g->range_max[i];
        volatile float inv = 1.0f / g->voxel_size[i];
        d.inv[i] = inv;
        volatile float span = g->range_max[i] - g->range_min[i];
        volatile float cells = span * inv;
        d.ext[i] = (int)ceilf(cells);
        volatile float q = span / g->voxel_size[i];
        d.nv[i] = (int)q;
        if (d.ext[i] < 1 || d.ext[i] > 1023) return fail(P3P_ERR_UNSUPPORTED, "grid axis %d: %d cells (supported: 1..1023)", i, d.ext[i]);
    }
    d.stride1 = d.ext[0];
    d.stride2 = d.ext[0] * d.ext[1];
    const long long cells = (long long)d.stride2 * d.ext[2];
    const long long keys = (long long)d.ext[0] + (long long)d.ext[1] * d.stride1 + (long long)d.ext[2] * d.stride2 + 1;
    d.flags = g->flags;
    d.num_cells = (int)cells;
    const long long nkeys = (g->flags & P3P_GRID_DROP_OVERFLOW) ? cells : keys;
    if (nkeys > kMaxKeys)
        return fail(P3P_ERR_UNSUPPORTED, "%lld pillar keys exceed the shared-memory ranking budget (%d)", nkeys, kMaxKeys);
    d.num_keys = (int)nkeys;
    if (g->max_points < 1 || g->max_points > 1024) return fail(P3P_ERR_UNSUPPORTED, "max_points %d (supported: 1..1024)", g->max_points);
    if (g->max_voxels < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "max_voxels %d", g->max_voxels);
    d.M = g->max_points;
    d.Vmax = g->max_voxels;
    d.ny = g->ny;
    d.nx = g->nx;
    // PointPillarsScatter writes canvas[:, y * nx + x]; the pillar filter bounds y < nv[1], x < nv[0].
    if (d.ny < d.nv[1] || d.nx < d.nv[0] || d.ny < 1 || d.nx < 1)
        return fail(P3P_ERR_INVALID_ARGUMENT, "scatter output_shape (%d, %d) smaller than the voxel grid (%d, %d)", d.ny, d.nx, d.nv[1], d.nv[0]);
    d.vx = g->voxel_size[0];
    d.vy = g->voxel_size[1];
    if (voxelize_smem_bytes(d) > kVoxelizeMaxSmem)
        return fail(P3P_ERR_UNSUPPORTED, "grid of %d keys and a %d x %d canvas needs %zu bytes of shared memory per CTA (limit %zu)",
                    d.num_keys, d.ny, d.nx, voxelize_smem_bytes(d), kVoxelizeMaxSmem);
    d.x_off = g->voxel_size[0] / 2 + g->range_min[0];
    d.y_off = g->voxel_size[1] / 2 + g->range_min[1];
    // fixed-point grid of the cluster-mean sums: |coordinate| * 2^k < 2^30, k <= 20
    float maxabs = 1.f;
    for (int i = 0; i < 3; ++i) maxabs = fmaxf(maxabs, fmaxf(fabsf(g->range_min[i]), fabsf(g->range_max[i])));
    int k = 30 - (int)ceilf(log2f(maxabs + 1.f));
    if (k > 20) k = 20;
    if (k < 0) return fail(P3P_ERR_UNSUPPORTED, "point_cloud_range magnitude %g too large", (double)maxabs);
    d.fix_scale = ldexpf(1.f, k);
    d.fix_inv = ldexpf(1.f, -k);
    // single-word variant: |coordinate| * 2^k2 * M < 2^31 (the tensor-core kernel sums a pillar's slots in one int32);
    // below 12 fractional bits the mean would lose accuracy against the fp32 contract -> not offered
    int mbits = 0;
    while ((1 << mbits) < g->max_points) ++mbits;
    int k2 = 30 - mbits - (int)ceilf(log2f(maxabs + 1.f));
    if (k2 > 20) k2 = 20;
    d.fix2_scale = k2 >= 12 ? ldexpf(1.f, k2) : 0.f;
    d.fix2_inv = k2 >= 12 ? ldexpf(1.f, -k2) : 0.f;
    *out = d;
    return P3P_OK;
}

int make_ws_layout(const GridDev& g, int B, int64_t total_points, WsLayout* out) {
    if (B < 0 || total_points < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "negative batch or point count");
    WsLayout l;
    memset(&l, 0, sizeof(l));
    l.B = B;
    const int target = kVoxCtasPerSm * device_sm_count();
    int64_t denom = target - B;
    if (denom < 64) denom = 64;
    int64_t S = (total_points + denom - 1) / denom;
    S = (S + kChunkGranule - 1) / kChunkGranule * kChunkGranule;  // every lane owns whole groups of 4 points
    if (S < kChunkGranule) S = kChunkGranule;
    if (S > kMaxChunkPoints) S = kMaxChunkPoints;
    l.chunk_points = (int)S;
    // chunks of a tile start at its first point rounded down to a multiple of 4: sum_b ceil((n_b + 3) / S) <= this
    const int64_t mc = (total_points + 3 * (int64_t)B) / S + B;
    if (mc > 0x7fffffff) return fail(P3P_ERR_UNSUPPORTED, "too many ranking chunks");
    l.max_chunks = (int)mc;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t HW = (size_t)g.ny * g.nx;
    const size_t sync_words = ((size_t)(1 + l.max_chunks + 2 * B) * sizeof(unsigned) + 15) / 16 * 16;
    l.sync_bytes = sync_words + (size_t)B * g.num_keys;  // ticket / flags / tile_done, then the edge flags: one memset
    l.off_sync = take(l.sync_bytes);
    l.off_edge = l.off_sync + sync_words;
    l.key_stride = (g.num_keys + 7) / 8 * 8;
    l.off_chunk_hist = take((size_t)l.max_chunks * l.key_stride * sizeof(uint16_t));
    l.off_totals = take((size_t)B * g.num_keys * sizeof(int32_t));
    l.off_slots = take((size_t)B * g.num_keys * g.M * sizeof(float4));
    l.off_pil_key = take((size_t)B * g.Vmax * sizeof(int32_t));
    l.off_pil_n = take((size_t)B * g.Vmax * sizeof(int32_t));
    l.off_pil_coord = take((size_t)B * g.Vmax * sizeof(int32_t));
    l.off_num_pil = take((size_t)B * sizeof(int32_t));
    l.off_tile_hi = take((size_t)B * sizeof(int32_t));
    l.off_owner = take((size_t)B * HW * sizeof(int32_t));
    l.off_cell_desc = take((size_t)B * HW * sizeof(int32_t));
    l.off_train_list = take((size_t)B * g.Vmax * sizeof(int4));
    l.off_train_count = take(4 * sizeof(int32_t));
    l.total_bytes = off;
    *out = l;
    return P3P_OK;
}

// per-thread profiling state (p3p_profile_begin / p3p_profile_end)
struct Profile {
    bool on = false;
    int used = 0;
    std::vector<cudaEvent_t> ev;  // 3 events per record: before voxelize, after voxelize, after PFN
};
static thread_local Profile g_prof;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int check_blob(int C, BlobLayout* bl) {
    if (C < 1 || C > 4096) return fail(P3P_ERR_INVALID_ARGUMENT, "channels %d", C);
    make_blob_layout(C, bl);
    return P3P_OK;
}

static int run_pfn(const PfnArgs& a, int precision, cudaStream_t st) {
    if (precision == P3P_PRECISION_FP32) return launch_pfn_simt(a, st);
    if (precision != P3P_PRECISION_TF32 && precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16)
        return fail(P3P_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
    // The tensor-core kernel covers the shipped encoder configs and the density ablation (M <= 512: a pillar takes 1, 2, 4
    // or 8 blocks of 64 operand rows; C <= 384); anything else takes the exact-fp32 kernel.
    if (a.g.M <= 512 && a.bl.MT <= 3 && a.g.fix2_scale > 0.f) return launch_pfn_tc(a, precision, st);
    return launch_pfn_simt(a, st);
}

}  // namespace p3p

using namespace p3p;

extern "C" {

const char* p3p_last_error(void) { return g_err; }
int p3p_version(void) { return P3P_VERSION; }

size_t p3p_workspace_bytes(const p3p_grid* grid, int32_t num_tiles, int64_t total_points) {
    GridDev g;
    WsLayout l;
    if (make_grid(grid, &g) != P3P_OK) return 0;
    if (make_ws_layout(g, num_tiles, total_points, &l) != P3P_OK) return 0;
    return l.total_bytes;
}

size_t p3p_pfn_blob_bytes(int32_t channels) {
    BlobLayout bl;
    if (check_blob(channels, &bl) != P3P_OK) return 0;
    return bl.total_bytes;
}

int p3p_pfn_prepare(const p3p_pfn_params* p, int32_t precision, void* blob, size_t blob_bytes, void* stream) {
    if (!p || !blob) return fail(P3P_ERR_INVALID_ARGUMENT, "null params or blob");
    if (!p->linear0_weight || !p->norm0_weight || !p->norm0_bias || !p->norm0_mean || !p->norm0_var ||
        !p->linear1_weight || !p->norm1_weight || !p->norm1_bias || !p->norm1_mean || !p->norm1_var)
        return fail(P3P_ERR_INVALID_ARGUMENT, "null weight pointer");
    if (precision < P3P_PRECISION_FP32 || precision > P3P_PRECISION_FP16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
    BlobLayout bl;
    int rc = check_blob(p->channels, &bl);
    if (rc) return rc;
    if (blob_bytes < bl.total_bytes) return fail(P3P_ERR_WORKSPACE, "blob needs %zu bytes, got %zu", bl.total_bytes, blob_bytes);
    if (!aligned16(blob)) return fail(P3P_ERR_INVALID_ARGUMENT, "blob must be 16-byte aligned");
    return launch_pfn_prepare(p, precision, static_cast<char*>(blob), bl, static_cast<cudaStream_t>(stream));
}

static int common_setup(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t B,
                        int64_t total_points, const p3p_grid* grid, void* workspace, size_t workspace_bytes,
                        GridDev* g, WsLayout* l, WsPtrs* ws) {
    if (B < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "num_tiles %d", B);
    if (B > 0 && !tile_offsets) return fail(P3P_ERR_INVALID_ARGUMENT, "tile_offsets is null");
    if (total_points > 0 && !points) return fail(P3P_ERR_INVALID_ARGUMENT, "points is null");
    if (point_stride < 3) return fail(P3P_ERR_INVALID_ARGUMENT, "point_stride %d (< 3)", point_stride);
    int rc = make_grid(grid, g);
    if (rc) return rc;
    rc = make_ws_layout(*g, B, total_points, l);
    if (rc) return rc;
    if (!workspace || !aligned16(workspace)) return fail(P3P_ERR_INVALID_ARGUMENT, "workspace null or misaligned");
    if (workspace_bytes < l->total_bytes) return fail(P3P_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", l->total_bytes, workspace_bytes);
    *ws = ws_ptrs(workspace, *l);
    return P3P_OK;
}

int p3p_voxelize(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
                 int64_t total_points, const p3p_grid* grid, const p3p_voxel_outputs* out, void* workspace,
                 size_t workspace_bytes, void* stream) {
    GridDev g;
    WsLayout l;
    WsPtrs ws;
    int rc = common_setup(points, point_stride, tile_offsets, num_tiles, total_points, grid, workspace, workspace_bytes, &g, &l, &ws);
    if (rc) return rc;
    if (num_tiles == 0) return P3P_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = launch_voxelize(points, point_stride, tile_offsets, num_tiles, total_points, g, l, ws, out ? out->point_hash : nullptr, 1, st);
    if (rc) return rc;
    if (out) return launch_export(g, num_tiles, ws, out, st);
    return P3P_OK;
}

static void fill_pfn_args(PfnArgs* a, const GridDev& g, const WsPtrs& ws, const void* blob, const BlobLayout& bl, int B) {
    memset(a, 0, sizeof(*a));
    a->g = g;
    a->ws = ws;
    a->blob = static_cast<const char*>(blob);
    a->bl = bl;
    a->B = B;
    a->row_stride = bl.C;
    a->row_offset = 0;
}

int p3p_pillar_features(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const void* blob, int32_t channels,
                        int32_t precision, float* features, void* workspace, size_t workspace_bytes, void* stream) {
    GridDev g;
    WsLayout l;
    BlobLayout bl;
    int rc = make_grid(grid, &g);
    if (rc) return rc;
    rc = make_ws_layout(g, num_tiles, total_points, &l);
    if (rc) return rc;
    rc = check_blob(channels, &bl);
    if (rc) return rc;
    if (!blob || !features || !workspace) return fail(P3P_ERR_INVALID_ARGUMENT, "null blob, features or workspace");
    if (!aligned16(blob) || !aligned16(features) || !aligned16(workspace)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    if (workspace_bytes < l.total_bytes) return fail(P3P_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", l.total_bytes, workspace_bytes);
    if (num_tiles == 0) return P3P_OK;
    PfnArgs a;
    fill_pfn_args(&a, g, ws_ptrs(workspace, l), blob, bl, num_tiles);
    a.item_mode = kItemsList;
    a.items_per_tile = g.Vmax;
    a.num_items = (int64_t)num_tiles * g.Vmax;
    a.out = features;
    a.out_layout = P3P_LAYOUT_NLC;
    a.out_dtype = P3P_DTYPE_F32;
    return run_pfn(a, precision, static_cast<cudaStream_t>(stream));
}

int p3p_encode(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
               int64_t total_points, const p3p_grid* grid, const void* blob, int32_t channels, int32_t precision, void* out,
               int32_t out_layout, int32_t out_dtype, int32_t c_total, int32_t c_offset, int32_t lidar_zero,
               void* workspace, size_t workspace_bytes, void* stream) {
    GridDev g;
    WsLayout l;
    WsPtrs ws;
    BlobLayout bl;
    int rc = common_setup(points, point_stride, tile_offsets, num_tiles, total_points, grid, workspace, workspace_bytes, &g, &l, &ws);
    if (rc) return rc;
    rc = check_blob(channels, &bl);
    if (rc) return rc;
    if (!out || !aligned16(out)) return fail(P3P_ERR_INVALID_ARGUMENT, "out null or misaligned");
    if (!lidar_zero && (!blob || !aligned16(blob))) return fail(P3P_ERR_INVALID_ARGUMENT, "blob null or misaligned");
    if (out_layout != P3P_LAYOUT_NCHW && out_layout != P3P_LAYOUT_NLC) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown layout %d", out_layout);
    if (out_dtype != P3P_DTYPE_F32 && out_dtype != P3P_DTYPE_BF16 && out_dtype != P3P_DTYPE_F16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown dtype %d", out_dtype);
    if ((out_layout == P3P_LAYOUT_NCHW || c_total > 0) && (c_offset < 0 || c_offset + channels > c_total))
        return fail(P3P_ERR_INVALID_ARGUMENT, "channels [%d, %d) outside c_total %d", c_offset, c_offset + channels, c_total);
    if (num_tiles == 0) return P3P_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PfnArgs a;
    fill_pfn_args(&a, g, ws, blob, bl, num_tiles);
    a.item_mode = kItemsCanvas;
    a.items_per_tile = g.ny * g.nx;
    a.num_items = (int64_t)num_tiles * a.items_per_tile;
    a.out = out;
    a.out_layout = out_layout;
    a.out_dtype = out_dtype;
    a.c_total = c_total;
    a.c_offset = c_offset;
    if (out_layout == P3P_LAYOUT_NLC && c_total > 0) {  // rows of a wider channels-last buffer (the fusion convolution's input)
        a.row_stride = c_total;
        a.row_offset = c_offset;
    }
    if (lidar_zero) return launch_zero_lidar(a, st);  // `x_lidar * 0.0` (early_fusion_vit.py:113-119)
    cudaEvent_t* ev = nullptr;
    if (g_prof.on && (size_t)(g_prof.used + 1) * 3 <= g_prof.ev.size()) ev = g_prof.ev.data() + (size_t)g_prof.used * 3;
    if (ev) cudaEventRecord(ev[0], st);
    rc = launch_voxelize(points, point_stride, tile_offsets, num_tiles, total_points, g, l, ws, nullptr, 0, st);
    if (rc) return rc;
    if (ev) cudaEventRecord(ev[1], st);
    rc = run_pfn(a, precision, st);
    if (ev) {
        cudaEventRecord(ev[2], st);
        ++g_prof.used;
    }
    return rc;
}

int p3p_encode_workspace(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const void* blob, int32_t channels,
                         int32_t precision, void* out, int32_t out_layout, int32_t out_dtype, int32_t c_total, int32_t c_offset,
                         void* workspace, size_t workspace_bytes, void* stream) {
    GridDev g;
    WsLayout l;
    BlobLayout bl;
    int rc = make_grid(grid, &g);
    if (rc) return rc;
    rc = make_ws_layout(g, num_tiles, total_points, &l);
    if (rc) return rc;
    rc = check_blob(channels, &bl);
    if (rc) return rc;
    if (!blob || !out || !workspace) return fail(P3P_ERR_INVALID_ARGUMENT, "null blob, out or workspace");
    if (!aligned16(blob) || !aligned16(out) || !aligned16(workspace)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    if (workspace_bytes < l.total_bytes) return fail(P3P_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", l.total_bytes, workspace_bytes);
    if (out_layout != P3P_LAYOUT_NCHW && out_layout != P3P_LAYOUT_NLC) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown layout %d", out_layout);
    if (out_dtype != P3P_DTYPE_F32 && out_dtype != P3P_DTYPE_BF16 && out_dtype != P3P_DTYPE_F16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown dtype %d", out_dtype);
    if ((out_layout == P3P_LAYOUT_NCHW || c_total > 0) && (c_offset < 0 || c_offset + channels > c_total))
        return fail(P3P_ERR_INVALID_ARGUMENT, "channels [%d, %d) outside c_total %d", c_offset, c_offset + channels, c_total);
    if (num_tiles == 0) return P3P_OK;
    PfnArgs a;
    fill_pfn_args(&a, g, ws_ptrs(workspace, l), blob, bl, num_tiles);
    a.item_mode = kItemsCanvas;
    a.items_per_tile = g.ny * g.nx;
    a.num_items = (int64_t)num_tiles * a.items_per_tile;
    a.out = out;
    a.out_layout = out_layout;
    a.out_dtype = out_dtype;
    a.c_total = c_total;
    a.c_offset = c_offset;
    if (out_layout == P3P_LAYOUT_NLC && c_total > 0) {
        a.row_stride = c_total;
        a.row_offset = c_offset;
    }
    return run_pfn(a, precision, static_cast<cudaStream_t>(stream));
}

int p3p_encode_tokens(const float* points, int32_t point_stride, const int64_t* tile_offsets, int32_t num_tiles,
                      int64_t total_points, const p3p_grid* grid, const void* blob, int32_t channels, int32_t precision,
                      const float* cls_token, const float* pos_embed, float* tokens, void* workspace, size_t workspace_bytes,
                      void* stream) {
    GridDev g;
    WsLayout l;
    WsPtrs ws;
    BlobLayout bl;
    int rc = common_setup(points, point_stride, tile_offsets, num_tiles, total_points, grid, workspace, workspace_bytes, &g, &l, &ws);
    if (rc) return rc;
    rc = check_blob(channels, &bl);
    if (rc) return rc;
    if (!tokens || !aligned16(tokens)) return fail(P3P_ERR_INVALID_ARGUMENT, "tokens null or misaligned");
    if (!blob || !aligned16(blob)) return fail(P3P_ERR_INVALID_ARGUMENT, "blob null or misaligned");
    if (!cls_token || !pos_embed) return fail(P3P_ERR_INVALID_ARGUMENT, "cls_token or pos_embed is null");
    if (num_tiles == 0) return P3P_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PfnArgs a;
    fill_pfn_args(&a, g, ws, blob, bl, num_tiles);
    a.item_mode = kItemsCanvas;
    a.items_per_tile = g.ny * g.nx;
    a.num_items = (int64_t)num_tiles * a.items_per_tile;
    a.out = tokens;
    a.out_layout = P3P_LAYOUT_NLC;
    a.out_dtype = P3P_DTYPE_F32;
    a.c_total = 0;
    a.c_offset = 0;
    a.pos_embed = pos_embed;
    a.token_rows = a.items_per_tile + 1;
    rc = launch_cls_rows(a, cls_token, st);
    if (rc) return rc;
    rc = launch_voxelize(points, point_stride, tile_offsets, num_tiles, total_points, g, l, ws, nullptr, 0, st);
    if (rc) return rc;
    return run_pfn(a, precision, st);
}

int p3p_las_to_pixels(const int32_t* X, const int32_t* Y, const int32_t* Z, const int64_t* tile_offsets, int32_t num_tiles,
                      int64_t total_points, const p3p_las_tile* tiles, double z_hi, int32_t* minmax_ws, float* points,
                      void* stream) {
    if (num_tiles < 0 || total_points < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "negative batch or point count");
    if (num_tiles == 0 || total_points == 0) return P3P_OK;
    if (!X || !Y || !Z || !tile_offsets || !tiles || !minmax_ws || !points) return fail(P3P_ERR_INVALID_ARGUMENT, "null pointer");
    if (!(z_hi > 0.0)) return fail(P3P_ERR_INVALID_ARGUMENT, "z_hi %g", z_hi);
    return launch_las_to_pixels(X, Y, Z, nullptr, nullptr, tile_offsets, num_tiles, total_points, tiles, z_hi, minmax_ws, points,
                                static_cast<cudaStream_t>(stream));
}

int p3p_las_packed_to_pixels(const uint16_t* deltas, const int32_t* tile_base, const int64_t* tile_offsets, int32_t num_tiles,
                             int64_t total_points, const p3p_las_tile* tiles, double z_hi, int32_t* minmax_ws, float* points,
                             void* stream) {
    if (num_tiles < 0 || total_points < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "negative batch or point count");
    if (num_tiles == 0 || total_points == 0) return P3P_OK;
    if (!deltas || !tile_base || !tile_offsets || !tiles || !minmax_ws || !points) return fail(P3P_ERR_INVALID_ARGUMENT, "null pointer");
    if (!(z_hi > 0.0)) return fail(P3P_ERR_INVALID_ARGUMENT, "z_hi %g", z_hi);
    return launch_las_to_pixels(nullptr, nullptr, nullptr, deltas, tile_base, tile_offsets, num_tiles, total_points, tiles, z_hi,
                                minmax_ws, points, static_cast<cudaStream_t>(stream));
}

size_t p3p_conv3x3_blob_bytes(int32_t in_channels, int32_t out_channels) {
    if (in_channels < 1 || out_channels < 1) return 0;
    return conv3x3_blob_bytes(in_channels, out_channels);
}

int p3p_conv3x3_prepare(const p3p_conv_params* p, int32_t precision, void* blob, size_t blob_bytes, void* stream) {
    if (!p || !blob || !p->weight) return fail(P3P_ERR_INVALID_ARGUMENT, "null params, weight or blob");
    if (p->norm_weight && (!p->norm_bias || !p->norm_mean || !p->norm_var)) return fail(P3P_ERR_INVALID_ARGUMENT, "incomplete BatchNorm parameters");
    if (p->in_channels < 1 || p->out_channels < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "channels must be positive");
    if (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16) return fail(P3P_ERR_UNSUPPORTED, "conv3x3 precision must be bf16 or fp16");
    if (!aligned16(blob)) return fail(P3P_ERR_INVALID_ARGUMENT, "blob must be 16-byte aligned");
    const size_t need = conv3x3_blob_bytes(p->in_channels, p->out_channels);
    if (blob_bytes < need) return fail(P3P_ERR_WORKSPACE, "blob needs %zu bytes, got %zu", need, blob_bytes);
    return launch_conv3x3_prepare(p, precision, blob, static_cast<cudaStream_t>(stream));
}

int p3p_conv3x3(const void* x, int32_t num_tiles, int32_t height, int32_t width, int32_t in_channels, const void* blob,
                int32_t out_channels, int32_t precision, int32_t relu, float* out, int32_t out_layout, int32_t c_total,
                int32_t c_offset, void* stream) {
    if (num_tiles < 0 || height < 1 || width < 1 || in_channels < 1 || out_channels < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "bad sizes");
    if (num_tiles == 0) return P3P_OK;
    if (!x || !blob || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null x, blob or out");
    if (!aligned16(x) || !aligned16(blob) || !aligned16(out)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    if (out_layout != P3P_LAYOUT_NCHW && out_layout != P3P_LAYOUT_NLC) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown layout %d", out_layout);
    if (c_offset < 0 || c_offset + out_channels > c_total) return fail(P3P_ERR_INVALID_ARGUMENT, "channels [%d, %d) outside c_total %d", c_offset, c_offset + out_channels, c_total);
    return launch_conv3x3(x, num_tiles, height, width, in_channels, blob, out_channels, precision, relu, out, out_layout, c_total, c_offset,
                          static_cast<cudaStream_t>(stream));
}

int p3p_conv3x3_vit_tokens(const void* x, int32_t num_tiles, int32_t height, int32_t width, int32_t in_channels, const void* blob,
                           int32_t out_channels, int32_t precision, const float* cls_token, const float* pos_embed, float* out,
                           void* stream) {
    if (num_tiles < 0 || height < 1 || width < 1 || in_channels < 1 || out_channels < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "bad sizes");
    if (!cls_token || !pos_embed) return fail(P3P_ERR_INVALID_ARGUMENT, "cls_token or pos_embed is null");
    if (num_tiles == 0) return P3P_OK;
    if (!x || !blob || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null x, blob or out");
    if (!aligned16(x) || !aligned16(blob) || !aligned16(out)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    return launch_conv3x3_vit_tokens(x, num_tiles, height, width, in_channels, blob, out_channels, precision, cls_token, pos_embed, out,
                                     static_cast<cudaStream_t>(stream));
}

int p3p_nchw_to_nhwc16(const float* x, int32_t num_tiles, int32_t channels, int32_t height, int32_t width, int32_t precision,
                       void* out, int32_t c_total, int32_t c_offset, void* stream) {
    if (num_tiles < 0 || channels < 1 || height < 1 || width < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "bad sizes");
    if (num_tiles == 0) return P3P_OK;
    if (!x || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null x or out");
    if (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16) return fail(P3P_ERR_UNSUPPORTED, "precision must be bf16 or fp16");
    if (c_offset < 0 || c_offset + channels > c_total) return fail(P3P_ERR_INVALID_ARGUMENT, "channels outside c_total");
    return launch_nchw_to_nhwc16(x, num_tiles, channels, height, width, precision, out, c_total, c_offset, static_cast<cudaStream_t>(stream));
}

int p3p_upsample_bilinear_nhwc16(const float* x, int32_t num_tiles, int32_t h, int32_t w, int32_t channels, int64_t src_batch_stride,
                                 int32_t out_h, int32_t out_w, int32_t precision, void* out, void* stream) {
    if (num_tiles < 0 || h < 1 || w < 1 || channels < 1 || out_h < 1 || out_w < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "bad sizes");
    if (num_tiles == 0) return P3P_OK;
    if (!x || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null x or out");
    if (precision != P3P_PRECISION_BF16 && precision != P3P_PRECISION_FP16) return fail(P3P_ERR_UNSUPPORTED, "precision must be bf16 or fp16");
    return launch_upsample_bilinear_nhwc16(x, num_tiles, h, w, channels, src_batch_stride, out_h, out_w, precision, out,
                                           static_cast<cudaStream_t>(stream));
}

int p3p_profile_begin(int32_t max_records) {
    if (max_records < 1 || max_records > 100000) return fail(P3P_ERR_INVALID_ARGUMENT, "max_records %d", max_records);
    for (cudaEvent_t e : g_prof.ev) cudaEventDestroy(e);
    g_prof.ev.assign((size_t)max_records * 3, nullptr);
    for (auto& e : g_prof.ev) P3P_CUDA_CHECK(cudaEventCreate(&e));
    g_prof.used = 0;
    g_prof.on = true;
    return P3P_OK;
}

int p3p_profile_end(float* ms_voxelize, float* ms_pfn, int32_t capacity, int32_t* num_records) {
    if (!g_prof.on) return fail(P3P_ERR_INVALID_ARGUMENT, "p3p_profile_end without p3p_profile_begin");
    g_prof.on = false;
    int n = g_prof.used < capacity ? g_prof.used : capacity;
    float* dst[2] = {ms_voxelize, ms_pfn};
    for (int i = 0; i < n; ++i) {
        cudaEvent_t* e = g_prof.ev.data() + (size_t)i * 3;
        P3P_CUDA_CHECK(cudaEventSynchronize(e[2]));
        for (int s = 0; s < 2; ++s) {
            float ms = 0.f;
            P3P_CUDA_CHECK(cudaEventElapsedTime(&ms, e[s], e[s + 1]));
            if (dst[s]) dst[s][i] = ms;
        }
    }
    if (num_records) *num_records = n;
    for (cudaEvent_t e : g_prof.ev) cudaEventDestroy(e);
    g_prof.ev.clear();
    g_prof.used = 0;
    return P3P_OK;
}

int p3p_patch_embed(const float* images, int32_t num_tiles, int32_t in_chans, int32_t height, int32_t width,
                    int32_t patch, const float* weight, const float* bias, int32_t channels, int32_t precision, void* out,
                    int32_t out_dtype, int32_t out_layout, int32_t c_total, int32_t c_offset, void* stream) {
    if (num_tiles < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "num_tiles %d", num_tiles);
    if (in_chans < 1 || height < 1 || width < 1 || patch < 1 || channels < 1)
        return fail(P3P_ERR_INVALID_ARGUMENT, "in_chans, height, width, patch and channels must be positive");
    if (height % patch != 0 || width % patch != 0)
        return fail(P3P_ERR_INVALID_ARGUMENT, "image %d x %d is not a whole number of %d-px patches", height, width, patch);
    if (precision < P3P_PRECISION_FP32 || precision > P3P_PRECISION_FP16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
    if (out_dtype != P3P_DTYPE_F32 && out_dtype != P3P_DTYPE_BF16 && out_dtype != P3P_DTYPE_F16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown dtype %d", out_dtype);
    if (out_layout != P3P_LAYOUT_NCHW && out_layout != P3P_LAYOUT_NLC) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown layout %d", out_layout);
    if (c_offset < 0 || c_offset + channels > c_total)
        return fail(P3P_ERR_INVALID_ARGUMENT, "channels [%d, %d) outside c_total %d", c_offset, c_offset + channels, c_total);
    if (num_tiles == 0) return P3P_OK;
    if (!images || !weight || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null images, weight or out");
    if (!aligned16(images) || !aligned16(weight) || !aligned16(out)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    return launch_patch_embed(images, num_tiles, in_chans, height, width, patch, weight, bias, nullptr, channels, precision, out,
                              out_dtype, out_layout, c_total, c_offset, static_cast<cudaStream_t>(stream));
}

size_t p3p_patch_embed_blob_bytes(int32_t channels, int32_t in_chans, int32_t patch) {
    if (channels < 1 || in_chans < 1 || patch < 1) return 0;
    return patch_embed_blob_bytes(channels, in_chans, patch);
}

int p3p_patch_embed_prepare(const float* weight, const float* bias, int32_t channels, int32_t in_chans, int32_t patch,
                            int32_t precision, void* blob, size_t blob_bytes, void* stream) {
    if (channels < 1 || in_chans < 1 || patch < 1) return fail(P3P_ERR_INVALID_ARGUMENT, "channels, in_chans and patch must be positive");
    if (precision < P3P_PRECISION_FP32 || precision > P3P_PRECISION_FP16) return fail(P3P_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
    if (!weight || !blob) return fail(P3P_ERR_INVALID_ARGUMENT, "null weight or blob");
    if (!aligned16(weight) || !aligned16(blob)) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    if (blob_bytes < patch_embed_blob_bytes(channels, in_chans, patch)) return fail(P3P_ERR_WORKSPACE, "blob of %zu bytes is too small", blob_bytes);
    return launch_patch_embed_prepare(weight, bias, channels, in_chans, patch, precision, blob, static_cast<cudaStream_t>(stream));
}

int p3p_patch_embed_prepared(const float* images, int32_t num_tiles, int32_t in_chans, int32_t height, int32_t width,
                             int32_t patch, const void* blob, const float* weight, const float* bias, int32_t channels,
                             int32_t precision, void* out, int32_t out_dtype, int32_t out_layout, int32_t c_total, int32_t c_offset,
                             void* stream) {
    if (!blob || !aligned16(blob)) return fail(P3P_ERR_INVALID_ARGUMENT, "null or misaligned blob");
    const int rc = p3p_patch_embed(images, 0, in_chans, height, width, patch, weight, bias, channels, precision, out, out_dtype,
                                   out_layout, c_total, c_offset, stream);  // (argument checks; no tiles: no launch)
    if (rc) return rc;
    if (num_tiles < 0) return fail(P3P_ERR_INVALID_ARGUMENT, "num_tiles %d", num_tiles);
    if (num_tiles == 0) return P3P_OK;
    if (!images || !out) return fail(P3P_ERR_INVALID_ARGUMENT, "null images or out");
    if (!aligned16(images) || !aligned16(out) || (weight && !aligned16(weight))) return fail(P3P_ERR_INVALID_ARGUMENT, "misaligned pointer");
    // only the tensor-core route reads the blob; shapes it does not cover fall through to the exact kernel and the raw weights
    return launch_patch_embed(images, num_tiles, in_chans, height, width, patch, weight, bias,
                              (patch == 8 && precision != P3P_PRECISION_FP32) ? blob : nullptr, channels, precision, out, out_dtype,
                              out_layout, c_total, c_offset, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
