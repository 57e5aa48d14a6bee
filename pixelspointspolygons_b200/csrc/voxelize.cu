// voxelize.cu -- point -> pillar assignment for a whole jagged batch in ONE kernel (sm_100a).
//
// Replaces the per-sample Python loop of Open3D-ML PointPillars.voxelize that the reference calls at
// R:pixelspointspolygons/models/pointpillars/pointpillars_o3d.py:92 (SURVEY 8a rows a4/a5, Appendix A.1/A.2).
//
// The reference sorts (hash, index) pairs per tile and keeps the first M indices of each run.  What the rest of the
// path consumes is, per key, the SET of its min(count, M) lowest-index points (the PFN is a max and an exact
// fixed-point mean over that set), so nothing is sorted here:
//
//   * a CTA takes a ticket (atomic counter) -> chunk of <= 4096 consecutive points of one tile.  Tickets, not
//     blockIdx, order the chunks, so a CTA only ever waits for CTAs that are already running.  Chunks start at
//     multiples of 4 points of the packed xyz array: a lane moves 4 points with three aligned 16-byte loads.
//   * every lane hashes its <= 16 points with the reference's fp32 operation order and counts them in ONE
//     shared-memory histogram of the chunk, one atomic per point; only the packed (key, value returned by the atomic)
//     word of a point stays in a register.
//   * the chunk's per-key counts are published to global memory and a flag is released; the CTA acquires the flags
//     of the earlier chunks of its tile and sums their counts per key (pre).  Keys with pre >= M keep nothing of the
//     chunk; keys with pre + own <= M keep everything, in slots pre + (atomic value) -- any bijection will do; the few
//     keys that cross M inside the chunk (at most one chunk per key and tile) keep their M - pre lowest-index points,
//     found exactly by a two-digit radix selection over the chunk-local index.  The kept set is therefore exactly the
//     reference's whatever order the hardware serves the atomics in; the order inside a pillar is not the reference's
//     (export_kernel sorts by index for the parity surface).
//   * a chunk that sees every regular cell full publishes that; later chunks of the tile (multi-wave launches: dense
//     tiles) then only handle the keys beyond the regular cells.
//   * the last CTA of a tile to finish runs the tile's plan: keys in ascending order -> run ordinal (max_voxels
//     cut), cell coordinates (decoded from the key; from the lowest-index point when the run holds a point on the
//     x / y max face, i.e. under hash aliasing), x/y bound filter, final voxel order, and the canvas owner table
//     (last pillar in voxel order wins a cell, Appendix A.5).
//
// export_kernel (optional) dumps the reference-shaped tensors for the parity tests.
#include <type_traits>

#include "p3p_internal.cuh"

namespace p3p {

// Optional phase timeline (build with -DP3P_TIMELINE): thread 0 of every CTA stamps %globaltimer at the phase
// boundaries; tools/timeline.py reads them back through p3p_debug_timeline.
#ifdef P3P_TIMELINE
__device__ unsigned long long g_timeline[8192][16];
__device__ __forceinline__ void tl_stamp(int cta, int slot) {
    if (threadIdx.x == 0 && cta < 8192) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_timeline[cta][slot] = t;
    }
}
#define TL(cta, slot) tl_stamp(cta, slot)
extern "C" int p3p_debug_timeline(unsigned long long* host, int ctas) {
    return (int)cudaMemcpyFromSymbol(host, g_timeline, sizeof(unsigned long long) * 16 * (size_t)ctas);
}
#else
#define TL(cta, slot)
#endif

namespace {

constexpr int kThreads = kVoxThreads;  // (build-time tunable, p3p_internal.cuh)
constexpr int kWarps = kThreads / 32;
constexpr int kIters = kMaxChunkPoints / kThreads;  // points per lane held in registers

struct ChunkLoc {
    int b;        // tile, -1 if this ticket has no chunk
    int c;        // chunk index inside the tile
    int nchunks;  // chunks of the tile
    int gstart;   // global index of the tile's chunk 0
    long long p0;      // first point of the chunk's nominal range: 16-byte aligned in the packed array (may lie up to 3 points before the tile)
    long long lo, hi;  // the tile's own points: [lo, hi)
    unsigned sat;      // the tile's saturation word as read once for the whole CTA
};

// predicated atomic increment of a 16-bit shared-memory counter (through its 32-bit word; counters never overflow into
// their neighbour); returns the counter's previous value
__device__ __forceinline__ unsigned atoms_add_u16(uint32_t addr, int pred) {
    unsigned r;
    const unsigned sh = (addr & 2u) * 8u;
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %3, 0;\n mov.b32 %0, 0;\n @p atom.shared.add.u32 %0, [%1], %2;\n}"
        : "=r"(r)
        : "r"(addr & ~3u), "r"(1u << sh), "r"(pred)
        : "memory");
    return (r >> sh) & 0xFFFFu;
}

__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Executed by warp 0: map ticket -> (tile, local chunk).  The chunks of a tile start at its first point rounded down to
// an index = phase (mod 4), the indices at which the packed xyz array is 16-byte aligned (address = base + 12 * index;
// phase = (base / 4) mod 4).  Storage (flags, chunk rows) is tile-major: chunk c of tile b lives at gstart(b) + c.
// Tickets are handed out CHUNK-major for batches of up to 32 tiles -- chunk 0 of every tile, then chunk 1 of every tile,
// ... -- so that in a multi-wave launch (dense tiles) the early chunks of all tiles run first and the later waves see
// the tiles' saturation hints; a chunk still only waits for chunks with smaller tickets (its own tile's earlier ones).
__device__ void locate_chunk(int g, const int64_t* __restrict__ offsets, int B, int S, int phase, ChunkLoc* out) {
    const int lane = threadIdx.x & 31;
    if (B <= 32) {
        long long o0 = 0, o1 = 0;
        if (lane < B) { o0 = offsets[lane]; o1 = offsets[lane + 1]; }
        const long long a0 = o0 - ((o0 - phase) & 3ll);  // largest index <= o0 that is = phase (mod 4)
        const long long n = o1 > o0 ? o1 - a0 : 0;
        const int nc = (int)((n + S - 1) / S);
        int incl = nc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        if (g >= total) {
            if (lane == 0) out->b = -1;
            return;
        }
        // f(c) = sum_b min(nc_b, c) = tickets of chunk index < c; the ticket's chunk index is the largest c with f(c) <= g
        int lo = 0, hi = __reduce_max_sync(0xffffffffu, nc) - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__reduce_add_sync(0xffffffffu, nc < mid ? nc : mid) <= g) lo = mid; else hi = mid - 1;
        }
        const int c = lo;
        const int r = g - __reduce_add_sync(0xffffffffu, nc < c ? nc : c);  // rank among the tiles that have a chunk c
        const bool has = nc > c;
        const unsigned bal = __ballot_sync(0xffffffffu, has);
        if (has && __popc(bal & ((1u << lane) - 1u)) == r) {
            out->b = lane;
            out->c = c;
            out->nchunks = nc;
            out->gstart = incl - nc;
            out->p0 = a0 + (long long)c * S;
            out->lo = o0;
            out->hi = o1;
        }
        return;
    }
    // more than 32 tiles: tile-major tickets, tiles walked 32 at a time
    int base = 0;
    bool found = false;
    for (int t0 = 0; t0 < B && !found; t0 += 32) {
        const int t = t0 + lane;
        long long o0 = 0, o1 = 0;
        if (t < B) { o0 = offsets[t]; o1 = offsets[t + 1]; }
        const long long a0 = o0 - ((o0 - phase) & 3ll);
        const long long n = o1 > o0 ? o1 - a0 : 0;
        const int nc = (int)((n + S - 1) / S);
        int incl = nc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int excl = base + incl - nc;
        const bool mine = (t < B) && (g >= excl) && (g < excl + nc);
        const unsigned bal = __ballot_sync(0xffffffffu, mine);
        if (bal) {
            found = true;
            if (mine) {
                out->b = t;
                out->c = g - excl;
                out->nchunks = nc;
                out->gstart = excl;
                out->p0 = a0 + (long long)(g - excl) * S;
                out->lo = o0;
                out->hi = o1;
            }
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (!found && lane == 0) out->b = -1;
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_tot, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();  // protect warp_tot reuse
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < kWarps; ++i) {
        const int t = warp_tot[i];
        if (i < w) off += t;
        tot += t;
    }
    *total = tot;
    return off + incl - v;
}

__device__ void write_empty_tile(const GridDev& g, const WsPtrs& ws, int b) {
    const int HW = g.ny * g.nx;
    for (int i = threadIdx.x; i < HW; i += kThreads) {
        ws.owner[(size_t)b * HW + i] = -1;
        ws.cell_desc[(size_t)b * HW + i] = -1;
    }
    if (threadIdx.x == 0) ws.num_pil[b] = 0;
}

// Per-tile plan, run by the CTA that finished the tile's last chunk.  Keff: keys that can be non-empty (the regular
// cells only, unless some point of the tile hashed beyond them).  scratch: >= (4 K + HW) ints of shared memory.
__device__ void plan_tile(const GridDev& g, const WsPtrs& ws, int b, int Keff, int* scratch, int* warp_tot) {
    const int K = g.num_keys, HW = g.ny * g.nx, M = g.M, tid = threadIdx.x;
    int* n_s = scratch;         // [K] min(count, M), 0 = empty
    int* cell_s = n_s + K;      // [K] packed cell of the run, -1 if dropped
    int* rkey_s = cell_s + K;   // [K] key of pillar r
    int* rn_s = rkey_s + K;     // [K] n of pillar r
    int* owner_s = rn_s + K;    // [HW]
    const int* totals = ws.totals + (size_t)b * K;
    const float4* slots = ws.slots + (size_t)b * K * M;
    const uint8_t* edge = ws.edge + (size_t)b * K;
    // counts of every key (written by other CTAs -> L2 loads, 8 independent loads per thread and batch); coordinates
    // come from the key itself unless the run holds an edge point, in which case its lowest-index kept point decides
    // (Appendix A.1: hash aliasing)
    for (int k0 = 0; k0 < Keff; k0 += kThreads * 8) {
        int t[8];
        uint8_t e[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int k = k0 + u * kThreads + tid;
            t[u] = 0; e[u] = 0;
            if (k < Keff) { t[u] = __ldcg(totals + k); e[u] = __ldcg(edge + k); }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int k = k0 + u * kThreads + tid;
            if (k >= Keff) continue;
            int cell = -1;
            const int n = t[u] < M ? t[u] : M;
            if (n > 0) {
                int cx, cy, cz;
                if (e[u]) {
                    float4 best = __ldcg(slots + (size_t)k * M);
                    for (int i = 1; i < n; ++i) {
                        const float4 p = __ldcg(slots + (size_t)k * M + i);
                        if (__float_as_int(p.w) < __float_as_int(best.w)) best = p;
                    }
                    point_cell(g, best.x, best.y, best.z, cx, cy, cz);
                } else {
                    cz = k / g.stride2;
                    const int rem = k - cz * g.stride2;
                    cy = rem / g.stride1;
                    cx = rem - cy * g.stride1;
                }
                if (cy < g.nv[1] && cx < g.nv[0]) cell = cx | (cy << 10) | (cz << 20);  // x/y bound filter (A.2)
            }
            n_s[k] = n;
            cell_s[k] = cell;
        }
    }
    for (int i = tid; i < HW; i += kThreads) owner_s[i] = -1;
    __syncthreads();
    const int per = (Keff + kThreads - 1) / kThreads;
    const int k0 = tid * per, k1 = (k0 + per < Keff) ? k0 + per : Keff;
    int cnt = 0;
    for (int k = k0; k < k1; ++k) cnt += (n_s[k] > 0);
    int total_runs;
    int ord = block_exclusive_scan(cnt, warp_tot, &total_runs);
    int cnt2 = 0;
    for (int k = k0; k < k1; ++k) {
        if (n_s[k] > 0) {
            const int r = ord++;
            if (r >= g.Vmax) cell_s[k] = -1;  // only the first max_voxels runs in hash order survive (A.1)
        }
        cnt2 += (cell_s[k] >= 0);
    }
    int total_pil;
    int ord2 = block_exclusive_scan(cnt2, warp_tot, &total_pil);
    for (int k = k0; k < k1; ++k) {
        const int st = cell_s[k];
        if (st < 0) continue;
        const int r = ord2++;
        const size_t pi = (size_t)b * g.Vmax + r;
        const int n = n_s[k];
        ws.pil_key[pi] = k;
        ws.pil_n[pi] = n;
        ws.pil_coord[pi] = st;
        rkey_s[r] = k;
        rn_s[r] = n;
        const int cx = st & 1023, cy = (st >> 10) & 1023;
        atomicMax(&owner_s[cy * g.nx + cx], r);  // scatter collisions: the later row (higher hash) wins (A.5)
    }
    if (tid == 0) ws.num_pil[b] = total_pil;
    __syncthreads();
    for (int i = tid; i < HW; i += kThreads) {
        const int o = owner_s[i];
        ws.owner[(size_t)b * HW + i] = o;
        ws.cell_desc[(size_t)b * HW + i] = (o >= 0) ? (rkey_s[o] | (rn_s[o] << 16)) : -1;
    }
}

// packed per-point word: key (13 bits) | arbitrary-order rank of the point among the chunk's points of its key (13 bits:
// a chunk holds <= 4096 points) << 13; -1: no key (out of range, outside the tile, or irrelevant in a saturated tile)
constexpr int kKeyBits = 13;
constexpr unsigned kKeyMask = (1u << kKeyBits) - 1u;
static_assert(kMaxKeys <= (1 << kKeyBits), "key field too narrow");
static_assert(kMaxChunkPoints * 8 < 65536, "8 chunk rows must add up inside 16-bit lanes");
constexpr int kGroups = kIters / 4;        // groups of 4 consecutive points (48 bytes = 3 x 16-byte loads) per thread
constexpr int kCrossBatch = 256;           // crossing keys resolved per round (512 measured: no change)
constexpr int kCells = kGroups * kWarps;   // the chunk-local order is (group, warp, lane, e): 32 cells (group, warp) of 128 consecutive points
static_assert(kMaxChunkPoints / kCells <= 255, "points of a cell must fit the 8-bit fields of the boundary word");
constexpr unsigned kCrossFlag = 0x8000u;   // base_s entry: the key crosses M inside this chunk; low 15 bits = crossing id

// kFast: packed xyz (stride 3), no per-point hash export, hashes beyond the cells kept (the shipped configuration): the
// per-point branches on those options are resolved at compile time and the points travel as 16-byte loads.
//
// Ranking.  The rest of the path consumes, per key, the SET of its min(count, M) lowest-index points.  A chunk counts its
// points per key with one shared-memory atomic per point; the value the atomic returns orders the chunk's points of a key
// arbitrarily.  With pre = points of the key in the earlier chunks of the tile and own = points in this chunk:
//   pre >= M            nothing of the chunk is kept;
//   pre + own <= M      everything is kept, and any bijection onto slots [pre, pre + own) will do: slot = pre + atomic value;
//   otherwise           (at most one chunk per key and tile) the M - pre lowest-index points of the chunk are kept: a
//                       two-digit radix selection over the chunk-local index (2 x 64 bins per crossing key) finds the
//                       index threshold exactly; survivors take the slots [pre, M) in arbitrary order.
// No step of this depends on the order in which the hardware serves same-address atomics.
template <bool kFast>
__global__ void __launch_bounds__(kThreads, kVoxCtasPerSm)
voxelize_kernel(const float* __restrict__ pts, int stride_arg, const int64_t* __restrict__ offsets, int B, GridDev g, int S, WsPtrs ws, int32_t* __restrict__ point_hash, int need_plan, int pdl_from) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int K = g.num_keys;
    const int Kp = ws.key_stride;  // K rounded up to 8: row stride of chunk_hist (16-byte rows)
    uint16_t* ctot_s = reinterpret_cast<uint16_t*>(smem_raw);   // [Kp] points of the key in this chunk; last chunk: min(count, M) of the tile
    uint16_t* base_s = ctot_s + Kp;                             // [Kp] min(pre, M), or kCrossFlag | crossing id
    uint16_t* need_s = base_s + Kp;                             // [Kp] by crossing id: M - pre
    unsigned* bnd_s = reinterpret_cast<unsigned*>(need_s + Kp); // [kCrossBatch] boundary cell | survivors in it << 8 | its count << 16
    uint16_t* cell_s = reinterpret_cast<uint16_t*>(bnd_s + kCrossBatch);  // [kCells][kCrossBatch] per-cell counts, then their exclusive prefix
    __shared__ ChunkLoc loc;
    __shared__ int s_ticket, s_last, s_runs[2], s_ncross;
    __shared__ int warp_tot[kWarps];

    const int tid = threadIdx.x, lane = tid & 31;
    const int stride = kFast ? 3 : stride_arg;
    TL(blockIdx.x, 0);
    if (tid == 0) { s_ticket = (int)atomicAdd(ws.sync, 1u); s_ncross = 0; }
    {
        uint4* h4 = reinterpret_cast<uint4*>(ctot_s);
        for (int i = tid; i < Kp / 8; i += kThreads) h4[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    const int ticket = s_ticket;
    // Let the dependent PFN grid start its prologue on the SMs this grid has left (it waits for this grid's completion
    // with griddepcontrol.wait before it reads anything written here).  Only the last tickets trigger early: the
    // dependent grid launches once every CTA has triggered or exited, i.e. when no CTA of this grid is still waiting
    // for an SM that a waiting PFN CTA could occupy.
    if (ticket >= pdl_from) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    unsigned* flags = ws.sync + 1;
    unsigned* tile_done = flags + ws.max_chunks;
    unsigned* tile_sat = tile_done + B;
    if (tid < 32) {
        locate_chunk(ticket, offsets, B, S, kFast ? (int)((reinterpret_cast<uintptr_t>(pts) >> 2) & 3u) : 0, &loc);
        __syncwarp();
        if (lane == 0 && loc.b >= 0) loc.sat = __ldcg(tile_sat + loc.b);  // one read: the whole CTA acts on the same value
    }
    // tiles without points have no chunk: ticket t < B writes the empty plan of tile t
    if (ticket < B && offsets[ticket + 1] <= offsets[ticket]) write_empty_tile(g, ws, ticket);
    __syncthreads();
    if (loc.b < 0) return;
    TL(blockIdx.x, 1);

    uint8_t* edge = ws.edge + (size_t)loc.b * K;
    const int M = g.M;
    // A chunk c0 that finds every regular cell full (pre + own >= M) publishes 0x7fffffff - c0; chunks behind it (only
    // those: their points have higher indices than M kept ones in every regular cell) then count the keys beyond the
    // regular cells only.  A hint: chunks that do not see it yet just do the full work.
    const unsigned sat_word = loc.sat;
    const bool saturated = sat_word != 0u && (int)(0x7fffffffu - sat_word) < loc.c;

    // ---- hash + count: chunk-local index ci = 4 * (256 * group + tid) + e; the chunk starts at a multiple of 4 points
    //      (loc.p0; the tile's own range is [lo, hi)), so a group of 4 points is three aligned 16-byte loads --------------
    int pk[kIters];
    // bit 0: some key may lie outside the regular cells or be aliased (a point on a max face: z == z_max, y == y_max, ...)
    // bit 1: some point sits on the x / y max face (its run's coordinates are not decodable from the key)
    int hi_key = 0;
    const long long lo = loc.lo, hi = loc.hi;
    const uint32_t ctot_sa = smem_u32(ctot_s);
    // a chunk that lies inside its tile (all but the first / last of a tile) issues its twelve 16-byte loads at once
    const bool interior = kFast && S == kMaxChunkPoints && loc.p0 >= lo && loc.p0 + S <= hi;  // (uniform)
    auto load_group = [&](int gi, float (&x)[4], float (&y)[4], float (&z)[4]) {
        const long long p = loc.p0 + 4ll * (kThreads * gi + tid);
        if (kFast && p >= lo && p + 4 <= hi) {
            const float4* q = reinterpret_cast<const float4*>(pts + p * 3);
            const float4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
            x[0] = a.x; y[0] = a.y; z[0] = a.z; x[1] = a.w; y[1] = b.x; z[1] = b.y;
            x[2] = b.z; y[2] = b.w; z[2] = c.x; x[3] = c.y; y[3] = c.z; z[3] = c.w;
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                x[e] = y[e] = z[e] = __int_as_float(0x7fc00000);  // NaN: no key
                if (p + e >= lo && p + e < hi) {
                    const float* q = pts + (p + e) * stride;
                    x[e] = __ldg(q); y[e] = __ldg(q + 1); z[e] = __ldg(q + 2);
                }
            }
        }
    };
    {
        unsigned edge_bits = 0;  // points on the x / y max face (rare: flags set on a slow path)
        int kmax = -1;
        auto hash_group = [&](int gi, const float (&x)[4], const float (&y)[4], const float (&z)[4]) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                bool on_edge;
                int k = point_key<!kFast>(g, x[e], y[e], z[e], on_edge);  // (kFast: the launcher checked the overflow flag)
                if (!kFast && point_hash) {
                    const long long p = loc.p0 + 4ll * (kThreads * gi + tid) + e;
                    if (p >= lo && p < hi) point_hash[p] = k;
                }
                edge_bits |= on_edge ? (1u << (4 * gi + e)) : 0u;
                kmax = k > kmax ? k : kmax;
                if (saturated && k < g.num_cells) k = -1;
                pk[4 * gi + e] = k;
            }
        };
        if (interior) {
            const float4* q = reinterpret_cast<const float4*>(pts + (loc.p0 + 4ll * tid) * 3);
            float4 v[kGroups][3];
#pragma unroll
            for (int gi = 0; gi < kGroups; ++gi) {
#pragma unroll
                for (int u = 0; u < 3; ++u) v[gi][u] = __ldg(q + (size_t)gi * (kThreads * 3) + u);
            }
#pragma unroll
            for (int gi = 0; gi < kGroups; ++gi) {
                const float4 a = v[gi][0], b = v[gi][1], c = v[gi][2];
                const float x[4] = {a.x, a.w, b.z, c.y}, y[4] = {a.y, b.x, b.w, c.z}, z[4] = {a.z, b.y, c.x, c.w};
                hash_group(gi, x, y, z);
            }
        } else {
#pragma unroll
            for (int gi = 0; gi < kGroups; ++gi) {
                if (4 * kThreads * gi < S) {  // (uniform)
                    float x[4], y[4], z[4];
                    load_group(gi, x, y, z);
                    hash_group(gi, x, y, z);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) pk[4 * gi + e] = -1;
                }
            }
        }
        hi_key |= ((kmax >= g.num_cells) ? 1 : 0) | (edge_bits ? 3 : 0);
        if (edge_bits) {
#pragma unroll
            for (int j = 0; j < kIters; ++j)
                if (((edge_bits >> j) & 1u) && pk[j] >= 0) edge[pk[j]] = 1;  // idempotent flag, read by the tile's plan
        }
        TL(blockIdx.x, 2);
#pragma unroll
        for (int j = 0; j < kIters; ++j) {
            const int k = pk[j];
            const int act = k >= 0 ? 1 : 0;
            const unsigned old = atoms_add_u16(ctot_sa + 2u * (unsigned)(act ? k : 0), act);
            if (act) pk[j] = k | (int)(old << kKeyBits);
        }
    }
    hi_key = (__syncthreads_or(hi_key & 1) ? 1 : 0) | (__syncthreads_or(hi_key & 2) ? 2 : 0);  // (the intrinsic ORs predicates)
    TL(blockIdx.x, 3);
    if (tid < 2) s_runs[tid] = 0;
    // ---- publish this chunk's per-key counts (full rows: zeros beyond the keys in use) ------------------------------
    const int Kreg = (g.num_cells + 7) / 8 * 8 < Kp ? (g.num_cells + 7) / 8 * 8 : Kp;  // regular cells, 16-byte granular
    {
        uint4* dst = reinterpret_cast<uint4*>(ws.chunk_hist + (size_t)(loc.gstart + loc.c) * Kp);
        for (int k8 = tid; k8 < Kp / 8; k8 += kThreads) dst[k8] = reinterpret_cast<const uint4*>(ctot_s)[k8];
        __syncthreads();  // every row store of the CTA happens before the release below (cumulativity)
        if (tid == 0) {
            __threadfence();
            st_release(flags + loc.gstart + loc.c, 1u | ((unsigned)hi_key << 1));  // bit 0: published
        }
        TL(blockIdx.x, 4);
        // wait for the earlier chunks of the tile; learn whether any of them holds keys beyond the regular cells
        int hi_before = 0;
        for (int cc = tid; cc < loc.c; cc += kThreads) {
            unsigned f;
            while ((f = ld_acquire(flags + loc.gstart + cc)) == 0u) {
            }
            hi_before |= (int)(f >> 1);
        }
        hi_key |= (__syncthreads_or(hi_before & 1) ? 1 : 0) | (__syncthreads_or(hi_before & 2) ? 2 : 0);
    }
    TL(blockIdx.x, 5);
    // ---- prefix over the earlier chunks: 8 keys per thread with 16-byte L2 loads, 8 rows in flight per batch; classify
    //      every key of the chunk (dead / free / crossing) ------------------------------------------------------------
    const bool last_chunk = (loc.c == loc.nchunks - 1);
    const int Kuse = (hi_key & 1) ? Kp : Kreg;  // keys that can be non-empty in this tile so far
    int open_keys = 0;  // keys of this chunk that still have room (pre < M): if none, nothing of the chunk is kept
    int all_full = 1;   // every regular cell holds >= M points after this chunk
    for (int k8 = tid; k8 < Kp / 8; k8 += kThreads) {
        unsigned acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (k8 * 8 < Kuse && !(saturated && k8 * 8 + 8 <= g.num_cells)) {
            const uint4* src = reinterpret_cast<const uint4*>(ws.chunk_hist + (size_t)loc.gstart * Kp) + k8;
            const size_t row = (size_t)Kp / 8;
            const uint4* rp = src;
            auto add_rows = [&](const uint4 (&v)[8]) {
                // 8 rows of 16-bit counts (<= 4096 each) add up inside their 16-bit lanes without a carry
                uint4 sum = v[0];
#pragma unroll
                for (int u = 1; u < 8; ++u) { sum.x += v[u].x; sum.y += v[u].y; sum.z += v[u].z; sum.w += v[u].w; }
                acc[0] += sum.x & 0xFFFFu; acc[1] += sum.x >> 16; acc[2] += sum.y & 0xFFFFu; acc[3] += sum.y >> 16;
                acc[4] += sum.z & 0xFFFFu; acc[5] += sum.z >> 16; acc[6] += sum.w & 0xFFFFu; acc[7] += sum.w >> 16;
            };
            int c0 = 0;
            for (; c0 + 8 <= loc.c; c0 += 8, rp += 8 * row) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldcg(rp + u * row);
                add_rows(v);
            }
            if (c0 < loc.c) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = (c0 + u < loc.c) ? __ldcg(rp + u * row) : make_uint4(0, 0, 0, 0);
                add_rows(v);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int k = k8 * 8 + u;
            const unsigned own = ctot_s[k];
            unsigned pre = acc[u];
            if (saturated && k < g.num_cells) pre = (unsigned)M;  // (the rows of saturated chunks hold no regular counts)
            unsigned st = pre < (unsigned)M ? pre : (unsigned)M;
            if (own > 0 && pre < (unsigned)M) {
                open_keys = 1;
                if (pre + own > (unsigned)M) {  // the key crosses M inside this chunk
                    const unsigned id = (unsigned)atomicAdd(&s_ncross, 1);
                    need_s[id] = (uint16_t)((unsigned)M - pre);
                    st = kCrossFlag | id;
                }
            }
            base_s[k] = (uint16_t)st;
            if (k < g.num_cells && pre + own < (unsigned)M) all_full = 0;
            if (last_chunk) {
                const unsigned tot = pre + own;
                if (k < K) ws.totals[(size_t)loc.b * K + k] = (int)tot;
                ctot_s[k] = (uint16_t)(tot < (unsigned)M ? tot : (unsigned)M);  // from here on: min(count, M) of the tile
            }
        }
    }
    open_keys = __syncthreads_or(open_keys);
    all_full = __syncthreads_and(all_full);
    if (all_full && !saturated && !last_chunk && tid == 0) atomicMax(tile_sat + loc.b, 0x7fffffffu - (unsigned)loc.c);
    TL(blockIdx.x, 6);
    // ---- the tile's last chunk knows every count: when no run can be cut, filtered or aliased, the canvas owner table
    //      follows from the keys directly and the tile needs no plan (SURVEY A.1 / A.2 / A.5) ------------------------------
    if (last_chunk) {
        int direct = 0, hi_ok = 0;
        if (!need_plan && !(hi_key & 2)) {
            int r = 0, h = 0;
            for (int k = tid; k < Kuse && k < K; k += kThreads) {
                const int nz = ctot_s[k] > 0 ? 1 : 0;
                if (k < g.num_cells) r += nz; else h += nz;
            }
            r = __reduce_add_sync(0xffffffffu, r);
            h = __reduce_add_sync(0xffffffffu, h);
            if (lane == 0) { atomicAdd(&s_runs[0], r); atomicAdd(&s_runs[1], h); }
            __syncthreads();
            const int R = s_runs[0], H = s_runs[1];
            // runs are numbered in key order and the first max_voxels survive: regular cells all survive iff R <= Vmax;
            // the runs beyond them survive all (R + H <= Vmax) or not at all (R == Vmax); anything else needs the plan
            hi_ok = (R + H <= g.Vmax) ? 1 : 0;
            direct = (R <= g.Vmax) && (H == 0 || hi_ok || R == g.Vmax);
        }
        if (direct) {
            const int HW = g.ny * g.nx;
            const int top = hi_ok ? g.ext[2] : g.ext[2] - 1;  // highest z layer whose runs survive
            for (int cell = tid; cell < HW; cell += kThreads) {
                const int cy = cell / g.nx, cx = cell - cy * g.nx;
                int d = -1;
                if (cx < g.nv[0] && cy < g.nv[1]) {
                    for (int cz = top; cz >= 0; --cz) {  // the last pillar in voxel order (highest key) owns the cell
                        const int k = cx + cy * g.stride1 + cz * g.stride2;
                        const int n = (k < Kuse && k < K) ? (int)ctot_s[k] : 0;
                        if (n > 0) { d = k | (n << 16); break; }
                    }
                }
                ws.cell_desc[(size_t)loc.b * HW + cell] = d;
            }
        }
        if (tid == 0) ws.tile_hi[loc.b] = (hi_key & 1) | (direct << 1);
    }
    // ---- slots: free keys take slot pre + atomic value; crossing keys are resolved below; then one store pass ---------
    // pk[j] becomes key | slot << 13 for a survivor, -1 otherwise
    float4* tile_slots = ws.slots + (size_t)loc.b * K * M;
    unsigned xmask = 0;  // this thread's points that belong to crossing keys
    const int w = tid >> 5;
    if (open_keys) {
#pragma unroll
        for (int j = 0; j < kIters; ++j) {
            if (pk[j] >= 0) {
                const unsigned key = (unsigned)pk[j] & kKeyMask;
                const unsigned st = base_s[key];
                if (st & kCrossFlag) xmask |= 1u << j;
                else if (st < (unsigned)M) pk[j] = (int)(key | ((st + ((unsigned)pk[j] >> kKeyBits)) << kKeyBits));
                else pk[j] = -1;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < kIters; ++j) pk[j] = -1;
    }
    TL(blockIdx.x, 7);
    // ---- crossing keys: the need = M - pre lowest chunk-local indices survive.  The chunk-local order is (group, warp,
    //      lane, e): 32 cells (group, warp) of 128 points.  Per crossing key: count per cell (one atomic per point, its
    //      return value orders the key's points of a cell arbitrarily), exclusive prefix over the cells, the cell in which
    //      the prefix crosses `need`: cells before it survive whole (slot = pre + prefix + atomic value), cells behind it
    //      not at all, and inside the boundary cell the warp that owns it ranks the key's points in (lane, e) order with
    //      ballots.  kCrossBatch keys per round.
    const int ncross = s_ncross;  // (written before the barriers above)
    for (int c0 = 0; c0 < ncross; c0 += kCrossBatch) {
        const int nb = ncross - c0 < kCrossBatch ? ncross - c0 : kCrossBatch;
        {
            uint4* c4 = reinterpret_cast<uint4*>(cell_s);
            for (int i = tid; i < kCells * kCrossBatch / 8; i += kThreads) c4[i] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
        const uint32_t cell_sa = smem_u32(cell_s);
        unsigned bmask = 0;  // this thread's crossing points of the batch
        if (xmask) {
#pragma unroll
            for (int j = 0; j < kIters; ++j) {
                if ((xmask >> j) & 1u) {
                    const unsigned key = (unsigned)pk[j] & kKeyMask;
                    const int id = (int)(base_s[key] & (kCrossFlag - 1u)) - c0;
                    if (id >= 0 && id < nb) {
                        bmask |= 1u << j;
                        const unsigned cell = (unsigned)((j >> 2) * kWarps + w);
                        const unsigned local = atoms_add_u16(cell_sa + 2u * (cell * kCrossBatch + (unsigned)id), 1);
                        pk[j] = (int)(key | (local << kKeyBits));
                    }
                }
            }
        }
        __syncthreads();
        for (int id = tid; id < nb; id += kThreads) {  // exclusive prefix over the cells (conflict-free: ids are the fast index), boundary cell
            const unsigned need = need_s[c0 + id];
            unsigned P = 0, bnd = 0;
            bool found = false;
#pragma unroll 8
            for (int c = 0; c < kCells; ++c) {
                const unsigned v = cell_s[c * kCrossBatch + id];
                cell_s[c * kCrossBatch + id] = (uint16_t)P;
                if (!found && P + v >= need) { found = true; bnd = (unsigned)c | ((need - P) << 8) | (v << 16); }
                P += v;
            }
            bnd_s[id] = bnd;  // cell | survivors inside it << 8 | its points of the key << 16
        }
        __syncthreads();
        if (__any_sync(0xffffffffu, bmask != 0)) {
#pragma unroll
            for (int gi = 0; gi < kGroups; ++gi) {
                const unsigned cell = (unsigned)(gi * kWarps + w);
                unsigned flag = 0;  // per e: boundary-cell point whose fate depends on the (lane, e) order
                int keyv[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = 4 * gi + e;
                    keyv[e] = -1;
                    if ((bmask >> j) & 1u) {
                        const unsigned key = (unsigned)pk[j] & kKeyMask, local = (unsigned)pk[j] >> kKeyBits;
                        const int id = (int)(base_s[key] & (kCrossFlag - 1u)) - c0;
                        const unsigned bnd = bnd_s[id], bc = bnd & 0xFFu, rem = (bnd >> 8) & 0xFFu, cnt = bnd >> 16;
                        const unsigned pre = (unsigned)M - need_s[c0 + id];
                        const unsigned P = cell_s[cell * kCrossBatch + (unsigned)id];
                        if (cell < bc || (cell == bc && rem == cnt)) pk[j] = (int)(key | ((pre + P + local) << kKeyBits));
                        else if (cell > bc) pk[j] = -1;
                        else { flag |= 1u << e; keyv[e] = (int)key; }
                    }
                }
                unsigned pending = __ballot_sync(0xffffffffu, flag != 0);
                while (pending) {  // one round per distinct boundary key of this cell (warp-uniform loop)
                    const int leader = __ffs(pending) - 1;
                    const int mine = (flag & 1u) ? keyv[0] : ((flag & 2u) ? keyv[1] : ((flag & 4u) ? keyv[2] : keyv[3]));
                    const int kk = __shfl_sync(0xffffffffu, mine, leader);
                    unsigned b[4], m = 0;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const bool hit = ((flag >> e) & 1u) && keyv[e] == kk;
                        m |= hit ? (1u << e) : 0u;
                        b[e] = __ballot_sync(0xffffffffu, hit);
                    }
                    if (m) {
                        const int id = (int)(base_s[kk] & (kCrossFlag - 1u)) - c0;
                        const unsigned rem = (bnd_s[id] >> 8) & 0xFFu;
                        const unsigned pre = (unsigned)M - need_s[c0 + id];
                        const unsigned P = cell_s[cell * kCrossBatch + (unsigned)id];
                        const unsigned lt = (1u << lane) - 1u;
                        unsigned below = (unsigned)(__popc(b[0] & lt) + __popc(b[1] & lt) + __popc(b[2] & lt) + __popc(b[3] & lt));
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            if ((m >> e) & 1u) {
                                pk[4 * gi + e] = below < rem ? (int)((unsigned)kk | ((pre + P + below) << kKeyBits)) : -1;
                                ++below;
                            }
                        }
                        flag &= ~m;
                    }
                    pending = __ballot_sync(0xffffffffu, flag != 0);
                }
            }
        }
        xmask &= ~bmask;
        __syncthreads();
    }
    TL(blockIdx.x, 8);
    // ---- store pass: survivors re-read their xyz (L1 / L2 hits; all loads of the chunk in flight at once) ----------------
    {
        unsigned live = 0;  // groups with a survivor
#pragma unroll
        for (int j = 0; j < kIters; ++j) live |= (pk[j] >= 0) ? (1u << (j >> 2)) : 0u;
        if (interior) {
            const float4* q = reinterpret_cast<const float4*>(pts + (loc.p0 + 4ll * tid) * 3);
#pragma unroll
            for (int h = 0; h < kGroups; h += 2) {  // two groups (six loads) in flight at a time: register budget
                float4 v[2][3];
#pragma unroll
                for (int g2 = 0; g2 < 2; ++g2) {
                    if (h + g2 < kGroups && ((live >> (h + g2)) & 1u)) {
#pragma unroll
                        for (int u = 0; u < 3; ++u) v[g2][u] = __ldg(q + (size_t)(h + g2) * (kThreads * 3) + u);
                    }
                }
#pragma unroll
                for (int g2 = 0; g2 < 2; ++g2) {
                    const int gi = (h + g2 < kGroups) ? h + g2 : kGroups - 1;
                    if (h + g2 < kGroups && ((live >> gi) & 1u)) {
                        const float4 a = v[g2][0], b = v[g2][1], c = v[g2][2];
                        const float x[4] = {a.x, a.w, b.z, c.y}, y[4] = {a.y, b.x, b.w, c.z}, z[4] = {a.z, b.y, c.x, c.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = 4 * gi + e;
                            if (pk[j] >= 0) {
                                const int ci = 4 * (kThreads * gi + tid) + e;
                                tile_slots[(size_t)((unsigned)pk[j] & kKeyMask) * M + ((unsigned)pk[j] >> kKeyBits)] =
                                    make_float4(x[e], y[e], z[e], __int_as_float((int)(loc.p0 + ci - lo)));
                            }
                        }
                    }
                }
            }
        } else {
#pragma unroll
            for (int gi = 0; gi < kGroups; ++gi) {
                if ((live >> gi) & 1u) {
                    float x[4], y[4], z[4];
                    load_group(gi, x, y, z);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int j = 4 * gi + e;
                        if (pk[j] >= 0) {
                            const int ci = 4 * (kThreads * gi + tid) + e;
                            tile_slots[(size_t)((unsigned)pk[j] & kKeyMask) * M + ((unsigned)pk[j] >> kKeyBits)] =
                                make_float4(x[e], y[e], z[e], __int_as_float((int)(loc.p0 + ci - lo)));
                        }
                    }
                }
            }
        }
    }
    // ---- the last CTA of the tile to get here plans the tile ------------------------------------------------------------
    __syncthreads();  // every slot / table store of the CTA happens before the fence of thread 0 (cumulativity)
    TL(blockIdx.x, 9);
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(tile_done + loc.b, 1u) == (unsigned)(loc.nchunks - 1)) ? 1 : 0;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    TL(blockIdx.x, 10);
    const int tile_hi = __ldcg(ws.tile_hi + loc.b);
    if (tile_hi & 2) return;  // owner table already written by the tile's last chunk
    plan_tile(g, ws, loc.b, (tile_hi & 1) ? K : (g.num_cells < K ? g.num_cells : K), reinterpret_cast<int*>(smem_raw), warp_tot);
    __syncthreads();
    TL(blockIdx.x, 11);
}

// Parity surface (p3p_voxel_outputs): the reference lists a pillar's points by ascending index; slots are unordered.
__global__ void __launch_bounds__(128)
export_kernel(GridDev g, int B, WsPtrs ws, p3p_voxel_outputs out) {
    __shared__ int idx_s[1024];
    const int b = blockIdx.y;
    const int HW = g.ny * g.nx;
    const int np = ws.num_pil[b];
    if (blockIdx.x == 0) {
        if (out.num_pillars && threadIdx.x == 0) out.num_pillars[b] = np;
        if (out.cell_owner)
            for (int i = threadIdx.x; i < HW; i += blockDim.x) out.cell_owner[(size_t)b * HW + i] = ws.owner[(size_t)b * HW + i];
    }
    for (int r = blockIdx.x; r < np; r += gridDim.x) {
        const size_t pi = (size_t)b * g.Vmax + r;
        const int key = ws.pil_key[pi], n = ws.pil_n[pi], pc = ws.pil_coord[pi];
        if (threadIdx.x == 0) {
            if (out.pillar_coords) {
                int* c = out.pillar_coords + pi * 4;
                c[0] = b; c[1] = pc >> 20; c[2] = (pc >> 10) & 1023; c[3] = pc & 1023;
            }
            if (out.pillar_num_points) out.pillar_num_points[pi] = n;
        }
        const float4* slot = ws.slots + ((size_t)b * g.num_keys + key) * g.M;
        __syncthreads();
        for (int s = threadIdx.x; s < n; s += blockDim.x) idx_s[s] = __float_as_int(slot[s].w);
        __syncthreads();
        for (int s = threadIdx.x; s < g.M; s += blockDim.x) {
            int pos = s;  // padding rows stay where they are
            float4 p = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
            if (s < n) {
                p = slot[s];
                const int me = idx_s[s];
                pos = 0;
                for (int i = 0; i < n; ++i) pos += (idx_s[i] < me) ? 1 : 0;  // indices are distinct
            }
            if (out.pillar_point_idx) out.pillar_point_idx[pi * g.M + pos] = __float_as_int(p.w);
            if (out.pillar_points) {
                float* d = out.pillar_points + (pi * g.M + pos) * 3;
                d[0] = p.x; d[1] = p.y; d[2] = p.z;
            }
        }
    }
}

}  // namespace

size_t voxelize_smem_bytes(const GridDev& g) {
    const size_t kp = ((size_t)g.num_keys + 7) / 8 * 8;
    // chunk counts, bases, crossing needs / counters (uint16 [kp] each), selection scratch
    const size_t rank = 3 * kp * sizeof(uint16_t) + kCrossBatch * sizeof(unsigned) + (size_t)kCells * kCrossBatch * sizeof(uint16_t);
    const size_t plan = (size_t)(4 * g.num_keys + g.ny * g.nx) * sizeof(int);
    return ((rank > plan ? rank : plan) + 15) / 16 * 16;
}

int launch_voxelize(const float* pts, int stride, const int64_t* offsets, int B, int64_t total, const GridDev& g,
                    const WsLayout& l, const WsPtrs& ws, int32_t* point_hash, int need_plan, cudaStream_t st) {
    (void)total;
    const size_t smem = voxelize_smem_bytes(g);
    if (smem > kVoxelizeMaxSmem) return fail(P3P_ERR_UNSUPPORTED, "voxel grid needs %zu bytes of shared memory per CTA (limit %zu)", smem, kVoxelizeMaxSmem);
    // (the attribute belongs to the current device's context: set per launch, it is cheap)
    P3P_CUDA_CHECK(cudaFuncSetAttribute(voxelize_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVoxelizeMaxSmem));
    P3P_CUDA_CHECK(cudaFuncSetAttribute(voxelize_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVoxelizeMaxSmem));
    // ticket counter, chunk flags and per-tile completion counters start at zero for every call
    P3P_CUDA_CHECK(cudaMemsetAsync(ws.sync, 0, l.sync_bytes, st));
    const int pdl_from = l.max_chunks - device_sm_count();  // tickets of the last (partial) wave
    if (stride == 3 && point_hash == nullptr && !(g.flags & kFlagDropOverflow))
        voxelize_kernel<true><<<l.max_chunks, kThreads, smem, st>>>(pts, stride, offsets, B, g, l.chunk_points, ws, point_hash, need_plan, pdl_from);
    else
        voxelize_kernel<false><<<l.max_chunks, kThreads, smem, st>>>(pts, stride, offsets, B, g, l.chunk_points, ws, point_hash, need_plan, pdl_from);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int launch_export(const GridDev& g, int B, const WsPtrs& ws, const p3p_voxel_outputs* out, cudaStream_t st) {
    dim3 grid((unsigned)(g.Vmax < 256 ? (g.Vmax > 0 ? g.Vmax : 1) : 256), (unsigned)B);
    export_kernel<<<grid, 128, 0, st>>>(g, B, ws, *out);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

}  // namespace p3p
