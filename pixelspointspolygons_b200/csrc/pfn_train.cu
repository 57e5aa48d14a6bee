// pfn_train.cu -- training step of the PillarFeatureNet (SURVEY 8f rank 4): BatchNorm batch statistics of both PFN layers
// and the backward pass to the PFN parameters, without ever materialising a (V, M, *) tensor (sm_100a).
//
// Replaces, for `module.train()`, the autograd graph PyTorch builds through Open3D-ML's PillarFeatureNet / PFNLayer
// (call site R:pixelspointspolygons/models/pointpillars/pointpillars_o3d.py:93; DDP / SyncBatchNorm wrap
// R:pixelspointspolygons/models/pix2poly/model_pix2poly.py:326-328).  Voxelisation carries no gradient (the reference runs
// it under @torch.no_grad); gradients reach the six PFN parameters only.
//
// Notation: rows = all V*M slots (padded slots are zero rows of the decorated tensor and DO take part in the statistics,
// as in the reference), d = decorated row (8), y0 = W0 d, yh0 = (y0 - mu0) rstd0, x0 = relu(g0 yh0 + b0),
// z = [x0, hmax] (64), y1 = W1 z, x1 = relu(g1 (y1 - mu1) rstd1 + b1), out = max over the M slots of x1.
//
// Forward.  y is linear in its input, so the batch statistics follow from input moments:
//     sum y_c = W_c . (sum in),   sum y_c^2 = W_c (sum in in^T) W_c^T
// stats0: s = sum d, S = sum d d^T over the kept points (one pass over the slots);
// stats1: sum z, Z = sum z z^T (64 x 64) with x0 from the layer-0 batch statistics (second pass), accumulated in fp32 about
//         a sampled centre and merged / un-centred in float64 (the fp64 pipe of this GPU is ~1 lane per clock and SM).
// Per-channel (sum y, sum y^2, rows) of each layer is what ranks exchange under SyncBatchNorm (65 and 2C + 1 values,
// SURVEY 8e).  With the batch statistics known, BatchNorm is the same affine map as in eval mode; the training forward
// (train_forward_kernel, exact fp32, thread = channel) applies it and keeps the winning row of every (pillar, channel).
// (The inference kernels of pfn.cu on a blob prepared from the batch statistics give the same output faster -- 
// p3p_pfn_train_stats2 + p3p_pfn_prepare + p3p_encode_workspace -- but their tf32 / fp16 operand rounding is amplified by the
// division by the batch's own standard deviation: 2e-3 of scale measured.)
//
// Backward (g = d loss / d out, zero for pillars that lost their canvas cell):
//   pass 1, per pillar and channel c: the winning row m* (kept by the forward), du = g [out > 0];
//           dbeta1_c += du, dgamma1_c += du yh1*, A1[c, :] += du z*  (the sparse part of dW1); (m*, du) kept for pass 2.
//   The BatchNorm backward makes dy1 dense: dy1 = a1 (du - dbeta1 / R - yh1 dgamma1 / R) with a1 = g1 rstd1, but
//           dz = dy1 W1 = G + kvec - Q z,    G = sparse rows, kvec (64), Q (64 x 64) batch constants,
//   so pass 2 needs 64 x 64 per row instead of C x 64.  pass 2, per pillar: dz rows -> dx0 (+ the hmax route) -> du0 =
//           dx0 [x0 > 0]; dbeta0, dgamma0, A0 = sum du0 d^T.
//   finish: dW = a (A - (dbeta / R) sum in - (dgamma / R) rstd (W M_in - mu sum in)) per layer, from the stored moments.
// Tie-breaking of the two arg maxima is immaterial: tied rows are identical rows (padded slots, duplicated points) or sit
// at relu's zero, where the gradient vanishes.
#include <cmath>
#include <cstring>

#include "p3p_internal.cuh"

namespace p3p {
namespace {

constexpr int kTrainMaxM = 512;
constexpr int kTrainMaxC = 512;  // thread = channel kernels: one CTA of at most 512 threads; back2 covers c and c + 256
constexpr int kXS = 36;  // floats per x0 / yh0 row in shared memory (16-byte aligned rows: broadcast float4 loads)

struct TrainLayout {
    int C;
    int64_t mom0, sums0, bn0, mom1, sums1, bn1, cen, back1, back1g, A1, kq, back0, back0g, A0, total;
};
TrainLayout make_train_layout(int C) {
    TrainLayout l;
    l.C = C;
    int64_t off = 0;
    auto take = [&](int64_t n) { int64_t o = off; off += (n + 15) / 16 * 16; return o; };
    l.mom0 = take(1 + 8 + 64);        // rows of this rank, s[8], S[8][8]
    l.sums0 = take(65);               // sum y0 [32], sum y0^2 [32], rows                    (all-reduced in place)
    l.bn0 = take(64);                 // mean0 [32], biased var0 [32]
    l.mom1 = take(64 + 4096);         // sum z [64], Z[64][64]
    l.sums1 = take(2 * (int64_t)C + 1);
    l.bn1 = take(2 * (int64_t)C);
    l.cen = take(65);                 // centre of the layer-1 moment accumulation: sum z over a sample of pillars [64], its rows
    l.back1 = take(2 * (int64_t)C);   // dbeta1 [C], dgamma1 [C] of this rank
    l.back1g = take(2 * (int64_t)C);  // the same summed over the ranks of the SyncBatchNorm group
    l.A1 = take((int64_t)C * 64);
    l.kq = take(64 + 4096);           // kvec [64], Q[64][64]
    l.back0 = take(64);
    l.back0g = take(64);
    l.A0 = take(256);
    l.total = off;
    return l;
}

struct TrainArgs {
    GridDev g;
    WsPtrs ws;
    int B, C, alias;
    float eps;
    const float *W0, *g0, *b0, *W1, *g1, *b1;
    double* st;
    TrainLayout tl;
    const float* gout;  // (B, ny nx, C) fp32
    float* out;         // (B, ny nx, C) fp32: the forward output (written by the forward, read by backward pass 1)
    float* du;          // (B Vmax, C)
    uint16_t* amax;     // (B Vmax, C)
};

struct Pillar {
    int b, r, n, key, cell, own;
    float ctr_x, ctr_y;
};
// descriptor of the compacted list: x = tile, y = voxel ordinal, z = key | n << 16, w = cell | owns-its-cell << 30
__device__ __forceinline__ Pillar unpack(const TrainArgs& a, const int4 d) {
    Pillar p;
    p.b = d.x; p.r = d.y; p.key = d.z & 0xFFFF; p.n = d.z >> 16; p.cell = d.w & 0x3FFFFFFF; p.own = (d.w >> 30) & 1;
    const int cy = p.cell / a.g.nx, cx = p.cell - cy * a.g.nx;
    p.ctr_x = __fmaf_rn((float)cx, a.g.vx, a.g.x_off);
    p.ctr_y = __fmaf_rn((float)cy, a.g.vy, a.g.y_off);
    return p;
}
__device__ __forceinline__ const float4* slots_of(const TrainArgs& a, const int4 d) {
    return a.ws.slots + ((int64_t)d.x * a.g.num_keys + (d.z & 0xFFFF)) * a.g.M;
}

// The batch's pillars in voxel order, compacted: the per-pillar kernels walk this list with the next descriptor and the
// next pillar's points already in registers (no dependent global load inside their loops).
__global__ void train_list_kernel(TrainArgs a) {
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    const int HW = a.g.ny * a.g.nx;
    if (item == 0) {
        int total = 0;
        for (int b = 0; b < a.B; ++b) total += a.ws.num_pil[b];
        a.ws.train_count[0] = total;
    }
    if (item >= a.B * a.g.Vmax) return;
    const int b = item / a.g.Vmax, r = item - b * a.g.Vmax;
    if (r >= a.ws.num_pil[b]) return;
    int base = 0;
    for (int bb = 0; bb < b; ++bb) base += a.ws.num_pil[bb];
    const int64_t pi = (int64_t)b * a.g.Vmax + r;
    const int pc = a.ws.pil_coord[pi];
    const int cell = ((pc >> 10) & 1023) * a.g.nx + (pc & 1023);
    const int own = a.ws.owner[(size_t)b * HW + cell] == r;
    a.ws.train_list[base + r] = make_int4(b, r, a.ws.pil_key[pi] | (a.ws.pil_n[pi] << 16), cell | (own << 30));
}

// Walk of the compacted list by one CTA: descriptors two pillars ahead, row `threadIdx.x` of the next pillar one ahead.
struct Walk {
    int i, count, step;
    int4 d0, d1, d2;
    float4 q0, q1;
};
__device__ __forceinline__ void walk_begin(Walk& w, const TrainArgs& a) {
    w.count = a.ws.train_count[0];
    w.step = gridDim.x;
    w.i = blockIdx.x;
    const int4 z = make_int4(0, 0, 0, 0);
    w.d0 = w.i < w.count ? a.ws.train_list[w.i] : z;
    w.d1 = w.i + w.step < w.count ? a.ws.train_list[w.i + w.step] : z;
    w.d2 = z;
    w.q0 = make_float4(0.f, 0.f, 0.f, 0.f);
    w.q1 = w.q0;
    if (w.i < w.count && (int)threadIdx.x < (w.d0.z >> 16)) w.q0 = slots_of(a, w.d0)[threadIdx.x];
}
// issue the loads of the following pillars (call at the top of an iteration)
__device__ __forceinline__ void walk_prefetch(Walk& w, const TrainArgs& a) {
    if (w.i + w.step < w.count && (int)threadIdx.x < (w.d1.z >> 16)) w.q1 = slots_of(a, w.d1)[threadIdx.x];
    if (w.i + 2 * w.step < w.count) w.d2 = a.ws.train_list[w.i + 2 * w.step];
}
__device__ __forceinline__ void walk_next(Walk& w) {
    w.i += w.step;
    w.d0 = w.d1; w.d1 = w.d2; w.q0 = w.q1;
}

// Shared-memory carve-up of the per-pillar kernels (floats).
struct Smem {
    float* D;     // [M][8]      decorated rows (r < n)
    float* X0;    // [M + 1][36] x0 rows; row n = one representative padded slot (present iff n < M)
    float* YH;    // [M + 1][36] yh0 rows (backward pass 2 only)
    float* w0;    // [32][8]
    float* a0;    // [32]  g0 rstd0
    float* sh0;   // [32]  b0 - mu0 a0
    float* mu0;   // [32]
    float* rs0;   // [32]
    float* hmax;  // [32]
    float* sx;    // [32]  sum over the M slots of x0
    int* am0;     // [32]  arg max row of hmax
    int* red;     // [16][6]
    float* part_max;  // [16][32] per-warp partials of the column scan
    float* part_sum;  // [16][32]
    int* part_arg;    // [16][32]
    float* extra;
};
__device__ __forceinline__ Smem carve(float* base, int M, bool want_yh) {
    Smem s;
    s.D = base;
    s.X0 = s.D + (size_t)M * 8;
    s.YH = s.X0 + (size_t)(M + 1) * kXS;
    s.w0 = s.YH + (want_yh ? (size_t)(M + 1) * kXS : 0);
    s.a0 = s.w0 + 256;
    s.sh0 = s.a0 + 32;
    s.mu0 = s.sh0 + 32;
    s.rs0 = s.mu0 + 32;
    s.hmax = s.rs0 + 32;
    s.sx = s.hmax + 32;
    s.am0 = reinterpret_cast<int*>(s.sx + 32);
    s.red = s.am0 + 32;
    s.part_max = reinterpret_cast<float*>(s.red + 96);
    s.part_sum = s.part_max + 512;
    s.part_arg = reinterpret_cast<int*>(s.part_sum + 512);
    s.extra = reinterpret_cast<float*>(s.part_arg + 512);
    return s;
}
size_t smem_floats(int M, bool want_yh) { return (size_t)M * 8 + (size_t)(M + 1) * kXS * (want_yh ? 2 : 1) + 256 + 6 * 32 + 32 + 96 + 3 * 512; }

constexpr int kStats0Acc = 45;  // static float64 accumulators of train_stats0_kernel: rows, s[8], upper triangle of S

// Dynamic shared memory (bytes) of every per-pillar kernel of the step, in one place: the launches take their sizes from
// here, and fill_args refuses a (C, M) that any of them could not launch before an entry point does anything.
struct TrainSmem {
    size_t stats0, centre, stats1, forward, back1, back2;
    size_t max_block;  // the largest dynamic + static shared memory of one CTA among them
};
TrainSmem train_smem(int M, int C) {
    TrainSmem t;
    const size_t base = smem_floats(M, false) * 4;
    t.stats0 = base;
    t.centre = base;
    t.stats1 = base + 64 * sizeof(float);                  // + the centre of the layer-1 moments
    t.forward = base;
    t.back1 = base + (size_t)64 * C * sizeof(float);       // + A1s, the sparse dW1 block of the CTA
    const size_t fl = smem_floats(M, false) + (size_t)(M + 1) * 33 + 3 * (size_t)C + 32 + 64 + 64 + 32 * 64;
    t.back2 = (fl + 8 * 32 * 10 + (size_t)M + 2 + C) * 4;  // see the carve-up at the top of train_back2_kernel
    t.max_block = t.stats0 + kStats0Acc * sizeof(double);
    for (size_t v : {t.centre, t.stats1, t.forward, t.back1, t.back2}) t.max_block = v > t.max_block ? v : t.max_block;
    return t;
}

// layer-0 constants of the batch into shared memory (bn0 must be final)
__device__ __forceinline__ void load_layer0(const TrainArgs& a, const Smem& s) {
    const double* bn0 = a.st + a.tl.bn0;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s.w0[i] = a.W0[i];
    if (threadIdx.x < 32) {
        const int k = threadIdx.x;
        const float mu = (float)bn0[k];
        const float rs = (float)(1.0 / sqrt(bn0[32 + k] + (double)a.eps));
        const float aa = a.g0[k] * rs;
        s.mu0[k] = mu; s.rs0[k] = rs; s.a0[k] = aa; s.sh0[k] = a.b0[k] - mu * aa;
    }
}

// decorated rows of one pillar (whole CTA; ends with a barrier).  q = the pillar's point of row threadIdx.x (prefetched).
__device__ __forceinline__ void decorate(const TrainArgs& a, const Pillar& p, const float4* slot, const float4 q0, const Smem& s) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nwarps = blockDim.x >> 5;
    int sl[3] = {0, 0, 0}, sh[3] = {0, 0, 0};
    for (int r = tid; r < p.n; r += blockDim.x) {
        const float4 q = (r == tid) ? q0 : slot[r];
        int lo, hi;
        fix_split(q.x, a.g.fix_scale, lo, hi); sl[0] += lo; sh[0] += hi;
        fix_split(q.y, a.g.fix_scale, lo, hi); sl[1] += lo; sh[1] += hi;
        fix_split(q.z, a.g.fix_scale, lo, hi); sl[2] += lo; sh[2] += hi;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        sl[i] = __reduce_add_sync(0xffffffffu, sl[i]);
        sh[i] = __reduce_add_sync(0xffffffffu, sh[i]);
        if (lane == 0) { s.red[w * 6 + i] = sl[i]; s.red[w * 6 + 3 + i] = sh[i]; }
    }
    __syncthreads();
    int tl[3] = {0, 0, 0}, th[3] = {0, 0, 0};
    for (int ww = 0; ww < nwarps; ++ww) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { tl[i] += s.red[ww * 6 + i]; th[i] += s.red[ww * 6 + 3 + i]; }
    }
    const float fn = (float)p.n;
    const float mx = fix_mean(tl[0], th[0], a.g.fix_inv, fn);
    const float my = fix_mean(tl[1], th[1], a.g.fix_inv, fn);
    const float mz = fix_mean(tl[2], th[2], a.g.fix_inv, fn);
    for (int r = tid; r < p.n; r += blockDim.x) {
        const float4 q = (r == tid) ? q0 : slot[r];
        const float xc = q.x - p.ctr_x, yc = q.y - p.ctr_y;
        float4 lo4, hi4;
        lo4.x = a.alias ? xc : q.x; lo4.y = a.alias ? yc : q.y; lo4.z = q.z; lo4.w = q.x - mx;
        hi4.x = q.y - my; hi4.y = q.z - mz; hi4.z = xc; hi4.w = yc;
        reinterpret_cast<float4*>(s.D + (size_t)r * 8)[0] = lo4;
        reinterpret_cast<float4*>(s.D + (size_t)r * 8)[1] = hi4;
    }
    __syncthreads();
}

// x0 (and yh0) rows, hmax with its arg max row, sx = sum over the M slots of x0 (whole CTA; ends with a barrier).
// Returns the number of distinct rows: n real ones + one representative padded slot when n < M.
template <bool kYH>
__device__ __forceinline__ int layer0_rows(const TrainArgs& a, const Pillar& p, const Smem& s) {
    const int tid = threadIdx.x, M = a.g.M;
    const int kg = tid & 3, rows_per_pass = blockDim.x >> 2;
    for (int r = tid >> 2; r < p.n; r += rows_per_pass) {
        const float4 dl = reinterpret_cast<const float4*>(s.D + (size_t)r * 8)[0];
        const float4 dh = reinterpret_cast<const float4*>(s.D + (size_t)r * 8)[1];
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            const int k = kg * 8 + kk;
            const float* wr = s.w0 + k * 8;
            float y = wr[0] * dl.x;
            y = __fmaf_rn(wr[1], dl.y, y); y = __fmaf_rn(wr[2], dl.z, y); y = __fmaf_rn(wr[3], dl.w, y);
            y = __fmaf_rn(wr[4], dh.x, y); y = __fmaf_rn(wr[5], dh.y, y); y = __fmaf_rn(wr[6], dh.z, y);
            y = __fmaf_rn(wr[7], dh.w, y);
            s.X0[(size_t)r * kXS + k] = fmaxf(__fmaf_rn(s.a0[k], y, s.sh0[k]), 0.f);
            if (kYH) s.YH[(size_t)r * kXS + k] = (y - s.mu0[k]) * s.rs0[k];
        }
    }
    const int rows = p.n + (p.n < M ? 1 : 0);
    if (p.n < M && tid < 32) {
        s.X0[(size_t)p.n * kXS + tid] = fmaxf(s.sh0[tid], 0.f);
        if (kYH) s.YH[(size_t)p.n * kXS + tid] = -s.mu0[tid] * s.rs0[tid];
    }
    __syncthreads();
    {   // column k by warp w: partial (max, arg max, weighted sum) over rows w, w + nwarps, ...; then 32 threads merge them
        const int k = tid & 31, wq = tid >> 5, nw = blockDim.x >> 5;
        float best = -1.f, sum = 0.f;
        int arg = 0;
        for (int r = wq; r < rows; r += nw) {
            const float v = s.X0[(size_t)r * kXS + k];
            sum += (r < p.n) ? v : v * (float)(M - p.n);
            if (v > best) { best = v; arg = r; }
        }
        s.part_max[wq * 32 + k] = best; s.part_arg[wq * 32 + k] = arg; s.part_sum[wq * 32 + k] = sum;
    }
    __syncthreads();
    if (tid < 32) {
        const int nw = blockDim.x >> 5;
        float best = -1.f, sum = 0.f;
        int arg = 0;
        for (int wq = 0; wq < nw; ++wq) {  // fixed order: deterministic; ties keep the lowest row
            const float v = s.part_max[wq * 32 + tid];
            const int ar = s.part_arg[wq * 32 + tid];
            sum += s.part_sum[wq * 32 + tid];
            if (v > best || (v == best && ar < arg)) { best = v; arg = ar; }
        }
        s.hmax[tid] = best; s.am0[tid] = arg; s.sx[tid] = sum;
    }
    __syncthreads();
    return rows;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------------
// forward statistics.  This GPU's fp64 pipe issues about one lane per clock and SM, so the moments are accumulated in
// fp32 about a centre close to the mean (then nothing cancels in E[y^2] - E[y]^2 and in the centred second moments of the
// backward) and only merged in float64.  Layer 0: the decorated channels are offsets, centre 0 is close enough.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) train_stats0_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    __shared__ double acc[kStats0Acc];
    const int tid = threadIdx.x;
    if (tid < kStats0Acc) acc[tid] = 0.0;
    float m1[8], m2[36];
#pragma unroll
    for (int i = 0; i < 8; ++i) m1[i] = 0.f;
#pragma unroll
    for (int i = 0; i < 36; ++i) m2[i] = 0.f;
    int pillars = 0;
    Walk w;
    walk_begin(w, a);
    for (; w.i < w.count; walk_next(w)) {
        walk_prefetch(w, a);
        const Pillar p = unpack(a, w.d0);
        ++pillars;
        decorate(a, p, slots_of(a, w.d0), w.q0, s);
        for (int r = tid; r < p.n; r += blockDim.x) {
            float d[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) d[i] = s.D[(size_t)r * 8 + i];
            int e = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                m1[i] += d[i];
#pragma unroll
                for (int j = i; j < 8; ++j) { m2[e] = __fmaf_rn(d[i], d[j], m2[e]); ++e; }
            }
        }
        __syncthreads();
    }
    const int lane = tid & 31;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const double v = warp_sum_d((double)m1[i]);
        if (lane == 0) atomicAdd(&acc[1 + i], v);
    }
#pragma unroll
    for (int e = 0; e < 36; ++e) {
        const double v = warp_sum_d((double)m2[e]);
        if (lane == 0) atomicAdd(&acc[9 + e], v);
    }
    if (tid == 0) acc[0] = (double)pillars * (double)a.g.M;
    __syncthreads();
    double* mom = a.st + a.tl.mom0;
    if (tid == 0) atomicAdd(mom, acc[0]);
    if (tid >= 1 && tid < 9) atomicAdd(mom + tid, acc[tid]);
    if (tid < 36) {  // upper triangle -> full symmetric matrix
        int i = 0, e = tid;
        while (e >= 8 - i) { e -= 8 - i; ++i; }
        const int j = i + e;
        atomicAdd(mom + 9 + i * 8 + j, acc[9 + tid]);
        if (j != i) atomicAdd(mom + 9 + j * 8 + i, acc[9 + tid]);
    }
}

// per-channel sums of a linear layer's outputs from the input moments: sum y = W s, sum y^2 = W S W^T
// (one CTA of 64 threads per channel, K <= 64)
__global__ void __launch_bounds__(64) train_sums_kernel(const float* __restrict__ W, int C, int K, const double* __restrict__ s,
                                                        const double* __restrict__ S, const double* __restrict__ rows_ptr,
                                                        double* __restrict__ sums) {
    __shared__ double part[4];
    const int c = blockIdx.x, i = threadIdx.x;
    double sy = 0.0, syy = 0.0;
    if (i < K) {
        const double wi = (double)W[(size_t)c * K + i];
        double t = 0.0;
        for (int j = 0; j < K; ++j) t = fma(S[i * K + j], (double)W[(size_t)c * K + j], t);
        sy = wi * s[i];
        syy = wi * t;
    }
    sy = warp_sum_d(sy);
    syy = warp_sum_d(syy);
    if ((i & 31) == 0) { part[(i >> 5) * 2] = sy; part[(i >> 5) * 2 + 1] = syy; }
    __syncthreads();
    if (i == 0) {
        sums[c] = part[0] + part[2];
        sums[C + c] = part[1] + part[3];
        if (c == 0) sums[2 * C] = *rows_ptr;
    }
}

// batch mean and biased variance from the (all-reduced) sums
__global__ void train_bn_kernel(const double* __restrict__ sums, int C, double* __restrict__ bn, float* __restrict__ mean_f, float* __restrict__ var_f) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double rows = sums[2 * C];
    double mean = 0.0, var = 0.0;
    if (rows > 0.0) {
        mean = sums[c] / rows;
        var = sums[C + c] / rows - mean * mean;
        if (var < 0.0) var = 0.0;
    }
    bn[c] = mean;
    bn[C + c] = var;
    if (mean_f) mean_f[c] = (float)mean;
    if (var_f) var_f[c] = (float)var;
}

// centre of the layer-1 moments: sum of z over a sample of the batch's pillars (any point within a spread of the mean
// will do; hmax in particular has a mean many times its spread)
constexpr int kCentreCtas = 32, kCentrePillars = 4;
__global__ void __launch_bounds__(256) train_centre_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    const int tid = threadIdx.x;
    load_layer0(a, s);
    __syncthreads();
    const int count = a.ws.train_count[0];
    double* cen = a.st + a.tl.cen;
    for (int t = 0, i = blockIdx.x; t < kCentrePillars && i < count; ++t, i += gridDim.x) {
        const int4 d = a.ws.train_list[i];
        const Pillar p = unpack(a, d);
        const float4* slot = slots_of(a, d);
        const float4 q0 = tid < p.n ? slot[tid] : make_float4(0.f, 0.f, 0.f, 0.f);
        decorate(a, p, slot, q0, s);
        layer0_rows<false>(a, p, s);
        if (tid < 32) {
            atomicAdd(cen + tid, (double)s.sx[tid]);
            atomicAdd(cen + 32 + tid, (double)((float)a.g.M * s.hmax[tid]));
        }
        if (tid == 0) atomicAdd(cen + 64, (double)a.g.M);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) train_stats1_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    float* cz = s.extra;  // [64] centre
    const int tid = threadIdx.x, M = a.g.M;
    load_layer0(a, s);
    if (tid < 64) {
        const double* cen = a.st + a.tl.cen;
        cz[tid] = cen[64] > 0.0 ? (float)(cen[tid] / cen[64]) : 0.f;
    }
    __syncthreads();
    const int i0 = (tid >> 4) * 2, j0 = (tid & 15) * 2;
    const float ci0 = cz[i0], ci1 = cz[i0 + 1], cj0 = cz[j0], cj1 = cz[j0 + 1];
    const float chi0 = cz[32 + i0], chi1 = cz[32 + i0 + 1], chj0 = cz[32 + j0], chj1 = cz[32 + j0 + 1];
    float aX[4] = {0, 0, 0, 0}, aC[4] = {0, 0, 0, 0}, aH[4] = {0, 0, 0, 0}, aS = 0.f, aSh = 0.f;
    Walk w;
    walk_begin(w, a);
    for (; w.i < w.count; walk_next(w)) {
        walk_prefetch(w, a);
        const Pillar p = unpack(a, w.d0);
        decorate(a, p, slots_of(a, w.d0), w.q0, s);
        const int rows = layer0_rows<false>(a, p, s);
        float x[4] = {0.f, 0.f, 0.f, 0.f};
        for (int r = 0; r < rows; ++r) {
            const float wt = (r < p.n) ? 1.f : (float)(M - p.n);
            const float2 vi = *reinterpret_cast<const float2*>(s.X0 + (size_t)r * kXS + i0);
            const float2 vj = *reinterpret_cast<const float2*>(s.X0 + (size_t)r * kXS + j0);
            const float xi0 = (vi.x - ci0) * wt, xi1 = (vi.y - ci1) * wt, xj0 = vj.x - cj0, xj1 = vj.y - cj1;
            x[0] = __fmaf_rn(xi0, xj0, x[0]); x[1] = __fmaf_rn(xi0, xj1, x[1]);
            x[2] = __fmaf_rn(xi1, xj0, x[2]); x[3] = __fmaf_rn(xi1, xj1, x[3]);
        }
        const float fm = (float)M;
        const float hi0 = s.hmax[i0] - chi0, hi1 = s.hmax[i0 + 1] - chi1, hj0 = s.hmax[j0] - chj0, hj1 = s.hmax[j0 + 1] - chj1;
        const float si0 = s.sx[i0] - fm * ci0, si1 = s.sx[i0 + 1] - fm * ci1;
        aX[0] += x[0]; aX[1] += x[1]; aX[2] += x[2]; aX[3] += x[3];
        aC[0] = __fmaf_rn(si0, hj0, aC[0]); aC[1] = __fmaf_rn(si0, hj1, aC[1]);
        aC[2] = __fmaf_rn(si1, hj0, aC[2]); aC[3] = __fmaf_rn(si1, hj1, aC[3]);
        aH[0] = __fmaf_rn(fm * hi0, hj0, aH[0]); aH[1] = __fmaf_rn(fm * hi0, hj1, aH[1]);
        aH[2] = __fmaf_rn(fm * hi1, hj0, aH[2]); aH[3] = __fmaf_rn(fm * hi1, hj1, aH[3]);
        if (tid < 32) { aS += s.sx[tid] - fm * cz[tid]; aSh += fm * (s.hmax[tid] - cz[32 + tid]); }
        __syncthreads();
    }
    double* sz = a.st + a.tl.mom1;
    double* Z = sz + 64;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int i = i0 + (e >> 1), j = j0 + (e & 1);
        atomicAdd(Z + i * 64 + j, (double)aX[e]);
        atomicAdd(Z + i * 64 + 32 + j, (double)aC[e]);
        atomicAdd(Z + (32 + j) * 64 + i, (double)aC[e]);
        atomicAdd(Z + (32 + i) * 64 + 32 + j, (double)aH[e]);
    }
    if (tid < 32) { atomicAdd(sz + tid, (double)aS); atomicAdd(sz + 32 + tid, (double)aSh); }
}

// centred -> raw moments, in float64: Z += c szc^T + szc c^T + R c c^T, sz = szc + R c
__global__ void __launch_bounds__(1024) train_uncentre_kernel(TrainArgs a) {
    __shared__ double c[64], szc[64];
    const int tid = threadIdx.x;
    const double R = a.st[a.tl.mom0];
    double* sz = a.st + a.tl.mom1;
    double* Z = sz + 64;
    const double* cen = a.st + a.tl.cen;
    if (tid < 64) {
        c[tid] = cen[64] > 0.0 ? (double)(float)(cen[tid] / cen[64]) : 0.0;  // (the fp32 value the kernel subtracted)
        szc[tid] = sz[tid];
    }
    __syncthreads();
    for (int e = tid; e < 4096; e += blockDim.x) {
        const int i = e >> 6, j = e & 63;
        Z[e] += c[i] * szc[j] + szc[i] * c[j] + R * c[i] * c[j];
    }
    if (tid < 64) sz[tid] = szc[tid] + R * c[tid];
}

// ------------------------------------------------------------------------------------------------
// training forward (exact fp32, thread = channel): out = relu(max over the rows of BatchNorm(y1)) for the pillars that own
// their canvas cell, together with the winning row of every (pillar, channel) for the backward pass
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) train_forward_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    const int tid = threadIdx.x, C = a.C, HW = a.g.ny * a.g.nx;
    load_layer0(a, s);
    const double* bn1 = a.st + a.tl.bn1;
    const int c = tid < C ? tid : 0;
    const float mu1 = (float)bn1[c];
    const float rs1 = (float)(1.0 / sqrt(bn1[C + c] + (double)a.eps));
    const float a1 = a.g1[c] * rs1;
    const float sh1 = a.b1[c] - mu1 * a1;
    float wf[64];  // folded row of W1: the arg max over the rows is taken on the BatchNorm output (the sign of a1 matters)
#pragma unroll
    for (int j = 0; j < 64; ++j) wf[j] = a1 * a.W1[(size_t)c * 64 + j];
    __syncthreads();
    Walk w;
    walk_begin(w, a);
    for (; w.i < w.count; walk_next(w)) {
        walk_prefetch(w, a);
        const Pillar p = unpack(a, w.d0);
        if (!p.own) continue;  // overwritten on the canvas (PointPillarsScatter's last writer wins)
        decorate(a, p, slots_of(a, w.d0), w.q0, s);
        const int rows = layer0_rows<false>(a, p, s);
        if (tid < C) {
            float gconst = sh1;
#pragma unroll
            for (int k = 0; k < 32; ++k) gconst = __fmaf_rn(wf[32 + k], s.hmax[k], gconst);
            float best = -INFINITY;
            int arg = 0;
            for (int r = 0; r < rows; ++r) {
                const float4* xr = reinterpret_cast<const float4*>(s.X0 + (size_t)r * kXS);
                float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
                for (int k4 = 0; k4 < 8; k4 += 2) {
                    const float4 x = xr[k4], y = xr[k4 + 1];
                    acc0 = __fmaf_rn(wf[k4 * 4 + 0], x.x, acc0); acc0 = __fmaf_rn(wf[k4 * 4 + 1], x.y, acc0);
                    acc0 = __fmaf_rn(wf[k4 * 4 + 2], x.z, acc0); acc0 = __fmaf_rn(wf[k4 * 4 + 3], x.w, acc0);
                    acc1 = __fmaf_rn(wf[k4 * 4 + 4], y.x, acc1); acc1 = __fmaf_rn(wf[k4 * 4 + 5], y.y, acc1);
                    acc1 = __fmaf_rn(wf[k4 * 4 + 6], y.z, acc1); acc1 = __fmaf_rn(wf[k4 * 4 + 7], y.w, acc1);
                }
                const float acc = acc0 + acc1;
                if (acc > best) { best = acc; arg = r; }
            }
            a.out[((size_t)p.b * HW + p.cell) * C + tid] = fmaxf(best + gconst, 0.f);
            a.amax[((size_t)p.b * a.g.Vmax + p.r) * C + tid] = (uint16_t)arg;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// backward pass 1 (thread = channel): du = g [out > 0] on the winning row kept by the forward
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) train_back1_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    float* A1s = s.extra;  // [64][C]
    const int tid = threadIdx.x, C = a.C, HW = a.g.ny * a.g.nx;
    load_layer0(a, s);
    for (int i = tid; i < 64 * C; i += blockDim.x) A1s[i] = 0.f;
    const double* bn1 = a.st + a.tl.bn1;
    const int c = tid < C ? tid : 0;
    const float mu1 = (float)bn1[c];
    const float rs1 = (float)(1.0 / sqrt(bn1[C + c] + (double)a.eps));
    float wr[64];  // raw row of W1
#pragma unroll
    for (int j = 0; j < 64; ++j) wr[j] = a.W1[(size_t)c * 64 + j];
    float dbeta = 0.f, dgamma = 0.f;  // (fp32 over this CTA's pillars, float64 across CTAs)
    __syncthreads();
    Walk w;
    walk_begin(w, a);
    // of this channel: d loss / d out masked by out > 0, and the winning row -- current pillar, next pillar
    float g0 = 0.f, g1 = 0.f;
    int m0 = 0, m1 = 0;
    auto fetch = [&](const int4 d, float& g, int& m) {
        g = 0.f; m = 0;
        if (!((d.w >> 30) & 1) || tid >= C) return;
        const size_t o = ((size_t)d.x * HW + (d.w & 0x3FFFFFFF)) * C + tid;
        g = a.out[o] > 0.f ? a.gout[o] : 0.f;
        m = a.amax[((size_t)d.x * a.g.Vmax + d.y) * C + tid];
    };
    if (w.i < w.count) fetch(w.d0, g0, m0);
    for (; w.i < w.count; walk_next(w), g0 = g1, m0 = m1) {
        walk_prefetch(w, a);
        if (w.i + w.step < w.count) fetch(w.d1, g1, m1);
        const Pillar p = unpack(a, w.d0);
        if (!p.own) continue;  // no gradient reaches it (backward 2 treats its du as zero)
        decorate(a, p, slots_of(a, w.d0), w.q0, s);
        layer0_rows<false>(a, p, s);
        if (tid < C) {
            const float du = g0;
            a.du[((size_t)p.b * a.g.Vmax + p.r) * C + tid] = du;
            if (du != 0.f) {
                const float4* xr = reinterpret_cast<const float4*>(s.X0 + (size_t)m0 * kXS);
                float y = 0.f;
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 x = xr[k4];
                    y = __fmaf_rn(wr[k4 * 4 + 0], x.x, y); y = __fmaf_rn(wr[k4 * 4 + 1], x.y, y);
                    y = __fmaf_rn(wr[k4 * 4 + 2], x.z, y); y = __fmaf_rn(wr[k4 * 4 + 3], x.w, y);
                    A1s[(k4 * 4 + 0) * C + tid] = __fmaf_rn(du, x.x, A1s[(k4 * 4 + 0) * C + tid]);
                    A1s[(k4 * 4 + 1) * C + tid] = __fmaf_rn(du, x.y, A1s[(k4 * 4 + 1) * C + tid]);
                    A1s[(k4 * 4 + 2) * C + tid] = __fmaf_rn(du, x.z, A1s[(k4 * 4 + 2) * C + tid]);
                    A1s[(k4 * 4 + 3) * C + tid] = __fmaf_rn(du, x.w, A1s[(k4 * 4 + 3) * C + tid]);
                }
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const float h = s.hmax[k];
                    y = __fmaf_rn(wr[32 + k], h, y);
                    A1s[(32 + k) * C + tid] = __fmaf_rn(du, h, A1s[(32 + k) * C + tid]);
                }
                dbeta += du;
                dgamma = __fmaf_rn(du, (y - mu1) * rs1, dgamma);
            }
        }
        __syncthreads();
    }
    if (tid < C) {
        double* back = a.st + a.tl.back1;
        atomicAdd(back + tid, (double)dbeta);
        atomicAdd(back + C + tid, (double)dgamma);
        double* A1 = a.st + a.tl.A1;
        for (int j = 0; j < 64; ++j) {
            const float v = A1s[j * C + tid];
            if (v != 0.f) atomicAdd(A1 + (size_t)tid * 64 + j, (double)v);
        }
    }
}

// batch constants of the dense part of dz (one CTA of 64 threads per row of Q, the last CTA: kvec):
//   kvec[j] = sum_c a1_c / R (-dbeta_c + dgamma_c rstd_c mu_c) W1[c][j],  Q[j][i] = sum_c a1_c (dgamma_c / R) rstd_c W1[c][j] W1[c][i]
__global__ void __launch_bounds__(64) train_kq_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    double* coef = reinterpret_cast<double*>(smem_f);  // [C]
    const int C = a.C, tid = threadIdx.x, j = blockIdx.x;
    const double* bn1 = a.st + a.tl.bn1;
    const double* bg = a.st + a.tl.back1g;
    const double rows = a.st[a.tl.sums1 + 2 * C];
    const double ir = rows > 0.0 ? 1.0 / rows : 0.0;
    for (int c = tid; c < C; c += blockDim.x) {
        const double rs = 1.0 / sqrt(bn1[C + c] + (double)a.eps);
        const double a1 = (double)a.g1[c] * rs;
        coef[c] = (j < 64) ? a1 * ir * bg[C + c] * rs * (double)a.W1[(size_t)c * 64 + j] : a1 * ir * (-bg[c] + bg[C + c] * rs * bn1[c]);
    }
    __syncthreads();
    double acc = 0.0;
    for (int c = 0; c < C; ++c) acc = fma(coef[c], (double)a.W1[(size_t)c * 64 + tid], acc);
    double* kq = a.st + a.tl.kq;
    if (j < 64) kq[64 + j * 64 + tid] = acc; else kq[tid] = acc;
}
// kvec <- kvec - Q zbar with zbar = this rank's mean of z: pass 2 applies Q to the centred rows z - zbar, so that no two
// large fp32 terms cancel there (Q z and the mean part of kvec are of size |mu1| / sigma1 against their difference)
__global__ void __launch_bounds__(64) train_kq2_kernel(TrainArgs a) {
    const int j = threadIdx.x;
    const double rows_loc = a.st[a.tl.mom0];
    const double* sz = a.st + a.tl.mom1;
    double* kq = a.st + a.tl.kq;
    double acc = kq[j];
    if (rows_loc > 0.0)
        for (int i = 0; i < 64; ++i) acc -= kq[64 + j * 64 + i] * (sz[i] / rows_loc);
    kq[j] = acc;
}

// ------------------------------------------------------------------------------------------------
// backward pass 2: per pillar dz rows -> layer-0 gradients.  Only the x0 half of dz is needed per row; the hmax half
// enters through its sum over the M slots, which has a closed form per pillar:
//   dh[k] = sum_c a1_c du_c W1[c][32 + k] + M kvec'[32 + k] - Q[32 + k, :] . (sum_slots z - M zbar)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) train_back2_kernel(TrainArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const Smem s = carve(smem_f, a.g.M, false);
    const int tid = threadIdx.x, C = a.C, M = a.g.M;
    float* zb = s.extra;                              // [64] this rank's mean of z   (16-byte aligned: float4 loads)
    float* kv = zb + 64;                              // [64]
    float* dh = kv + 64;                              // [32]
    float* Qh = dh + 32;                              // [32][64] rows 32..63 of Q
    float* dus = Qh + 32 * 64;                        // [C]  a1_c du_c of the pillar
    int* ams = reinterpret_cast<int*>(dus + C);       // [C]  its arg max rows
    float* coef = reinterpret_cast<float*>(ams + C);  // [C]  a1_c
    float* G = coef + C;                              // [M + 1][33]  x0 half of the dz rows
    float* accf = G + (size_t)(M + 1) * 33;           // [8][32][10] per-thread partials at the end
    int* hist = reinterpret_cast<int*>(accf + 8 * 32 * 10);  // [M + 2] channels per winning row, then their prefix
    int* order = hist + M + 2;                         // [C] channels sorted by winning row
    load_layer0(a, s);
    const double* bn1 = a.st + a.tl.bn1;
    for (int c = tid; c < C; c += blockDim.x) coef[c] = a.g1[c] * (float)(1.0 / sqrt(bn1[C + c] + (double)a.eps));
    const double* kq = a.st + a.tl.kq;
    if (tid < 64) {
        kv[tid] = (float)kq[tid];
        const double rows_loc = a.st[a.tl.mom0];
        zb[tid] = rows_loc > 0.0 ? (float)(a.st[a.tl.mom1 + tid] / rows_loc) : 0.f;
    }
    for (int i = tid; i < 32 * 64; i += blockDim.x) Qh[i] = (float)kq[64 + 32 * 64 + i];
    const int j = tid & 31, mg = tid >> 5;  // column of the x0 half, one of 8 row / channel groups
    float db = 0.f, dg = 0.f, a0r[8];      // dbeta0[j], dgamma0[j], A0[j][:] over this thread's rows of this CTA's pillars
#pragma unroll
    for (int i = 0; i < 8; ++i) a0r[i] = 0.f;
    float q[64];  // row j of Q
#pragma unroll
    for (int i = 0; i < 64; ++i) q[i] = (float)kq[64 + j * 64 + i];
    __syncthreads();
    float w0r[8];  // row j of W0 and the layer-0 statistics of channel j (yh0 is recomputed from the decorated rows)
#pragma unroll
    for (int i = 0; i < 8; ++i) w0r[i] = s.w0[j * 8 + i];
    const float mu0 = s.mu0[j], rs0 = s.rs0[j];
    Walk w;
    walk_begin(w, a);
    // (du, arg max) of channels tid and tid + 256 of the next pillar
    float du0 = 0.f, du1 = 0.f, dn0 = 0.f, dn1 = 0.f;
    int am0 = 0, am1 = 0, an0 = 0, an1 = 0;
    auto fetch_route = [&](const int4 d, float& x0, float& x1, int& m0, int& m1) {
        x0 = x1 = 0.f; m0 = m1 = 0;
        if (!((d.w >> 30) & 1)) return;
        const size_t ro = ((size_t)d.x * a.g.Vmax + d.y) * C;
        if (tid < C) { x0 = a.du[ro + tid]; m0 = a.amax[ro + tid]; }
        if (tid + 256 < C) { x1 = a.du[ro + tid + 256]; m1 = a.amax[ro + tid + 256]; }
    };
    if (w.i < w.count) fetch_route(w.d0, du0, du1, am0, am1);
    for (; w.i < w.count; walk_next(w), du0 = dn0, du1 = dn1, am0 = an0, am1 = an1) {
        walk_prefetch(w, a);
        if (w.i + w.step < w.count) fetch_route(w.d1, dn0, dn1, an0, an1);
        const Pillar p = unpack(a, w.d0);
        if (tid < C) { dus[tid] = coef[tid] * du0; ams[tid] = am0; }
        if (tid + 256 < C) { dus[tid + 256] = coef[tid + 256] * du1; ams[tid + 256] = am1; }
        decorate(a, p, slots_of(a, w.d0), w.q0, s);
        const int rows = layer0_rows<false>(a, p, s);
        // The pillar's channels sorted by their winning row (counting sort; shared-memory float atomics are CAS loops, the
        // integer ones are native): row m then sums its own list, G[m][:32] = sum_{c: m*_c = m} a1_c du_c W1[c][:32].
        for (int i = tid; i <= rows; i += blockDim.x) hist[i] = 0;
        if (tid < 32) dh[tid] = 0.f;
        __syncthreads();
        int pos0 = -1, pos1 = -1;
        if (p.own) {
            if (tid < C && dus[tid] != 0.f) pos0 = atomicAdd(&hist[ams[tid]], 1);
            if (tid + 256 < C && dus[tid + 256] != 0.f) pos1 = atomicAdd(&hist[ams[tid + 256]], 1);
        }
        __syncthreads();
        if (tid < 32) {  // exclusive prefix of hist[0 .. rows] (lane = a run of consecutive rows)
            const int per = (rows + 32) / 32, lo = tid * per, hi = min(lo + per, rows + 1);
            int sum = 0;
            for (int i = lo; i < hi; ++i) sum += hist[i];
            int inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (tid >= o) inc += t;
            }
            int run = inc - sum;
            for (int i = lo; i < hi; ++i) { const int h = hist[i]; hist[i] = run; run += h; }
        }
        __syncthreads();
        if (pos0 >= 0) order[hist[ams[tid]] + pos0] = tid;
        if (pos1 >= 0) order[hist[ams[tid + 256]] + pos1] = tid + 256;
        float dhp = 0.f;  // sparse part of dh[j]: the hmax half of the sparse rows enters only through its sum
        if (p.own) {
            for (int c = mg; c < C; c += 8) {
                const float v = dus[c];
                if (v != 0.f) dhp = __fmaf_rn(v, __ldg(a.W1 + (size_t)c * 64 + 32 + j), dhp);
            }
        }
        __syncthreads();
        atomicAdd(&dh[j], dhp);
        // dz[m][j] = G[m][j] + w_m (kvec'[j] - sum_i Q[j][i] (z[m][i] - zbar[i])); row n carries all M - n padded slots
        float qh = 0.f;  // the hmax half of z is the same for every row
#pragma unroll
        for (int i = 0; i < 32; ++i) qh = __fmaf_rn(q[32 + i], s.hmax[i] - zb[32 + i], qh);
        for (int m = mg; m < rows; m += 8) {
            const float4* xr = reinterpret_cast<const float4*>(s.X0 + (size_t)m * kXS);
            const float4* zr = reinterpret_cast<const float4*>(zb);
            float acc = qh;
#pragma unroll
            for (int i4 = 0; i4 < 8; ++i4) {
                const float4 x = xr[i4], z = zr[i4];
                acc = __fmaf_rn(q[i4 * 4 + 0], x.x - z.x, acc); acc = __fmaf_rn(q[i4 * 4 + 1], x.y - z.y, acc);
                acc = __fmaf_rn(q[i4 * 4 + 2], x.z - z.z, acc); acc = __fmaf_rn(q[i4 * 4 + 3], x.w - z.w, acc);
            }
            float gs = 0.f;
            const int t1 = hist[m + 1];
            for (int t = hist[m]; t < t1; ++t) {
                const int c = order[t];
                gs = __fmaf_rn(dus[c], __ldg(a.W1 + (size_t)c * 64 + j), gs);
            }
            const float wt = (m < p.n) ? 1.f : (float)(M - p.n);
            G[(size_t)m * 33 + j] = gs + wt * (kv[j] - acc);
        }
        if (mg == 0) {  // dense part of dh[j]: M kvec'[32 + j] - Q[32 + j, :] . (sum over the slots of z - M zbar)
            const float fm = (float)M;
            float acc = 0.f;
#pragma unroll 8
            for (int i = 0; i < 32; ++i) {
                acc = __fmaf_rn(Qh[j * 64 + i], s.sx[i] - fm * zb[i], acc);
                acc = __fmaf_rn(Qh[j * 64 + 32 + i], fm * (s.hmax[i] - zb[32 + i]), acc);
            }
            atomicAdd(&dh[j], fm * kv[32 + j] - acc);
        }
        __syncthreads();
        {
            const int arg = s.am0[j];
            const float dhk = dh[j];
            for (int m = mg; m < rows; m += 8) {
                float dx = G[(size_t)m * 33 + j] + (m == arg ? dhk : 0.f);
                if (!(s.X0[(size_t)m * kXS + j] > 0.f)) dx = 0.f;
                db += dx;
                float yh = -mu0 * rs0;  // a padded slot: y0 = 0
                if (m < p.n) {
                    const float4 dl = reinterpret_cast<const float4*>(s.D + (size_t)m * 8)[0];
                    const float4 dhi = reinterpret_cast<const float4*>(s.D + (size_t)m * 8)[1];
                    float y = w0r[0] * dl.x;
                    y = __fmaf_rn(w0r[1], dl.y, y); y = __fmaf_rn(w0r[2], dl.z, y); y = __fmaf_rn(w0r[3], dl.w, y);
                    y = __fmaf_rn(w0r[4], dhi.x, y); y = __fmaf_rn(w0r[5], dhi.y, y); y = __fmaf_rn(w0r[6], dhi.z, y);
                    y = __fmaf_rn(w0r[7], dhi.w, y);
                    yh = (y - mu0) * rs0;
                    a0r[0] = __fmaf_rn(dx, dl.x, a0r[0]); a0r[1] = __fmaf_rn(dx, dl.y, a0r[1]);
                    a0r[2] = __fmaf_rn(dx, dl.z, a0r[2]); a0r[3] = __fmaf_rn(dx, dl.w, a0r[3]);
                    a0r[4] = __fmaf_rn(dx, dhi.x, a0r[4]); a0r[5] = __fmaf_rn(dx, dhi.y, a0r[5]);
                    a0r[6] = __fmaf_rn(dx, dhi.z, a0r[6]); a0r[7] = __fmaf_rn(dx, dhi.w, a0r[7]);
                }
                dg = __fmaf_rn(dx, yh, dg);
            }
        }
        __syncthreads();
    }
    accf[(mg * 32 + j) * 10 + 0] = db;
    accf[(mg * 32 + j) * 10 + 1] = dg;
#pragma unroll
    for (int i = 0; i < 8; ++i) accf[(mg * 32 + j) * 10 + 2 + i] = a0r[i];
    __syncthreads();
    for (int e = tid; e < 320; e += blockDim.x) {  // e = column * 10 + field: merge the 8 row groups in float64
        double t = 0.0;
        for (int g8 = 0; g8 < 8; ++g8) t += (double)accf[(g8 * 32 + e / 10) * 10 + e % 10];
        const int k = e / 10, f = e % 10;
        if (f == 0) atomicAdd(a.st + a.tl.back0 + k, t);
        else if (f == 1) atomicAdd(a.st + a.tl.back0 + 32 + k, t);
        else atomicAdd(a.st + a.tl.A0 + k * 8 + (f - 2), t);
    }
}

// ------------------------------------------------------------------------------------------------
// parameter gradients from the accumulators and the stored moments
//   dW[c][j] = a_c (A[c][j] - (dbeta_c / R) s[j] - (dgamma_c / R) rstd_c (sum_i W[c][i] Min[i][j] - mu_c s[j]))
// ------------------------------------------------------------------------------------------------
__global__ void train_grads_kernel(const float* __restrict__ W, const float* __restrict__ gamma, int C, int K, float eps,
                                   const double* __restrict__ bn, const double* __restrict__ sums, const double* __restrict__ s,
                                   const double* __restrict__ Min, const double* __restrict__ A, const double* __restrict__ back,
                                   const double* __restrict__ backg, float* __restrict__ dW, float* __restrict__ dgamma,
                                   float* __restrict__ dbeta) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= C * K) return;
    const int c = e / K, j = e - c * K;
    const double rows = sums[2 * C];
    const double ir = rows > 0.0 ? 1.0 / rows : 0.0;
    const double rs = 1.0 / sqrt(bn[C + c] + (double)eps);
    const double ac = (double)gamma[c] * rs;
    double wm = 0.0;
    for (int i = 0; i < K; ++i) wm += (double)W[(size_t)c * K + i] * Min[i * K + j];
    const double v = ac * (A[(size_t)c * K + j] - backg[c] * ir * s[j] - backg[C + c] * ir * rs * (wm - bn[c] * s[j]));
    dW[e] = (float)v;
    if (j == 0) {
        dbeta[c] = (float)back[c];
        dgamma[c] = (float)back[C + c];
    }
}

int check_channels(int C) {
    if (C < 1 || C > kTrainMaxC) return fail(P3P_ERR_UNSUPPORTED, "training kernels cover 1..%d channels, got %d", kTrainMaxC, C);
    return P3P_OK;
}

int fill_args(TrainArgs* a, const p3p_grid* grid, int B, int64_t total, const p3p_pfn_params* p, double* state, void* ws, size_t ws_bytes) {
    if (!grid || !p || !state) return fail(P3P_ERR_INVALID_ARGUMENT, "null grid, params or state");
    if (!p->linear0_weight || !p->norm0_weight || !p->norm0_bias || !p->linear1_weight || !p->norm1_weight || !p->norm1_bias)
        return fail(P3P_ERR_INVALID_ARGUMENT, "null weight pointer");
    int rc = check_channels(p->channels);
    if (rc) return rc;
    memset(a, 0, sizeof(*a));
    rc = make_grid(grid, &a->g);
    if (rc) return rc;
    if (a->g.M > kTrainMaxM) return fail(P3P_ERR_UNSUPPORTED, "training kernels cover max_points <= %d, got %d", kTrainMaxM, a->g.M);
    const size_t need = train_smem(a->g.M, p->channels).max_block, cap = device_smem_optin();
    if (need > cap)
        return fail(P3P_ERR_UNSUPPORTED, "training kernels need %zu bytes of shared memory per CTA at max_points %d, channels %d; "
                    "the device allows %zu", need, a->g.M, p->channels, cap);
    if (B < 0 || (int64_t)B * a->g.Vmax > 0x7fffffff) return fail(P3P_ERR_INVALID_ARGUMENT, "num_tiles %d", B);
    if (ws) {
        WsLayout l;
        rc = make_ws_layout(a->g, B, total, &l);
        if (rc) return rc;
        if (ws_bytes < l.total_bytes) return fail(P3P_ERR_WORKSPACE, "workspace needs %zu bytes, got %zu", l.total_bytes, ws_bytes);
        a->ws = ws_ptrs(ws, l);
    }
    a->B = B;
    a->C = p->channels;
    a->alias = p->center_alias;
    a->eps = p->eps;
    a->W0 = p->linear0_weight; a->g0 = p->norm0_weight; a->b0 = p->norm0_bias;
    a->W1 = p->linear1_weight; a->g1 = p->norm1_weight; a->b1 = p->norm1_bias;
    a->st = state;
    a->tl = make_train_layout(p->channels);
    return P3P_OK;
}

// (fill_args has checked every size against the device's opt-in limit)
template <typename K>
int opt_in(K kernel, size_t smem) {
    P3P_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return P3P_OK;
}

int grid_size(int B, int Vmax, int per_sm) {
    const int64_t items = (int64_t)B * Vmax;
    const int64_t cap = (int64_t)device_sm_count() * per_sm;
    return (int)(items < cap ? (items > 0 ? items : 1) : cap);
}

}  // namespace
}  // namespace p3p

using namespace p3p;

extern "C" {

int64_t p3p_pfn_train_state_doubles(int32_t channels, int64_t* offsets) {
    if (check_channels(channels)) return 0;
    const TrainLayout l = make_train_layout(channels);
    if (offsets) {
        const int64_t o[14] = {l.mom0, l.sums0, l.bn0, l.mom1, l.sums1, l.bn1, l.cen, l.back1, l.back1g, l.A1, l.kq, l.back0, l.back0g, l.A0};
        for (int i = 0; i < 14; ++i) offsets[i] = o[i];
    }
    return l.total;
}

size_t p3p_pfn_train_route_bytes(const p3p_grid* grid, int32_t num_tiles, int32_t channels) {
    if (!grid || num_tiles < 0 || channels < 1) return 0;
    const size_t n = (size_t)num_tiles * (size_t)grid->max_voxels * (size_t)channels;
    return (n * 4 + 255) / 256 * 256 + n * 2;
}

int p3p_pfn_train_stats0(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                         double* state, void* workspace, size_t workspace_bytes, void* stream) {
    TrainArgs a;
    int rc = fill_args(&a, grid, num_tiles, total_points, params, state, workspace, workspace_bytes);
    if (rc) return rc;
    if (!workspace) return fail(P3P_ERR_INVALID_ARGUMENT, "workspace is null");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    P3P_CUDA_CHECK(cudaMemsetAsync(state, 0, (size_t)a.tl.total * sizeof(double), st));
    const size_t smem = train_smem(a.g.M, a.C).stats0;
    rc = opt_in(train_stats0_kernel, smem);
    if (rc) return rc;
    if (num_tiles > 0) {
        train_list_kernel<<<(num_tiles * a.g.Vmax + 255) / 256, 256, 0, st>>>(a);
        train_stats0_kernel<<<grid_size(num_tiles, a.g.Vmax, 4), 256, smem, st>>>(a);
    }
    const double* mom = state + a.tl.mom0;
    train_sums_kernel<<<32, 64, 0, st>>>(a.W0, 32, 8, mom + 1, mom + 9, mom, state + a.tl.sums0);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int p3p_pfn_train_stats1(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                         double* state, void* workspace, size_t workspace_bytes, void* stream) {
    TrainArgs a;
    int rc = fill_args(&a, grid, num_tiles, total_points, params, state, workspace, workspace_bytes);
    if (rc) return rc;
    if (!workspace) return fail(P3P_ERR_INVALID_ARGUMENT, "workspace is null");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    train_bn_kernel<<<1, 32, 0, st>>>(state + a.tl.sums0, 32, state + a.tl.bn0, nullptr, nullptr);
    const TrainSmem sm = train_smem(a.g.M, a.C);
    rc = opt_in(train_stats1_kernel, sm.stats1);
    if (rc) return rc;
    rc = opt_in(train_centre_kernel, sm.centre);
    if (rc) return rc;
    if (num_tiles > 0) {
        train_centre_kernel<<<kCentreCtas, 256, sm.centre, st>>>(a);
        train_stats1_kernel<<<grid_size(num_tiles, a.g.Vmax, 3), 256, sm.stats1, st>>>(a);
        train_uncentre_kernel<<<1, 1024, 0, st>>>(a);
    }
    const double* mom = state + a.tl.mom1;
    train_sums_kernel<<<a.C, 64, 0, st>>>(a.W1, a.C, 64, mom, mom + 64, state + a.tl.mom0, state + a.tl.sums1);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int p3p_pfn_train_stats2(const p3p_pfn_params* params, double* state, float* mean0, float* var0, float* mean1, float* var1,
                         void* stream) {
    if (!params || !state || !mean0 || !var0 || !mean1 || !var1) return fail(P3P_ERR_INVALID_ARGUMENT, "null pointer");
    const int rc = check_channels(params->channels);
    if (rc) return rc;
    const TrainLayout l = make_train_layout(params->channels);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    train_bn_kernel<<<1, 32, 0, st>>>(state + l.sums0, 32, state + l.bn0, mean0, var0);
    train_bn_kernel<<<(l.C + 127) / 128, 128, 0, st>>>(state + l.sums1, l.C, state + l.bn1, mean1, var1);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

static void set_route(TrainArgs* a, void* route, int num_tiles) {
    const size_t n = (size_t)num_tiles * a->g.Vmax * a->C;
    a->du = static_cast<float*>(route);
    a->amax = reinterpret_cast<uint16_t*>(static_cast<char*>(route) + (n * 4 + 255) / 256 * 256);
}

int p3p_pfn_train_forward(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params,
                          double* state, float* out, void* route, void* workspace, size_t workspace_bytes, void* stream) {
    TrainArgs a;
    int rc = fill_args(&a, grid, num_tiles, total_points, params, state, workspace, workspace_bytes);
    if (rc) return rc;
    if (!workspace || !out || !route) return fail(P3P_ERR_INVALID_ARGUMENT, "null workspace, out or route");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    set_route(&a, route, num_tiles);
    a.out = out;
    train_bn_kernel<<<(a.C + 127) / 128, 128, 0, st>>>(state + a.tl.sums1, a.C, state + a.tl.bn1, nullptr, nullptr);
    P3P_CUDA_CHECK(cudaMemsetAsync(out, 0, (size_t)num_tiles * a.g.ny * a.g.nx * a.C * sizeof(float), st));  // empty cells
    const int threads = a.C <= 256 ? 256 : (a.C + 31) / 32 * 32;
    const size_t smem = train_smem(a.g.M, a.C).forward;
    rc = opt_in(train_forward_kernel, smem);
    if (rc) return rc;
    if (num_tiles > 0) train_forward_kernel<<<grid_size(num_tiles, a.g.Vmax, 1), threads, smem, st>>>(a);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int p3p_pfn_backward1(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params, double* state,
                      const float* grad_out, const float* out, void* route, void* workspace, size_t workspace_bytes, void* stream) {
    TrainArgs a;
    int rc = fill_args(&a, grid, num_tiles, total_points, params, state, workspace, workspace_bytes);
    if (rc) return rc;
    if (!workspace || !grad_out || !out || !route) return fail(P3P_ERR_INVALID_ARGUMENT, "null workspace, grad_out, out or route");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    set_route(&a, route, num_tiles);
    a.gout = grad_out;
    a.out = const_cast<float*>(out);
    const size_t zero_from = (size_t)a.tl.back1, zero_to = (size_t)a.tl.total;  // every backward accumulator
    P3P_CUDA_CHECK(cudaMemsetAsync(state + zero_from, 0, (zero_to - zero_from) * sizeof(double), st));
    const int threads = a.C <= 256 ? 256 : (a.C + 31) / 32 * 32;
    const size_t smem = train_smem(a.g.M, a.C).back1;
    rc = opt_in(train_back1_kernel, smem);
    if (rc) return rc;
    if (num_tiles > 0) train_back1_kernel<<<grid_size(num_tiles, a.g.Vmax, 1), threads, smem, st>>>(a);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int p3p_pfn_backward2(const p3p_grid* grid, int32_t num_tiles, int64_t total_points, const p3p_pfn_params* params, double* state,
                      const void* route, void* workspace, size_t workspace_bytes, void* stream) {
    TrainArgs a;
    int rc = fill_args(&a, grid, num_tiles, total_points, params, state, workspace, workspace_bytes);
    if (rc) return rc;
    if (!workspace || !route) return fail(P3P_ERR_INVALID_ARGUMENT, "null workspace or route");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    set_route(&a, const_cast<void*>(route), num_tiles);
    train_kq_kernel<<<65, 64, (size_t)a.C * sizeof(double), st>>>(a);
    train_kq2_kernel<<<1, 64, 0, st>>>(a);
    const size_t smem = train_smem(a.g.M, a.C).back2;
    rc = opt_in(train_back2_kernel, smem);
    if (rc) return rc;
    if (num_tiles > 0) train_back2_kernel<<<grid_size(num_tiles, a.g.Vmax, 2), 256, smem, st>>>(a);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

int p3p_pfn_backward3(const p3p_pfn_params* params, const double* state, float* d_linear0, float* d_norm0_weight,
                      float* d_norm0_bias, float* d_linear1, float* d_norm1_weight, float* d_norm1_bias, void* stream) {
    if (!params || !state || !d_linear0 || !d_norm0_weight || !d_norm0_bias || !d_linear1 || !d_norm1_weight || !d_norm1_bias)
        return fail(P3P_ERR_INVALID_ARGUMENT, "null pointer");
    const int rc = check_channels(params->channels);
    if (rc) return rc;
    const TrainLayout l = make_train_layout(params->channels);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const double* m0 = state + l.mom0;
    const double* m1 = state + l.mom1;
    train_grads_kernel<<<1, 256, 0, st>>>(params->linear0_weight, params->norm0_weight, 32, 8, params->eps, state + l.bn0, state + l.sums0,
                                          m0 + 1, m0 + 9, state + l.A0, state + l.back0, state + l.back0g, d_linear0, d_norm0_weight,
                                          d_norm0_bias);
    train_grads_kernel<<<(l.C * 64 + 255) / 256, 256, 0, st>>>(params->linear1_weight, params->norm1_weight, l.C, 64, params->eps,
                                                               state + l.bn1, state + l.sums1, m1, m1 + 64, state + l.A1, state + l.back1,
                                                               state + l.back1g, d_linear1, d_norm1_weight, d_norm1_bias);
    P3P_CUDA_CHECK(cudaGetLastError());
    return P3P_OK;
}

}  // extern "C"
