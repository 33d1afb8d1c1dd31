// common.cuh — shared device helpers for libtrb_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/trb.h"

#ifndef __CUDA_ARCH__
#define TRB_HOST_PASS 1
#endif

namespace trb {

constexpr int kThreads = 256;          // threads per CTA for the reduction kernels
constexpr int kWarps = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;

void set_error(const char *fmt, ...);
int check_cuda(cudaError_t e, const char *what);
// SM count of the current device, queried once per device.  Returns TRB_OK, or the CUDA error with trb_last_error() set.
int sm_count(int &n);
// The longest spatial axis the 1.5*2^23 floor / rint below (floor_frac, round_idx, and kMagic in the TMA-staged
// kernels) can index: TRB_ERR_UNSUPPORTED, with trb_last_error() naming the limit, when an axis of (D,) H, W is longer.
// Every entry point whose kernels index a volume through them calls it.
constexpr int kMaxFastFloorAxis = 1 << 22;
int check_fast_floor_axes(int ndim, int D, int H, int W);
// The shape rules of every call that samples a flow-layout field (flow.cu, transform.cu): ndim 2 or 3, every spatial
// axis >= 2, D*H*W < 2^31 (TRB_ERR_ARG), and check_fast_floor_axes.  2-D callers pass any D: it is not read.
int validate_flow(int ndim, int D, int H, int W);
// Grid of the one-thread-per-voxel flow kernels (for_each_voxel): enough CTAs for every SM to hold 8, at most
// kFlowMaxBlocks (the partial rows of the flow workspace, trb_flow_workspace_bytes).
constexpr int kFlowMaxBlocks = 2048;
int flow_grid(size_t vol, unsigned &grid);

// ---- loads ---------------------------------------------------------------
__device__ __forceinline__ float ldg_f(const float *p) { return __ldg(p); }

// streaming (read-once) load: keep it out of L1 so the gathered volume owns the cache
__device__ __forceinline__ float ld_stream_f(const float *p)
{
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ---- fixed-order (deterministic) block and grid reductions of fp64 sums, for 256-thread CTAs ----------------------
// Every sum is formed in the same order on every run: the warp_sum shuffle tree, then warps 0..7 in order, then the
// blocks in index order.  The caller declares the shared rows, so each kernel's footprint stays visible.

// Block total of each entry: thread i < N returns the total of v[i] (fp32 inputs are widened first), others 0.
template <int N, typename T>
__device__ __forceinline__ double block_sum(const T (&v)[N], double (&sh)[kWarps][N])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const double s = warp_sum((double)v[i]);
        if (lane == 0) sh[warp][i] = s;
    }
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x < N) {
#pragma unroll
        for (int w = 0; w < kWarps; ++w) t += sh[w][threadIdx.x];
    }
    return t;
}

// The same order, but every thread gets all N totals in v.  Starts with a barrier, so consecutive calls can share sh
// (any M >= N columns).
template <int N, int M>
__device__ __forceinline__ void block_sum_all(double (&v)[N], double (&sh)[kWarps][M])
{
    static_assert(N <= M, "shared rows too short");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = warp_sum(v[i]);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < N; ++i) sh[warp][i] = v[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < N; ++i) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) t += sh[w][i];
        v[i] = t;
    }
}
template <int M>
__device__ __forceinline__ double block_sum_all(double v, double (&sh)[kWarps][M])
{
    double a[1] = {v};
    block_sum_all(a, sh);
    return a[0];
}

// Called by every thread of a block after it has stored its share of a grid-wide result.  True, in every thread, for
// the block that arrives last of `expected`; that block then sees what the others stored.  The fences pair the others'
// stores with this block's loads; the caller re-arms the ticket (*ticket = 0) once it is done.
__device__ __forceinline__ bool last_to_arrive(unsigned *ticket, unsigned expected)
{
    __threadfence();
    __syncthreads();
    int last = 0;
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == expected - 1;
    last = __syncthreads_or(last);
    if (last) __threadfence();
    return last;
}

// One warp: sum over blocks 0..n_blocks-1 of part[b * stride + k], lane l taking blocks l, l+32, ... then warp_sum.
__device__ __forceinline__ double fold_blocks(const double *part, int n_blocks, size_t stride, int k)
{
    double t = 0.0;
    for (int b = threadIdx.x & 31; b < n_blocks; b += 32) t += __ldcg(part + (size_t)b * stride + k);
    return warp_sum(t);
}

// Grid total of each entry: the block totals go to partials[block][N], and the last block to arrive adds them in block
// order into sh[0][0..N) and re-arms the ticket.  Returns true in every thread of that block (sh is then ready), false
// in the others.
template <int N, typename T>
__device__ __forceinline__ bool grid_sum(const T (&v)[N], double (&sh)[kWarps][N], double *partials, unsigned *ticket)
{
    const double t = block_sum(v, sh);
    if (threadIdx.x < N) __stcg(partials + (size_t)blockIdx.x * N + threadIdx.x, t);
    if (!last_to_arrive(ticket, gridDim.x)) return false;
    const int warp = threadIdx.x >> 5;
    for (int i = warp; i < N; i += kWarps) {
        const double s = fold_blocks(partials, gridDim.x, N, i);
        if ((threadIdx.x & 31) == 0) sh[0][i] = s;
    }
    if (threadIdx.x == 0) *ticket = 0u;
    __syncthreads();
    return true;
}

// Row-wise voxel loop: a 256-thread CTA takes two rows (z,y) at a time, 128 threads along x each, so the only
// integer division is one 32-bit div per row (the per-voxel 64-bit idx % W, idx / W of the first version cost
// more than the whole interpolation).  f(idx, x, y, z).
template <int UNROLL = 1, typename F>
__device__ __forceinline__ void for_each_voxel(int D, int H, int W, F f)
{
    const int rows = D * H;
    const int rx = threadIdx.x & 127, ry = threadIdx.x >> 7;
    for (int row = 2 * blockIdx.x + ry; row < rows; row += 2 * gridDim.x) {
        const int z = row / H, y = row - z * H;
        const size_t base = (size_t)row * W;
        // UNROLL 2 keeps two voxels in flight per thread: pays for the light warp kernels (+15 %), costs the
        // statistics / gradient kernels 20 registers and occupancy (-12 %)
#pragma unroll(UNROLL)
        for (int x = rx; x < W; x += 128) f(base + x, x, y, z);
    }
}

// ---- flow sample positions and zero-padded (tri|bi)linear sampling (flow.cu, flow_direct.cu) ----------------
// The reference normalises voxel position + flow to [-1,1] (utils.py:354-356) and grid_sample(align_corners=True)
// un-normalises again; the fp32 round trip is kept op for op.  Its IEEE division by the loop-invariant S-1 is done
// with the hoisted correctly rounded reciprocal: q0 = RN(a*r), q = RN(q0 + (a - d*q0)*r) is the correctly rounded
// quotient (Markstein), 3 instructions instead of the ~14 of the generic division sequence.
struct AxisMap {
    float d, r;      // S-1 and RN(1/(S-1))
};
__device__ __forceinline__ AxisMap axis_map(int S)
{
    AxisMap a;
    a.d = (float)(S - 1);
    a.r = __frcp_rn(a.d);
    return a;
}
__device__ __forceinline__ float flow_pos(const AxisMap &m, int i, float f)
{
    const float loc = (float)i + f;
    const float q0 = __fmul_rn(loc, m.r);
    const float q = __fmaf_rn(__fmaf_rn(-m.d, q0, loc), m.r, q0);
    const float nrm = 2.f * (q - 0.5f);
    return __fmul_rn(__fmul_rn(__fadd_rn(nrm, 1.f), 0.5f), m.d);
}

// The same round trip as torch evaluates it on a CUDA device: there a division by a Python scalar is a multiply by the
// scalar's fp32 reciprocal (PyTorch's div_true_kernel_cuda), which differs from the IEEE quotient in the last bit for some
// positions.  A bilinear sample moves by ~1e-7 of a voxel with that bit; a nearest sample can flip at an exact half-voxel
// position, so the nearest flow warp follows the device's grid.
__device__ __forceinline__ float flow_pos_rcp(const AxisMap &m, int i, float f)
{
    const float loc = (float)i + f;
    const float nrm = 2.f * (__fmul_rn(loc, m.r) - 0.5f);
    return __fmul_rn(__fmul_rn(__fadd_rn(nrm, 1.f), 0.5f), m.d);
}

// floor and fraction without the quarter-rate conversion pipe: adding 1.5*2^23 rounding down leaves floor(p) in the
// low mantissa bits, exactly for |p| <= 2^22.  Further out the sum's spacing differs from 1 and the index is wrong, but it
// is >= 2^22 or < -2^22 (inf and NaN included), so with every axis at most 2^22 voxels long (kMaxFastFloorAxis; hosts
// refuse longer ones) such a position still lands on the zero padding.  On a longer axis it would read a wrong voxel
// inside the volume: p = 4195304.25 gives index 4194804.
__device__ __forceinline__ void floor_frac(float p, int &i0, float &t, float &fl)
{
    const float m = __fadd_rd(p, 12582912.f);
    i0 = __float_as_int(m) - 0x4B400000;
    fl = m - 12582912.f;
    t = p - fl;
}
__device__ __forceinline__ void floor_frac(float p, int &i0, float &t)
{
    float fl;
    floor_frac(p, i0, t, fl);
}

// grid_sample(mode='nearest')'s source index: p rounded half to even, as torch's nearbyint does.  The same 1.5*2^23 add
// as floor_frac, in round-to-nearest mode, rather than __float2int_rn: the conversion maps NaN to index 0, a voxel of
// every volume, where torch samples the zero padding.  Exact for |p| < 2^22; anything further out, inf and NaN included,
// lands on an index >= 2^22 or < -2^22: the zero padding of any axis of at most kMaxFastFloorAxis voxels (see floor_frac).
__device__ __forceinline__ int round_idx(float p)
{
    return __float_as_int(__fadd_rn(p, 12582912.f)) - 0x4B400000;
}

// The voxel grid_sample(mode='nearest', padding_mode='zeros') reads at (px,py,pz): its linear offset (64-bit), and
// false when it lies in the zero padding.  2-D: D = 1, pz = 0.
__device__ __forceinline__ bool nearest_offset(int D, int H, int W, float px, float py, float pz, long long &o)
{
    const int x = round_idx(px), y = round_idx(py), z = round_idx(pz);
    o = ((long long)z * H + y) * W + x;
    return (unsigned)x < (unsigned)W && (unsigned)y < (unsigned)H && (unsigned)z < (unsigned)D;
}

// the 8 corners of the cell with origin (x0,y0,z0), zero outside the volume: predicated loads, 64-bit offsets
__device__ __forceinline__ void load_cell3(const float *__restrict__ m, int D, int H, int W, int x0, int y0, int z0,
                                           float (&c)[8])
{
    const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)(x0 + 1) < (unsigned)W;
    const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
    const bool vz0 = (unsigned)z0 < (unsigned)D, vz1 = (unsigned)(z0 + 1) < (unsigned)D;
    const long long HW = (long long)H * W;
    const float *q = m + (((long long)z0 * H + y0) * W + x0);
    c[0] = (vz0 & vy0 & vx0) ? __ldg(q) : 0.f;
    c[1] = (vz0 & vy0 & vx1) ? __ldg(q + 1) : 0.f;
    c[2] = (vz0 & vy1 & vx0) ? __ldg(q + W) : 0.f;
    c[3] = (vz0 & vy1 & vx1) ? __ldg(q + W + 1) : 0.f;
    c[4] = (vz1 & vy0 & vx0) ? __ldg(q + HW) : 0.f;
    c[5] = (vz1 & vy0 & vx1) ? __ldg(q + HW + 1) : 0.f;
    c[6] = (vz1 & vy1 & vx0) ? __ldg(q + HW + W) : 0.f;
    c[7] = (vz1 & vy1 & vx1) ? __ldg(q + HW + W + 1) : 0.f;
}
// cells that straddle the volume boundary (rare: kept out of line so the common path stays small)
static __device__ __noinline__ void gather_border3(const float *__restrict__ m, int D, int H, int W, int x0, int y0, int z0,
                                                   float (&c)[8])
{
    load_cell3(m, D, H, W, x0, y0, z0, c);
}
// the 2-D twin: the 4 corners of the cell with origin (x0,y0)
__device__ __forceinline__ void load_cell2(const float *__restrict__ m, int H, int W, int x0, int y0, float (&c)[4])
{
    const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)(x0 + 1) < (unsigned)W;
    const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
    const float *q = m + ((long long)y0 * W + x0);
    c[0] = (vy0 & vx0) ? __ldg(q) : 0.f;
    c[1] = (vy0 & vx1) ? __ldg(q + 1) : 0.f;
    c[2] = (vy1 & vx0) ? __ldg(q + W) : 0.f;
    c[3] = (vy1 & vx1) ? __ldg(q + W + 1) : 0.f;
}

template <int NDIM>
struct Sample {
    float val;
    float g[NDIM];      // d val / d (x, y[, z]) in voxel units
};

// The 8 corners of the cell around (px,py,pz) + the fractions: the loads can be issued early and blended later.
struct Cell3 {
    float c[8];
    float tx, ty, tz;
    float fx, fy, fz;       // floor of the position (the cell's origin), for sample_near
};
// BRANCH_FREE: predicated loads, no control flow — the compiler can overlap the gathers of neighbouring voxels and
// phases (what latency-bound kernels want: warp_flow -22 %, fused direct-flow epoch -10 %); otherwise interior cells
// take an unpredicated fast path and boundary cells an out-of-line one (fewer instructions: flow node -11 %).
template <bool BRANCH_FREE = true>
__device__ __forceinline__ Cell3 gather_cell3(const float *__restrict__ m, int D, int H, int W, float px, float py, float pz)
{
    Cell3 k;
    int x0, y0, z0;
    floor_frac(px, x0, k.tx, k.fx);
    floor_frac(py, y0, k.ty, k.fy);
    floor_frac(pz, z0, k.tz, k.fz);
    if constexpr (BRANCH_FREE) {
        const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)(x0 + 1) < (unsigned)W;
        const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
        const bool vz0 = (unsigned)z0 < (unsigned)D, vz1 = (unsigned)(z0 + 1) < (unsigned)D;
        const int HW = H * W;
        const float *q = m + ((z0 * H + y0) * W + x0);
        k.c[0] = (vz0 & vy0 & vx0) ? __ldg(q) : 0.f;
        k.c[1] = (vz0 & vy0 & vx1) ? __ldg(q + 1) : 0.f;
        k.c[2] = (vz0 & vy1 & vx0) ? __ldg(q + W) : 0.f;
        k.c[3] = (vz0 & vy1 & vx1) ? __ldg(q + W + 1) : 0.f;
        k.c[4] = (vz1 & vy0 & vx0) ? __ldg(q + HW) : 0.f;
        k.c[5] = (vz1 & vy0 & vx1) ? __ldg(q + HW + 1) : 0.f;
        k.c[6] = (vz1 & vy1 & vx0) ? __ldg(q + HW + W) : 0.f;
        k.c[7] = (vz1 & vy1 & vx1) ? __ldg(q + HW + W + 1) : 0.f;
        return k;
    }
    if ((unsigned)x0 < (unsigned)(W - 1) && (unsigned)y0 < (unsigned)(H - 1) && (unsigned)z0 < (unsigned)(D - 1)) {
        const float *q = m + ((z0 * H + y0) * W + x0);          // the whole cell is inside: no predicates
        k.c[0] = __ldg(q); k.c[1] = __ldg(q + 1); k.c[2] = __ldg(q + W); k.c[3] = __ldg(q + W + 1);
        q += H * W;
        k.c[4] = __ldg(q); k.c[5] = __ldg(q + 1); k.c[6] = __ldg(q + W); k.c[7] = __ldg(q + W + 1);
    } else {
        float b[8];                                             // only this rare path touches local memory
        gather_border3(m, D, H, W, x0, y0, z0, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) k.c[i] = b[i];
    }
    return k;
}
template <bool WANT_GRAD>
__device__ __forceinline__ Sample<3> blend_cell3(const Cell3 &k)
{
    Sample<3> s;
    const float d00 = k.c[1] - k.c[0], d01 = k.c[3] - k.c[2], d10 = k.c[5] - k.c[4], d11 = k.c[7] - k.c[6];
    const float v00 = fmaf(k.tx, d00, k.c[0]), v01 = fmaf(k.tx, d01, k.c[2]);
    const float v10 = fmaf(k.tx, d10, k.c[4]), v11 = fmaf(k.tx, d11, k.c[6]);
    const float e0 = v01 - v00, e1 = v11 - v10;
    const float w0 = fmaf(k.ty, e0, v00), w1 = fmaf(k.ty, e1, v10);
    const float gz = w1 - w0;
    s.val = fmaf(k.tz, gz, w0);
    if (WANT_GRAD) {
        s.g[2] = gz;
        s.g[1] = fmaf(k.tz, e1 - e0, e0);
        const float dx0 = fmaf(k.ty, d01 - d00, d00), dx1 = fmaf(k.ty, d11 - d10, d10);
        s.g[0] = fmaf(k.tz, dx1 - dx0, dx0);
    }
    return s;
}

// the 2-D twin: corners (c00, c01, c10, c11) with x fastest, and the fractions
struct Cell2 {
    float c[4];
    float tx, ty;
};
template <bool WANT_GRAD>
__device__ __forceinline__ Sample<2> blend_cell2(const Cell2 &k)
{
    Sample<2> s;
    const float d0 = k.c[1] - k.c[0], d1 = k.c[3] - k.c[2];
    const float v0 = fmaf(k.tx, d0, k.c[0]), v1 = fmaf(k.tx, d1, k.c[2]);
    const float gy = v1 - v0;
    s.val = fmaf(k.ty, gy, v0);
    if (WANT_GRAD) {
        s.g[1] = gy;
        s.g[0] = fmaf(k.ty, d1 - d0, d0);
    }
    return s;
}

// Value at a second position that usually lies in the cell already gathered (a gradient step moves a sample by a
// fraction of a voxel): same corners, new fractions — bit-identical to a fresh gather, without its 8 loads.
__device__ __forceinline__ float sample_near(const Cell3 &k, const float *__restrict__ m, int D, int H, int W,
                                             float qx, float qy, float qz);

// grid_sample(mode='bilinear', padding_mode='zeros') at voxel coordinates (px,py,pz).  Needs D*H*W < 2^31 (hosts check).
template <int NDIM, bool WANT_GRAD, bool BRANCH_FREE = true>
__device__ __forceinline__ Sample<NDIM> sample_zero_pad(const float *__restrict__ m, int D, int H, int W,
                                                        float px, float py, float pz)
{
    if constexpr (NDIM == 3) {
        return blend_cell3<WANT_GRAD>(gather_cell3<BRANCH_FREE>(m, D, H, W, px, py, pz));
    } else {
        Cell2 k;
        int x0, y0;
        floor_frac(px, x0, k.tx);
        floor_frac(py, y0, k.ty);
        load_cell2(m, H, W, x0, y0, k.c);
        return blend_cell2<WANT_GRAD>(k);
    }
}

__device__ __forceinline__ float sample_near(const Cell3 &k, const float *__restrict__ m, int D, int H, int W,
                                             float qx, float qy, float qz)
{
    const float tx = qx - k.fx, ty = qy - k.fy, tz = qz - k.fz;
    if (tx >= 0.f && tx < 1.f && ty >= 0.f && ty < 1.f && tz >= 0.f && tz < 1.f) {
        Cell3 c2 = k;
        c2.tx = tx; c2.ty = ty; c2.tz = tz;
        return blend_cell3<false>(c2).val;
    }
    return sample_zero_pad<3, false>(m, D, H, W, qx, qy, qz).val;
}

// ---- similarity coefficients from the five global moments -------------------
// dL/dw_v = cw*w_v + ct*t_v + c0   (SURVEY.md §8 a-5; reference utils.py:197-205,
// nn.MSELoss at warpings.py:37,124; weighted sum warpings.py:78-79,144-145)
struct LossCoef {
    double loss, cw, ct, c0;
};
__device__ __forceinline__ LossCoef loss_coefficients(double n, double St, double Sw, double Stt,
                                                      double Sww, double Stw, double w_mse, double w_ncc)
{
    LossCoef o;
    double L = 0.0, gm = 0.0, ga = 0.0, gb = 0.0;
    // one reciprocal of n and one of S instead of eight divisions: this runs on the critical path between two epochs
    // of a single pair (a dependent fp64 division is ~150 cycles)
    const double inv_n = 1.0 / n;
    if (w_mse != 0.0) {
        L += w_mse * ((Stt - 2.0 * Stw + Sww) * inv_n);
        gm = 2.0 * w_mse * inv_n;
    }
    if (w_ncc != 0.0) {
        double A = Stt - St * St * inv_n, B = Sww - Sw * Sw * inv_n, C = Stw - St * Sw * inv_n;
        double S = sqrt(A * B + 1e-10);
        const double inv_S = 1.0 / S;
        L += w_ncc * 100.0 * (1.0 - C * inv_S);
        ga = -100.0 * w_ncc * inv_S;
        gb = 100.0 * w_ncc * C * A * (inv_S * inv_S * inv_S);
    }
    o.loss = L;
    o.cw = gm + gb;
    o.ct = ga - gm;
    o.c0 = -(ga * St + gb * Sw) * inv_n;
    return o;
}

}  // namespace trb
