// transform.cu — algebra of registration transforms (sm_100a): an affine result as a flow, "first, then second"
// composition with a flow second, and the inverse of a flow.
//
// Flows are the planar fp32 [ndim][D][H][W] of every flow call here, in voxel units, channel i displacing spatial axis i
// ((z, y, x) in 3-D, (y, x) in 2-D); u stands for phi_u(p) = p + u(p), and warp_flow(m, u) samples m at phi_u(p).
// get_affine_warp(theta, m) samples m at T(q) = M q + c in voxel units (affine_grid(align_corners=False) un-normalised by
// grid_sample); with the sizes S_r of sampling coordinate r (0 = x/W, 1 = y/H, 2 = z/D) and theta row r sampling it:
//   M_rc = theta_rc S_r / S_c,   c_r = S_r/2 (theta_r,nd + 1 - sum_c theta_rc (1 - 1/S_c)) - 1/2.
// "first, then second" gives w with warp_flow(m, w) = warp(warp(m, first), second) up to the second interpolation:
//   first a theta:  w(p) = T(p + u(p)) - p = u + A q + c,  q = p + u,  A = M - I   (exact: T is affine)
//   first a flow f: w(p) = u(p) + f~(p + u(p))
// f~ is the bi/trilinear interpolant with border padding: each coordinate clamped to [0, S-1] before the floor (every
// axis <= 2^22, so floor_frac is exact there); the corner past S-1 then has weight 0 and load_cell3's predicate gives it 0.
// The inverse v of u is the fixed point of v(p) = -u~(p + v(p)), so that phi_u(phi_v(p)) = p.  A non-finite sample
// position gives NaN at its voxel (checked explicitly: the clamp would turn NaN into 0).
//
// Algorithmic traffic per voxel (3-D; 2-D in brackets): affine -> flow 12 B written [8]; theta first 12 read + 12 written
// [8 + 8]; flow first 12 + 12 streamed [8 + 8] plus the gathered cells of f; inverse 12 read + 12 written [8 + 8] plus the
// gathers of every iteration.
#include "common.cuh"

namespace trb {

constexpr int kInvMaxBlocks = kFlowMaxBlocks;     // partial rows in the flow workspace

__device__ __forceinline__ float nan_f() { return __int_as_float(0x7fffffff); }

// p in flow channel order: (z, y, x) or (y, x)
template <int NDIM>
__device__ __forceinline__ void voxel_pos(int x, int y, int z, float (&p)[NDIM])
{
    if constexpr (NDIM == 3) { p[0] = (float)z; p[1] = (float)y; p[2] = (float)x; }
    else { p[0] = (float)y; p[1] = (float)x; }
}

// s = f~(q) for every channel of f, q finite (channel order).  One cell origin and one set of corner predicates
// serve all channels.
template <int NDIM>
__device__ __forceinline__ void sample_border(const float *__restrict__ f, size_t vol, int D, int H, int W,
                                              const float (&q)[NDIM], float (&s)[NDIM])
{
    const auto clamp = [](float v, int S) { return fminf(fmaxf(v, 0.f), (float)(S - 1)); };
    if constexpr (NDIM == 3) {
        Cell3 k;
        int x0, y0, z0;
        floor_frac(clamp(q[2], W), x0, k.tx);
        floor_frac(clamp(q[1], H), y0, k.ty);
        floor_frac(clamp(q[0], D), z0, k.tz);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            load_cell3(f + c * vol, D, H, W, x0, y0, z0, k.c);
            s[c] = blend_cell3<false>(k).val;
        }
    } else {
        Cell2 k;
        int x0, y0;
        floor_frac(clamp(q[1], W), x0, k.tx);
        floor_frac(clamp(q[0], H), y0, k.ty);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            load_cell2(f + c * vol, H, W, x0, y0, k.c);
            s[c] = blend_cell2<false>(k).val;
        }
    }
}

// w = u + A (p + u) + c; HAS_FLOW false: u = 0, w = A p + c (the affine's own displacement).  theta is read on the
// device (Register.theta lives there): no host synchronisation.  A and c are formed once per thread in fp64.
template <int NDIM, bool HAS_FLOW>
__global__ void __launch_bounds__(256, 4) compose_affine_flow_kernel(const float *__restrict__ theta, const float *__restrict__ flow,
                                                                   float *__restrict__ out, int D, int H, int W)
{
    constexpr int NC = NDIM + 1;
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const double S[3] = {(double)W, (double)H, (double)D};          // by sampling coordinate
    float A[NDIM][NDIM], c[NDIM];                                   // by flow channel
#pragma unroll
    for (int i = 0; i < NDIM; ++i) {
        const int r = NDIM - 1 - i;
        double cr = (double)__ldg(theta + r * NC + NDIM) + 1.0;
#pragma unroll
        for (int j = 0; j < NDIM; ++j) {
            const int cc = NDIM - 1 - j;
            const double t = (double)__ldg(theta + r * NC + cc);
            cr -= t * (1.0 - 1.0 / S[cc]);
            A[i][j] = (float)(t * S[r] / S[cc] - (i == j ? 1.0 : 0.0));
        }
        c[i] = (float)(0.5 * S[r] * cr - 0.5);
    }
    for_each_voxel<2>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float q[NDIM], u[NDIM];
        voxel_pos<NDIM>(x, y, z, q);
        bool ok = true;
        if constexpr (HAS_FLOW) {
#pragma unroll
            for (int i = 0; i < NDIM; ++i) {
                u[i] = ld_stream_f(flow + i * vol + idx);
                q[i] += u[i];
                ok &= isfinite(q[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < NDIM; ++i) {
            float t = c[i];
#pragma unroll
            for (int j = 0; j < NDIM; ++j) t = fmaf(A[i][j], q[j], t);
            if constexpr (HAS_FLOW) t = ok ? u[i] + t : nan_f();
            out[i * vol + idx] = t;
        }
    });
}

// w = u + f~(p + u), u = second, f = first
template <int NDIM>
__global__ void __launch_bounds__(256, 4) compose_flows_kernel(const float *__restrict__ first, const float *__restrict__ second,
                                                             float *__restrict__ out, int D, int H, int W)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    for_each_voxel<2>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float q[NDIM], u[NDIM], s[NDIM];
        voxel_pos<NDIM>(x, y, z, q);
        bool ok = true;
#pragma unroll
        for (int i = 0; i < NDIM; ++i) {
            u[i] = ld_stream_f(second + i * vol + idx);
            q[i] += u[i];
            ok &= isfinite(q[i]);
        }
        if (!ok) {
#pragma unroll
            for (int i = 0; i < NDIM; ++i) out[i * vol + idx] = nan_f();
            return;
        }
        sample_border<NDIM>(first, vol, D, H, W, q, s);
#pragma unroll
        for (int i = 0; i < NDIM; ++i) out[i * vol + idx] = u[i] + s[i];
    });
}

// The fixed point v = -u~(p + v) per voxel, in registers: v_0 = -u(p); iteration k evaluates s = u~(p + v_k) and
// r_k = |v_k + s|_inf, stops when r_k <= tol or k = max_iter - 1, else v_{k+1} = -s.  The v_k whose residual was
// evaluated is returned.  A non-finite position or residual stops the voxel with NaN in every channel.
// Work items: 256 consecutive voxels, walked grid-stride by at most kInvMaxBlocks CTAs (a lane whose voxel converges
// idles until its warp's slowest lane is done).
// workspace (doubles): [4] ticket (as unsigned) ; [8 ..) sums[blocks][3] ; then max r [blocks]
template <int NDIM>
__global__ void __launch_bounds__(kThreads) invert_flow_kernel(const float *__restrict__ flow, float *__restrict__ inv,
                                                               int D, int H, int W, long long n_items, int max_iter,
                                                               float tol, double *__restrict__ stats, double *ws)
{
    const int HW = H * W;
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * HW;
    double acc[3] = {0.0, 0.0, 0.0};        // n not converged (finite), n non-finite, residual evaluations
    double rmax = 0.0;                      // over finite voxels
    for (long long it = blockIdx.x; it < n_items; it += gridDim.x) {
        const long long lin = it * kThreads + threadIdx.x;
        if (lin >= (long long)vol) continue;
        const int idx = (int)lin, z = idx / HW, rem = idx - z * HW, y = rem / W, x = rem - y * W;
        float p[NDIM], v[NDIM];
        voxel_pos<NDIM>(x, y, z, p);
#pragma unroll
        for (int i = 0; i < NDIM; ++i) v[i] = -__ldg(flow + i * vol + idx);
        float r = 0.f;
        int k = 0;
        bool finite = true;
        for (;;) {
            ++k;
            float q[NDIM], s[NDIM];
#pragma unroll
            for (int i = 0; i < NDIM; ++i) {
                q[i] = p[i] + v[i];
                finite &= isfinite(q[i]);
            }
            if (!finite) break;
            sample_border<NDIM>(flow, vol, D, H, W, q, s);
            r = 0.f;
#pragma unroll
            for (int i = 0; i < NDIM; ++i) {
                const float d = v[i] + s[i];
                finite &= isfinite(d);
                r = fmaxf(r, fabsf(d));
            }
            if (!finite || r <= tol || k == max_iter) break;
#pragma unroll
            for (int i = 0; i < NDIM; ++i) v[i] = -s[i];
        }
#pragma unroll
        for (int i = 0; i < NDIM; ++i) inv[i * vol + idx] = finite ? v[i] : nan_f();
        acc[2] += (double)k;
        if (finite) {
            acc[0] += r > tol ? 1.0 : 0.0;
            rmax = fmax(rmax, (double)r);
        } else {
            acc[1] += 1.0;
        }
    }
    // max r: exact in any order, per-block slots folded by the last block (as flow_jacobian_kernel)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ double mx[kWarps];
    __shared__ double red[kWarps][3];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(kFull, rmax, o));
    if (lane == 0) mx[warp] = rmax;
    __syncthreads();
    double *mx_part = ws + 8 + (size_t)gridDim.x * 3;
    if (threadIdx.x == 0) {
        for (int w = 1; w < kWarps; ++w) rmax = fmax(rmax, mx[w]);
        __stcg(mx_part + blockIdx.x, rmax);
    }
    if (!grid_sum(acc, red, ws + 8, (unsigned *)(ws + 4)) || warp != 0) return;
    rmax = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32) rmax = fmax(rmax, __ldcg(mx_part + b));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(kFull, rmax, o));
    if (lane == 0) { stats[0] = red[0][0]; stats[1] = red[0][1]; stats[2] = rmax; stats[3] = red[0][2]; }
}

// [a, a + na) and [b, b + nb) share a byte
static bool overlap(const void *a, size_t na, const void *b, size_t nb)
{
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return a && b && x < y + nb && y < x + na;
}

}  // namespace trb

using namespace trb;

extern "C" int trb_compose_affine_flow(int ndim, const float *theta_dev, const float *flow_dev, int D, int H, int W,
                                       float *out_dev, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (ndim == 2) D = 1;
    if (!theta_dev || !out_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)D * H * W, fbytes = ndim * vol * sizeof(float);
    if (overlap(out_dev, fbytes, theta_dev, ndim * (ndim + 1) * sizeof(float)) || overlap(out_dev, fbytes, flow_dev, fbytes)) {
        set_error("out must not overlap theta or the flow");
        return TRB_ERR_ARG;
    }
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) {
        if (flow_dev) compose_affine_flow_kernel<3, true><<<g, 256, 0, s>>>(theta_dev, flow_dev, out_dev, D, H, W);
        else compose_affine_flow_kernel<3, false><<<g, 256, 0, s>>>(theta_dev, nullptr, out_dev, D, H, W);
    } else {
        if (flow_dev) compose_affine_flow_kernel<2, true><<<g, 256, 0, s>>>(theta_dev, flow_dev, out_dev, 1, H, W);
        else compose_affine_flow_kernel<2, false><<<g, 256, 0, s>>>(theta_dev, nullptr, out_dev, 1, H, W);
    }
    return check_cuda(cudaGetLastError(), "compose_affine_flow");
}

extern "C" int trb_compose_flows(int ndim, const float *first_dev, const float *second_dev, int D, int H, int W,
                                 float *out_dev, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (ndim == 2) D = 1;
    if (!first_dev || !second_dev || !out_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)D * H * W, fbytes = ndim * vol * sizeof(float);
    if (overlap(out_dev, fbytes, first_dev, fbytes) || overlap(out_dev, fbytes, second_dev, fbytes)) {
        set_error("out must not overlap either input flow");
        return TRB_ERR_ARG;
    }
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) compose_flows_kernel<3><<<g, 256, 0, s>>>(first_dev, second_dev, out_dev, D, H, W);
    else compose_flows_kernel<2><<<g, 256, 0, s>>>(first_dev, second_dev, out_dev, 1, H, W);
    return check_cuda(cudaGetLastError(), "compose_flows");
}

extern "C" int trb_invert_flow(int ndim, const float *flow_dev, int D, int H, int W, int max_iter, float tol,
                               float *inv_out_dev, double *stats_out_dev, void *workspace_dev, size_t workspace_bytes,
                               void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (ndim == 2) D = 1;
    if (!flow_dev || !inv_out_dev || !stats_out_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)D * H * W, fbytes = ndim * vol * sizeof(float), sbytes = TRB_INV_NSTATS * sizeof(double);
    if (overlap(inv_out_dev, fbytes, flow_dev, fbytes) || overlap(stats_out_dev, sbytes, flow_dev, fbytes) ||
        overlap(stats_out_dev, sbytes, inv_out_dev, fbytes)) {
        set_error("the inverse and the statistics must not overlap the flow or each other");
        return TRB_ERR_ARG;
    }
    if (max_iter < 1 || max_iter > 1000) { set_error("max_iter must lie in [1, 1000] (got %d)", max_iter); return TRB_ERR_ARG; }
    if (!(tol > 0.f) || !isfinite(tol)) { set_error("tol must be finite and > 0 (got %g)", (double)tol); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_flow_workspace_bytes()) {
        set_error("workspace too small: need %zu bytes (trb_flow_workspace_bytes)", trb_flow_workspace_bytes());
        return TRB_ERR_WORKSPACE;
    }
    const long long n_items = (long long)((vol + kThreads - 1) / kThreads);
    const unsigned grid = (unsigned)(n_items < kInvMaxBlocks ? n_items : kInvMaxBlocks);
    double *ws = (double *)workspace_dev;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3)
        invert_flow_kernel<3><<<grid, kThreads, 0, s>>>(flow_dev, inv_out_dev, D, H, W, n_items, max_iter, tol, stats_out_dev, ws);
    else
        invert_flow_kernel<2><<<grid, kThreads, 0, s>>>(flow_dev, inv_out_dev, 1, H, W, n_items, max_iter, tol, stats_out_dev, ws);
    return check_cuda(cudaGetLastError(), "invert_flow");
}
