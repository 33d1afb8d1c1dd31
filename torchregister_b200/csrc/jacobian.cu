// jacobian.cu — Jacobian determinant of a displacement field and its statistics (sm_100a).
//
// phi(p) = p + u(p) in voxel units, u the planar flow [ndim][D][H][W] of every flow here (channel i displaces spatial
// axis i: (z, y, x) in 3-D, (y, x) in 2-D).  J_ij = delta_ij + du_i/dp_j, each derivative numpy.gradient's: the central
// difference inside, the first-order one-sided difference at both ends of an axis.  The differences and the determinant
// are formed in fp64 from the fp32 flow, so the sign of det (the folding count) is exact up to fp64 rounding.
//
// One thread owns an (x, y) column and marches along z with the z-1 / z / z+1 flow values in registers, so every flow
// value is read from HBM once (its x / y neighbours are the same lines, read by the warp and the neighbouring warps of the
// CTA through L1).  Algorithmic traffic: 12 B/voxel read (8 in 2-D), + 4 B/voxel when the field is written.
#include "common.cuh"

namespace trb {

constexpr int kJacMaxBlocks = 2048;      // partial rows in the flow workspace (trb_flow_workspace_bytes)
constexpr int kJacTX = 32, kJacTY = kWarps;
constexpr int kJacZC = 32;               // z slices per thread: 2 halo slices per 32 read twice

// workspace (doubles): [4] ticket (as unsigned) ; [8 ..) sums[blocks][6] ; then (min, max)[blocks]
template <int NDIM>
__global__ void __launch_bounds__(kThreads) flow_jacobian_kernel(const float *__restrict__ flow, int D, int H, int W,
                                                                  int tiles_x, int n_chunks, long long n_items,
                                                                  float *__restrict__ det_out, double *__restrict__ stats,
                                                                  double *ws)
{
    const size_t HW = (size_t)H * W, vol = HW * D;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};     // n det <= 0, n non-finite, sum det, det^2, L, L^2
    double lo = INFINITY, hi = -INFINITY;
    for (long long it = blockIdx.x; it < n_items; it += gridDim.x) {
        const long long col = it / n_chunks;
        const int chunk = (int)(it - col * n_chunks);
        const int x = (int)(col % tiles_x) * kJacTX + tx, y = (int)(col / tiles_x) * kJacTY + ty;
        if (x >= W || y >= H) continue;
        const int xl = max(x - 1, 0), xr = min(x + 1, W - 1), yl = max(y - 1, 0), yr = min(y + 1, H - 1);
        const double sx = xr - xl == 2 ? 0.5 : 1.0, sy = yr - yl == 2 ? 0.5 : 1.0;
        const int z0 = chunk * kJacZC, z1 = min(z0 + kJacZC, D);
        const size_t rc = (size_t)y * W + x;
        float prev[NDIM], cur[NDIM], next[NDIM];
#pragma unroll
        for (int i = 0; i < NDIM; ++i) {
            cur[i] = __ldg(flow + i * vol + (size_t)z0 * HW + rc);
            prev[i] = z0 > 0 ? __ldg(flow + i * vol + (size_t)(z0 - 1) * HW + rc) : cur[i];
        }
        for (int z = z0; z < z1; ++z) {
            const size_t pl = (size_t)z * HW;
            const double sz = (z > 0 && z + 1 < D) ? 0.5 : 1.0;
            double J[NDIM][NDIM];
#pragma unroll
            for (int i = 0; i < NDIM; ++i) {
                const float *f = flow + i * vol + pl;
                next[i] = z + 1 < D ? __ldg(f + HW + rc) : cur[i];
                const double dx = ((double)__ldg(f + (size_t)y * W + xr) - (double)__ldg(f + (size_t)y * W + xl)) * sx;
                const double dy = ((double)__ldg(f + (size_t)yr * W + x) - (double)__ldg(f + (size_t)yl * W + x)) * sy;
                if constexpr (NDIM == 3) {
                    J[i][0] = ((double)next[i] - (double)prev[i]) * sz;
                    J[i][1] = dy;
                    J[i][2] = dx;
                } else {
                    J[i][0] = dy;
                    J[i][1] = dx;
                }
                J[i][i] += 1.0;
            }
            double det;
            if constexpr (NDIM == 3)
                det = J[0][0] * (J[1][1] * J[2][2] - J[1][2] * J[2][1]) - J[0][1] * (J[1][0] * J[2][2] - J[1][2] * J[2][0]) +
                      J[0][2] * (J[1][0] * J[2][1] - J[1][1] * J[2][0]);
            else
                det = J[0][0] * J[1][1] - J[0][1] * J[1][0];
            if (det_out) det_out[pl + rc] = (float)det;
            if (isfinite(det)) {
                const double L = log(fmin(fmax(det, 1e-9), 1e9));
                acc[0] += det <= 0.0 ? 1.0 : 0.0;
                acc[2] += det;
                acc[3] = fma(det, det, acc[3]);
                acc[4] += L;
                acc[5] = fma(L, L, acc[5]);
                lo = fmin(lo, det);
                hi = fmax(hi, det);
            } else {
                acc[1] += 1.0;
            }
#pragma unroll
            for (int i = 0; i < NDIM; ++i) { prev[i] = cur[i]; cur[i] = next[i]; }
        }
    }
    // min / max are exact in any order: per-block slots, folded by the last block
    __shared__ double mm[kWarps][2];
    __shared__ double red[kWarps][6];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(kFull, lo, o));
        hi = fmax(hi, __shfl_xor_sync(kFull, hi, o));
    }
    if (tx == 0) { mm[ty][0] = lo; mm[ty][1] = hi; }
    __syncthreads();
    double *mm_part = ws + 8 + (size_t)gridDim.x * 6;
    if (threadIdx.x == 0) {
        for (int w = 1; w < kWarps; ++w) { lo = fmin(lo, mm[w][0]); hi = fmax(hi, mm[w][1]); }
        __stcg(mm_part + 2 * (size_t)blockIdx.x, lo);
        __stcg(mm_part + 2 * (size_t)blockIdx.x + 1, hi);
    }
    if (!grid_sum(acc, red, ws + 8, (unsigned *)(ws + 4)) || ty != 0) return;
    lo = INFINITY; hi = -INFINITY;
    for (int b = tx; b < (int)gridDim.x; b += 32) {
        lo = fmin(lo, __ldcg(mm_part + 2 * (size_t)b));
        hi = fmax(hi, __ldcg(mm_part + 2 * (size_t)b + 1));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(kFull, lo, o));
        hi = fmax(hi, __shfl_xor_sync(kFull, hi, o));
    }
    if (tx == 0) {
        stats[0] = red[0][0]; stats[1] = red[0][1]; stats[2] = lo; stats[3] = hi;
        stats[4] = red[0][2]; stats[5] = red[0][3]; stats[6] = red[0][4]; stats[7] = red[0][5];
    }
}

}  // namespace trb

using namespace trb;

extern "C" int trb_flow_jacobian(int ndim, const float *flow_dev, int D, int H, int W, float *det_out_dev,
                                 double *stats_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (ndim == 2) D = 1;
    if (H < 2 || W < 2 || (ndim == 3 && D < 2)) {
        set_error("the Jacobian needs every spatial axis >= 2 (got %dx%dx%d)", D, H, W);
        return TRB_ERR_ARG;
    }
    if (!flow_dev || !stats_out_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_flow_workspace_bytes()) {
        set_error("workspace too small: need %zu bytes (trb_flow_workspace_bytes)", trb_flow_workspace_bytes());
        return TRB_ERR_WORKSPACE;
    }
    const int tiles_x = (W + kJacTX - 1) / kJacTX, tiles_y = (H + kJacTY - 1) / kJacTY;
    const int n_chunks = (D + kJacZC - 1) / kJacZC;
    const long long n_items = (long long)tiles_x * tiles_y * n_chunks;
    const unsigned grid = (unsigned)(n_items < kJacMaxBlocks ? n_items : kJacMaxBlocks);
    double *ws = (double *)workspace_dev;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3)
        flow_jacobian_kernel<3><<<grid, kThreads, 0, s>>>(flow_dev, D, H, W, tiles_x, n_chunks, n_items, det_out_dev, stats_out_dev, ws);
    else
        flow_jacobian_kernel<2><<<grid, kThreads, 0, s>>>(flow_dev, D, H, W, tiles_x, n_chunks, n_items, det_out_dev, stats_out_dev, ws);
    return check_cuda(cudaGetLastError(), "flow_jacobian");
}
