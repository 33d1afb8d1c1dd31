// edge.cu — Edge3D pre-filter (SURVEY.md §8 f-4; reference utils.py:82-183): nine 3x3x3 Sobel-type cross-correlations
// of a reflect-padded volume, gradient magnitude over filters and channels, min-max normalisation, band threshold —
// as ONE stencil pass (27 neighbours read once, all nine filters from registers/constant memory) plus one threshold
// pass, instead of the reference's 9*C conv3d launches over a padded copy.
#include "common.cuh"

namespace trb {

constexpr double kEdgeEps = 1e-10;      // utils.py:15 EPSILON, added where the reference adds it (:172-173)
__constant__ float c_sobel[9 * 27];

__device__ __forceinline__ int reflect1(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }
__device__ __forceinline__ unsigned f2ord(float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(unsigned u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

// grad[b][x][y][z] = (1/C) * sqrt( sum_s ( sum_c (corr_s(img[b][c]) + eps) )^2 + eps ) ; minmax: ordered-uint min / max
__global__ void __launch_bounds__(256) edge_grad_kernel(const float *__restrict__ img, float *__restrict__ grad, int B, int C,
                                                         int X, int Y, int Z, unsigned *minmax)
{
    const size_t vol = (size_t)X * Y * Z, total = vol * B;
    float lo = 3.4e38f, hi = -3.4e38f;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(idx / vol);
        const size_t r = idx - (size_t)b * vol;
        const int x = (int)(r / ((size_t)Y * Z)), y = (int)((r / Z) % Y), z = (int)(r % Z);
        float q[9];
#pragma unroll
        for (int s = 0; s < 9; ++s) q[s] = 0.f;
        for (int c = 0; c < C; ++c) {
            const float *v = img + ((size_t)b * C + c) * vol;
            float acc[9];
#pragma unroll
            for (int s = 0; s < 9; ++s) acc[s] = 0.f;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int xx = reflect1(x + a - 1, X);
#pragma unroll
                for (int bb = 0; bb < 3; ++bb) {
                    const int yy = reflect1(y + bb - 1, Y);
#pragma unroll
                    for (int cc = 0; cc < 3; ++cc) {
                        const int zz = reflect1(z + cc - 1, Z);
                        const float val = __ldg(v + ((size_t)xx * Y + yy) * Z + zz);
#pragma unroll
                        for (int s = 0; s < 9; ++s) acc[s] = fmaf(c_sobel[s * 27 + (a * 3 + bb) * 3 + cc], val, acc[s]);
                    }
                }
            }
#pragma unroll
            for (int s = 0; s < 9; ++s) q[s] += acc[s] + (float)kEdgeEps;
        }
        float m = 0.f;
#pragma unroll
        for (int s = 0; s < 9; ++s) m += fmaf(q[s], q[s], (float)kEdgeEps);
        const float g = sqrtf(m) / (float)C;
        grad[idx] = g;
        lo = fminf(lo, g); hi = fmaxf(hi, g);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { lo = fminf(lo, __shfl_xor_sync(kFull, lo, o)); hi = fmaxf(hi, __shfl_xor_sync(kFull, hi, o)); }
    if ((threadIdx.x & 31) == 0) { atomicMin(minmax, f2ord(lo)); atomicMax(minmax + 1, f2ord(hi)); }
}

// edges = (g - min) / ((max - min) + 1e-9) ; out = (edges > lo && edges < hi) ? 1 : 0      (utils.py:262-267,176-181)
__global__ void __launch_bounds__(256) edge_threshold_kernel(float *__restrict__ grad, size_t total, const unsigned *minmax,
                                                              float t_lo, float t_hi, float *__restrict__ norm_out)
{
    const float mn = ord2f(minmax[0]), mx = ord2f(minmax[1]);
    const float den = (mx - mn) + 1e-9f;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const float e = (grad[idx] - mn) / den;
        if (norm_out) norm_out[idx] = e;
        grad[idx] = (e > t_lo && e < t_hi) ? 1.f : 0.f;
    }
}

}  // namespace trb

using namespace trb;

// out_dev: [B][X][Y][Z] fp32 (doubles as the scratch for the gradient magnitude); minmax_dev: 2 x u32 scratch;
// weights_host: [9][27] fp32 = the nine 3x3x3 kernels of get_sobel_kernel3D (utils.py:82-127) in (x,y,z) order;
// norm_out_dev (optional): the normalised gradient magnitude before thresholding (tests / diagnostics).
extern "C" int trb_edge3d(const float *img_dev, float *out_dev, int B, int C, int X, int Y, int Z, const float *weights_host,
                          float thresh_lo, float thresh_hi, unsigned *minmax_dev, float *norm_out_dev, void *stream)
{
    if (!img_dev || !out_dev || !weights_host || !minmax_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (B < 1 || C < 1 || X < 2 || Y < 2 || Z < 2) { set_error("Edge3D needs [B,C,X,Y,Z] with every spatial axis >= 2"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyToSymbolAsync(c_sobel, weights_host, 9 * 27 * sizeof(float), 0, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return check_cuda(e, "cudaMemcpyToSymbolAsync(sobel)");
    const unsigned init[2] = {0xffffffffu, 0u};
    e = cudaMemcpyAsync(minmax_dev, init, sizeof(init), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return check_cuda(e, "cudaMemcpyAsync(minmax)");
    const size_t total = (size_t)B * X * Y * Z;
    int sms;
    if (int rc = sm_count(sms)) return rc;
    size_t nb = (total + 255) / 256;
    if (nb > (size_t)sms * 8) nb = (size_t)sms * 8;
    edge_grad_kernel<<<(unsigned)nb, 256, 0, s>>>(img_dev, out_dev, B, C, X, Y, Z, minmax_dev);
    edge_threshold_kernel<<<(unsigned)nb, 256, 0, s>>>(out_dev, total, minmax_dev, thresh_lo, thresh_hi, norm_out_dev);
    return check_cuda(cudaGetLastError(), "edge3d");
}
