// thinconv.cu — SURVEY.md §8 f-3 (U-Net-side work of flow mode): 3x3x3 valid convolutions with very few channels
// (C_in, C_out <= 4), forward, input gradient and weight / bias gradient.
//
// Replaces, from the reference (paths relative to /root/reference/src/TorchRegister/):
//   the full-resolution nn.Conv3d(kernel_size=3) layers of Attention_UNet (layer1, layer9; utils.py:409-520) at the
//   reference's width divisor n = 32 (channels 1 -> 2 -> 2 and 4 -> 2 -> 2), and autograd's backward of them.
//
// Why: cuDNN maps these onto tensor-core implicit GEMMs whose tiles are 64..256 output channels wide and converts
// NCDHW <-> NHWC around them; with 2 output channels that is 74 ms of a 106 ms epoch at 256^3 (four layers; torch.profiler,
// profiles/r02_unet_flow_profile.txt).  As a gather/stencil this is 27 * C_in loads and 27 * C_in * C_out FMAs per voxel
// — L1-resident loads, weights as constant-bank operands (copied device -> constant memory on the stream): no layout
// change, no im2col.
//   forward: one thread per (x, y) and block of 4 output slices, all C_out at once (an input plane serves three slices).
//   dgrad  : the same on the input side, all C_in at once (dy read with bounds predicates = the zero extension).
//   wgrad  : groups (c_in, dz): a warp walks rows of the output, 9 * C_out (+ C_out for the bias) running sums per
//            thread, block partials in fp64, fixed-order final sum (deterministic).
#include "common.cuh"

namespace trb {

constexpr int kTcMaxC = 4;                    // every pair up to here; above it the U-Net's own pairs (8,4), (4,8), (8,8)
constexpr int kTcMaxC8 = 8;
__constant__ float c_tc_w[kTcMaxC8 * kTcMaxC8 * 27];
__constant__ float c_tc_b[kTcMaxC8];

// y[co][z][y][x] = b[co] + sum_{ci,dz,dy,dx} w[co][ci][dz][dy][dx] * x[ci][z+dz][y+dy][x+dx]
// A thread owns kZB consecutive output slices of one (x, y): every input plane it loads serves up to three of them, so a voxel
// costs 13.5 C_in loads instead of 27 C_in, with kZB * C_out independent accumulator chains.
constexpr int kZB = 4;
template <int CI, int CO>
__global__ void __launch_bounds__(256) thinconv_fwd_kernel(const float *__restrict__ x, float *__restrict__ y, int D, int H, int W,
                                                            int has_bias)
{
    const int OD = D - 2, OH = H - 2, OW = W - 2;
    const int ox = blockIdx.x * 128 + (threadIdx.x & 127);
    const int oy = blockIdx.y * 2 + (threadIdx.x >> 7);
    const int oz0 = blockIdx.z * kZB;
    if (ox >= OW || oy >= OH) return;
    const size_t HW = (size_t)H * W, vol = HW * D, ovol = (size_t)OD * OH * OW;
    float acc[kZB][CO];
#pragma unroll
    for (int zo = 0; zo < kZB; ++zo)
#pragma unroll
        for (int co = 0; co < CO; ++co) acc[zo][co] = has_bias ? c_tc_b[co] : 0.f;
#pragma unroll
    for (int ci = 0; ci < CI; ++ci)
#pragma unroll
        for (int p = 0; p < kZB + 2; ++p) {
            if (oz0 + p >= D) break;                       // uniform over the block
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const float *row = x + ci * vol + (size_t)(oz0 + p) * HW + (size_t)(oy + dy) * W + ox;
                const float v0 = __ldg(row), v1 = __ldg(row + 1), v2 = __ldg(row + 2);
#pragma unroll
                for (int dz = 0; dz < 3; ++dz) {
                    const int zo = p - dz;                 // compile-time after unrolling
                    if (zo < 0 || zo >= kZB) continue;
#pragma unroll
                    for (int co = 0; co < CO; ++co) {
                        const int wi = ((co * CI + ci) * 3 + dz) * 9 + dy * 3;
                        acc[zo][co] = fmaf(c_tc_w[wi], v0, acc[zo][co]);
                        acc[zo][co] = fmaf(c_tc_w[wi + 1], v1, acc[zo][co]);
                        acc[zo][co] = fmaf(c_tc_w[wi + 2], v2, acc[zo][co]);
                    }
                }
            }
        }
#pragma unroll
    for (int zo = 0; zo < kZB; ++zo) {
        if (oz0 + zo >= OD) break;
        const size_t o = ((size_t)(oz0 + zo) * OH + oy) * OW + ox;
#pragma unroll
        for (int co = 0; co < CO; ++co) y[co * ovol + o] = acc[zo][co];
    }
}

// dx[ci][z][y][x] = sum_{co,dz,dy,dx} w[co][ci][dz][dy][dx] * dy[co][z-dz][y-dy][x-dx]   (dy = 0 outside its extent)
// The same z blocking on the input side: gradient plane q serves the input slices q, q + 1, q + 2.
template <int CI, int CO>
__global__ void __launch_bounds__(256) thinconv_dgrad_kernel(const float *__restrict__ gy, float *__restrict__ gx, int D, int H, int W)
{
    const int OD = D - 2, OH = H - 2, OW = W - 2;
    const int ix = blockIdx.x * 128 + (threadIdx.x & 127);
    const int iy = blockIdx.y * 2 + (threadIdx.x >> 7);
    const int iz0 = blockIdx.z * kZB;
    if (ix >= W || iy >= H) return;
    const size_t HW = (size_t)H * W, vol = HW * D, OHW = (size_t)OH * OW, ovol = OHW * OD;
    float acc[kZB][CI];
#pragma unroll
    for (int zi = 0; zi < kZB; ++zi)
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) acc[zi][ci] = 0.f;
    const bool p0 = (unsigned)ix < (unsigned)OW, p1 = (unsigned)(ix - 1) < (unsigned)OW, p2 = (unsigned)(ix - 2) < (unsigned)OW;
#pragma unroll
    for (int co = 0; co < CO; ++co)
#pragma unroll
        for (int p = 0; p < kZB + 2; ++p) {
            const int q = iz0 + p - 2;                     // gradient plane; uniform over the block
            if ((unsigned)q >= (unsigned)OD) continue;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const int yy = iy - dy;
                if ((unsigned)yy >= (unsigned)OH) continue;
                const float *row = gy + co * ovol + (size_t)q * OHW + (size_t)yy * OW + ix;
                const float v0 = p0 ? __ldg(row) : 0.f, v1 = p1 ? __ldg(row - 1) : 0.f, v2 = p2 ? __ldg(row - 2) : 0.f;
#pragma unroll
                for (int dz = 0; dz < 3; ++dz) {
                    const int zi = p - 2 + dz;             // input slice iz0 + zi = q + dz; compile-time after unrolling
                    if (zi < 0 || zi >= kZB) continue;
#pragma unroll
                    for (int ci = 0; ci < CI; ++ci) {
                        const int wi = ((co * CI + ci) * 3 + dz) * 9 + dy * 3;
                        acc[zi][ci] = fmaf(c_tc_w[wi], v0, acc[zi][ci]);
                        acc[zi][ci] = fmaf(c_tc_w[wi + 1], v1, acc[zi][ci]);
                        acc[zi][ci] = fmaf(c_tc_w[wi + 2], v2, acc[zi][ci]);
                    }
                }
            }
        }
#pragma unroll
    for (int zi = 0; zi < kZB; ++zi) {
        if (iz0 + zi >= D) break;
        const size_t o = (size_t)(iz0 + zi) * HW + (size_t)iy * W + ix;
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) gx[ci * vol + o] = acc[zi][ci];
    }
}

// grid (blocks, CI * 3 * co_groups): group g = (ci * 3 + dz) * co_groups + cg handles output channels [cg * COG, (cg + 1) * COG).
// part[g][block][9 * COG + COG] in fp64 (the last COG entries: sum dy, taken from the groups with ci = dz = 0).  A lane takes 4
// x positions per step so that 4 x (COG + 9) loads are in flight before the first FMA.
template <int COG>
__global__ void __launch_bounds__(256) thinconv_wgrad_kernel(const float *__restrict__ x, const float *__restrict__ gy, int D, int H, int W,
                                                              int co_groups, double *__restrict__ part)
{
    constexpr int NA = 9 * COG + COG, XB = 4;
    __shared__ double sh[kWarps][NA];
    const int OD = D - 2, OH = H - 2, OW = W - 2;
    const int g = blockIdx.y, cg = g % co_groups, cd = g / co_groups, ci = cd / 3, dz = cd - ci * 3;
    const size_t HW = (size_t)H * W, vol = HW * D, OHW = (size_t)OH * OW, ovol = OHW * OD;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rows = OD * OH;
    float a[NA];
    double A[NA];
#pragma unroll
    for (int i = 0; i < NA; ++i) { a[i] = 0.f; A[i] = 0.0; }
    int since = 0;
    for (int r = blockIdx.x * 8 + warp; r < rows; r += gridDim.x * 8) {
        const int z = r / OH, yy = r - z * OH;
        const float *xr = x + ci * vol + (size_t)(z + dz) * HW + (size_t)yy * W;
        const float *gr = gy + (size_t)(cg * COG) * ovol + (size_t)z * OHW + (size_t)yy * OW;
        for (int x0 = 0; x0 < OW; x0 += 32 * XB) {
            float gv[XB][COG], xv[XB][9];
#pragma unroll
            for (int j = 0; j < XB; ++j) {
                const int xx = x0 + 32 * j + lane;
                const bool in = xx < OW;
#pragma unroll
                for (int co = 0; co < COG; ++co) gv[j][co] = in ? __ldg(gr + co * ovol + xx) : 0.f;
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) xv[j][dy * 3 + dx] = in ? __ldg(xr + (size_t)dy * W + xx + dx) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < XB; ++j) {
#pragma unroll
                for (int k = 0; k < 9; ++k)
#pragma unroll
                    for (int co = 0; co < COG; ++co) a[co * 9 + k] = fmaf(gv[j][co], xv[j][k], a[co * 9 + k]);
#pragma unroll
                for (int co = 0; co < COG; ++co) a[9 * COG + co] += gv[j][co];
            }
        }
        if (++since == 4) {                    // fp32 runs of at most 4 rows per lane, fp64 above
#pragma unroll
            for (int i = 0; i < NA; ++i) { A[i] += (double)a[i]; a[i] = 0.f; }
            since = 0;
        }
    }
#pragma unroll
    for (int i = 0; i < NA; ++i) A[i] += (double)a[i];
    const double v = block_sum(A, sh);
    if (threadIdx.x < NA) part[((size_t)g * gridDim.x + blockIdx.x) * NA + threadIdx.x] = v;
}

// dw[co][ci][dz][dy][dx] and db[co] from the block partials, fixed order
__global__ void thinconv_wgrad_final_kernel(const double *__restrict__ part, int blocks, int CI, int CO, int COG, float *__restrict__ gw,
                                            float *__restrict__ gb)
{
    const int NA = 9 * COG + COG, co_groups = CO / COG;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < CO * CI * 27) {
        const int d = i % 9, dz = (i / 9) % 3, ci = (i / 27) % CI, co = i / (27 * CI);
        const int g = (ci * 3 + dz) * co_groups + co / COG, k = (co % COG) * 9 + d;
        double v = 0.0;
        for (int b = 0; b < blocks; ++b) v += part[((size_t)g * blocks + b) * NA + k];
        gw[i] = (float)v;
    } else if (gb && i < CO * CI * 27 + CO) {
        const int co = i - CO * CI * 27;
        const int g = co / COG;                                  // ci = dz = 0
        double v = 0.0;
        for (int b = 0; b < blocks; ++b) v += part[((size_t)g * blocks + b) * NA + 9 * COG + co % COG];
        gb[co] = (float)v;
    }
}

constexpr int kTcWgradBlocks = 96;

static bool tc_pair_ok(int CI, int CO)
{
    if (CI >= 1 && CI <= kTcMaxC && CO >= 1 && CO <= kTcMaxC) return true;
    return (CI == 8 && CO == 4) || (CI == 4 && CO == 8) || (CI == 8 && CO == 8);
}

static int tc_validate(int CI, int CO, int D, int H, int W)
{
    if (!tc_pair_ok(CI, CO)) { set_error("thin convolution handles 1..%d channels each way and 8->4, 4->8, 8->8 (got %d -> %d)", kTcMaxC, CI, CO); return TRB_ERR_UNSUPPORTED; }
    if (D < 3 || H < 3 || W < 3 || D > 65537) { set_error("bad volume shape %dx%dx%d", D, H, W); return TRB_ERR_ARG; }
    if ((unsigned long long)D * H * W * kTcMaxC8 >= (1ull << 40)) { set_error("volume too large"); return TRB_ERR_UNSUPPORTED; }
    return TRB_OK;
}

static int tc_upload(const float *w, const float *b, int CI, int CO, cudaStream_t s)
{
    cudaError_t e = cudaMemcpyToSymbolAsync(c_tc_w, w, (size_t)CO * CI * 27 * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess && b) e = cudaMemcpyToSymbolAsync(c_tc_b, b, (size_t)CO * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    return e == cudaSuccess ? TRB_OK : check_cuda(e, "cudaMemcpyToSymbolAsync(thin conv weights)");
}

#define TC_DISPATCH(KERNEL, ...)                                                                               \
    switch (CI * 8 + CO) {                                                                                     \
    case 1 * 8 + 1: KERNEL<1, 1> __VA_ARGS__; break; case 1 * 8 + 2: KERNEL<1, 2> __VA_ARGS__; break;          \
    case 1 * 8 + 3: KERNEL<1, 3> __VA_ARGS__; break; case 1 * 8 + 4: KERNEL<1, 4> __VA_ARGS__; break;          \
    case 2 * 8 + 1: KERNEL<2, 1> __VA_ARGS__; break; case 2 * 8 + 2: KERNEL<2, 2> __VA_ARGS__; break;          \
    case 2 * 8 + 3: KERNEL<2, 3> __VA_ARGS__; break; case 2 * 8 + 4: KERNEL<2, 4> __VA_ARGS__; break;          \
    case 3 * 8 + 1: KERNEL<3, 1> __VA_ARGS__; break; case 3 * 8 + 2: KERNEL<3, 2> __VA_ARGS__; break;          \
    case 3 * 8 + 3: KERNEL<3, 3> __VA_ARGS__; break; case 3 * 8 + 4: KERNEL<3, 4> __VA_ARGS__; break;          \
    case 4 * 8 + 1: KERNEL<4, 1> __VA_ARGS__; break; case 4 * 8 + 2: KERNEL<4, 2> __VA_ARGS__; break;          \
    case 4 * 8 + 3: KERNEL<4, 3> __VA_ARGS__; break; default: KERNEL<4, 4> __VA_ARGS__; break;                 \
    }
#define TC_DISPATCH3(KERNEL, ...)                                                                              \
    if (CI == 8 && CO == 4) { KERNEL<8, 4> __VA_ARGS__; }                                                      \
    else if (CI == 4 && CO == 8) { KERNEL<4, 8> __VA_ARGS__; }                                                 \
    else if (CI == 8 && CO == 8) { KERNEL<8, 8> __VA_ARGS__; }                                                 \
    else { TC_DISPATCH(KERNEL, __VA_ARGS__) }

}  // namespace trb

using namespace trb;

static int tc_cog(int CO) { return CO > 4 ? 4 : CO; }

extern "C" size_t trb_thinconv3_workspace_bytes(int CI, int CO)
{
    if (!tc_pair_ok(CI, CO)) return 0;
    const int COG = tc_cog(CO);
    return (size_t)CI * 3 * (CO / COG) * kTcWgradBlocks * (9 * COG + COG) * sizeof(double);
}

extern "C" int trb_thinconv3_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int n_batch, int CI,
                                     int CO, int D, int H, int W, void *stream)
{
    int rc = tc_validate(CI, CO, D, H, W);
    if (rc) return rc;
    if (!x_dev || !w_dev || !y_dev || n_batch < 1) { set_error("null pointer / batch"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    rc = tc_upload(w_dev, b_dev, CI, CO, s);
    if (rc) return rc;
    const int OD = D - 2, OH = H - 2, OW = W - 2;
    const dim3 grid((OW + 127) / 128, (OH + 1) / 2, (OD + kZB - 1) / kZB);
    const size_t vol = (size_t)D * H * W, ovol = (size_t)OD * OH * OW;
    for (int n = 0; n < n_batch; ++n) {
        const float *xn = x_dev + (size_t)n * CI * vol;
        float *yn = y_dev + (size_t)n * CO * ovol;
        TC_DISPATCH3(thinconv_fwd_kernel, <<<grid, 256, 0, s>>>(xn, yn, D, H, W, b_dev ? 1 : 0))
    }
    return check_cuda(cudaGetLastError(), "thinconv3_forward");
}

extern "C" int trb_thinconv3_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev,
                                      float *gb_dev, int n_batch, int CI, int CO, int D, int H, int W, void *workspace_dev,
                                      size_t workspace_bytes, void *stream)
{
    int rc = tc_validate(CI, CO, D, H, W);
    if (rc) return rc;
    if (!x_dev || !w_dev || !gy_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (n_batch != 1 && gw_dev) { set_error("weight gradient: one sample per call"); return TRB_ERR_UNSUPPORTED; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t vol = (size_t)D * H * W, ovol = (size_t)(D - 2) * (H - 2) * (W - 2);
    if (gx_dev) {
        rc = tc_upload(w_dev, nullptr, CI, CO, s);
        if (rc) return rc;
        const dim3 grid((W + 127) / 128, (H + 1) / 2, (D + kZB - 1) / kZB);
        for (int n = 0; n < n_batch; ++n) {
            const float *gn = gy_dev + (size_t)n * CO * ovol;
            float *xn = gx_dev + (size_t)n * CI * vol;
            TC_DISPATCH3(thinconv_dgrad_kernel, <<<grid, 256, 0, s>>>(gn, xn, D, H, W))
        }
    }
    if (gw_dev) {
        if (!workspace_dev || workspace_bytes < trb_thinconv3_workspace_bytes(CI, CO)) {
            set_error("workspace too small: need %zu bytes", trb_thinconv3_workspace_bytes(CI, CO));
            return TRB_ERR_WORKSPACE;
        }
        double *part = (double *)workspace_dev;
        const int COG = tc_cog(CO), cgs = CO / COG;
        const dim3 grid(kTcWgradBlocks, CI * 3 * cgs);
        switch (COG) {
        case 1: thinconv_wgrad_kernel<1><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, cgs, part); break;
        case 2: thinconv_wgrad_kernel<2><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, cgs, part); break;
        case 3: thinconv_wgrad_kernel<3><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, cgs, part); break;
        default: thinconv_wgrad_kernel<4><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, cgs, part); break;
        }
        const int n = CI * 27 * CO + CO;
        thinconv_wgrad_final_kernel<<<(n + 127) / 128, 128, 0, s>>>(part, kTcWgradBlocks, CI, CO, COG, gw_dev, gb_dev);
    }
    return check_cuda(cudaGetLastError(), "thinconv3_backward");
}

// ---- 1x1x1 convolutions with few channels (the attention gates of the U-Net: utils.py:368-406) -----------------------
// y[co][o] = b[co] + sum_ci w[co][ci] * x[ci][o * stride]  (stride 3 for the gate's projection of the skip, else 1).
// Pure streaming: C_in loads and C_out stores per output voxel; cuDNN spends 1-3.5 ms per call on them at 236^3..252^3.
namespace trb {

// forward: one thread per output voxel
template <int CI, int CO>
__global__ void __launch_bounds__(256) pointconv_fwd_kernel(const float *__restrict__ x, float *__restrict__ y, int D, int H, int W,
                                                             int OD, int OH, int OW, int stride, int has_bias)
{
    const size_t vol = (size_t)D * H * W, ovol = (size_t)OD * OH * OW;
    for (size_t o = (size_t)blockIdx.x * 256 + threadIdx.x; o < ovol; o += (size_t)gridDim.x * 256) {
        size_t i = o;
        if (stride != 1) {
            const int ox = (int)(o % OW);
            const size_t r = o / OW;
            const int oy = (int)(r % OH), oz = (int)(r / OH);
            i = ((size_t)oz * stride * H + (size_t)oy * stride) * W + (size_t)ox * stride;
        }
        float v[CI];
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) v[ci] = __ldg(x + ci * vol + i);
#pragma unroll
        for (int co = 0; co < CO; ++co) {
            float a = has_bias ? c_tc_b[co] : 0.f;
#pragma unroll
            for (int ci = 0; ci < CI; ++ci) a = fmaf(c_tc_w[co * CI + ci], v[ci], a);
            y[co * ovol + o] = a;
        }
    }
}

// input gradient: one thread per INPUT voxel (zeros where the stride skips it)
template <int CI, int CO>
__global__ void __launch_bounds__(256) pointconv_dgrad_kernel(const float *__restrict__ gy, float *__restrict__ gx, int D, int H, int W,
                                                               int OD, int OH, int OW, int stride)
{
    const size_t vol = (size_t)D * H * W, ovol = (size_t)OD * OH * OW;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < vol; i += (size_t)gridDim.x * 256) {
        size_t o = i;
        bool hit = true;
        if (stride != 1) {
            const int ix = (int)(i % W);
            const size_t r = i / W;
            const int iy = (int)(r % H), iz = (int)(r / H);
            const int ox = ix / stride, oy = iy / stride, oz = iz / stride;
            hit = ox * stride == ix && oy * stride == iy && oz * stride == iz && ox < OW && oy < OH && oz < OD;
            o = ((size_t)oz * OH + oy) * OW + ox;
        }
        float g[CO];
#pragma unroll
        for (int co = 0; co < CO; ++co) g[co] = hit ? __ldg(gy + co * ovol + o) : 0.f;
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) {
            float a = 0.f;
#pragma unroll
            for (int co = 0; co < CO; ++co) a = fmaf(c_tc_w[co * CI + ci], g[co], a);
            gx[ci * vol + i] = a;
        }
    }
}

// weight / bias gradient: CI*CO + CO running sums per thread over the output voxels; block partials in fp64
template <int CI, int CO>
__global__ void __launch_bounds__(256) pointconv_wgrad_kernel(const float *__restrict__ x, const float *__restrict__ gy, int D, int H, int W,
                                                               int OD, int OH, int OW, int stride, double *__restrict__ part)
{
    constexpr int NA = CI * CO + CO;
    __shared__ double sh[kWarps][NA];
    const size_t vol = (size_t)D * H * W, ovol = (size_t)OD * OH * OW;
    float a[NA];
    double A[NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) { a[k] = 0.f; A[k] = 0.0; }
    int since = 0;
    for (size_t o = (size_t)blockIdx.x * 256 + threadIdx.x; o < ovol; o += (size_t)gridDim.x * 256) {
        size_t i = o;
        if (stride != 1) {
            const int ox = (int)(o % OW);
            const size_t r = o / OW;
            const int oy = (int)(r % OH), oz = (int)(r / OH);
            i = ((size_t)oz * stride * H + (size_t)oy * stride) * W + (size_t)ox * stride;
        }
        float v[CI], g[CO];
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) v[ci] = __ldg(x + ci * vol + i);
#pragma unroll
        for (int co = 0; co < CO; ++co) g[co] = __ldg(gy + co * ovol + o);
#pragma unroll
        for (int co = 0; co < CO; ++co) {
#pragma unroll
            for (int ci = 0; ci < CI; ++ci) a[co * CI + ci] = fmaf(g[co], v[ci], a[co * CI + ci]);
            a[CI * CO + co] += g[co];
        }
        if (++since == 32) {
#pragma unroll
            for (int k = 0; k < NA; ++k) { A[k] += (double)a[k]; a[k] = 0.f; }
            since = 0;
        }
    }
#pragma unroll
    for (int k = 0; k < NA; ++k) A[k] += (double)a[k];
    const double s = block_sum(A, sh);
    if (threadIdx.x < NA) part[(size_t)blockIdx.x * NA + threadIdx.x] = s;
}

// one warp per sum: lanes stride over the block partials (fixed order), then a shuffle tree
__global__ void pointconv_wgrad_final_kernel(const double *__restrict__ part, int blocks, int CI, int CO, float *__restrict__ gw,
                                             float *__restrict__ gb)
{
    const int NA = CI * CO + CO, k = blockIdx.x;
    if (k >= NA) return;
    const double s = fold_blocks(part, blocks, NA, k);
    if (threadIdx.x == 0) {
        if (k < CI * CO) gw[k] = (float)s;
        else if (gb) gb[k - CI * CO] = (float)s;
    }
}

constexpr int kPcBlocks = 148 * 4;

static int pc_validate(int CI, int CO, int D, int H, int W, int stride)
{
    if (CI < 1 || CI > kTcMaxC || CO < 1 || CO > kTcMaxC) { set_error("thin 1x1 convolution handles 1..%d channels (got %d -> %d)", kTcMaxC, CI, CO); return TRB_ERR_UNSUPPORTED; }
    if (D < 1 || H < 1 || W < 1 || stride < 1) { set_error("bad shape %dx%dx%d / stride %d", D, H, W, stride); return TRB_ERR_ARG; }
    return TRB_OK;
}

}  // namespace trb

extern "C" size_t trb_pointconv_workspace_bytes(int CI, int CO)
{
    if (CI < 1 || CI > kTcMaxC || CO < 1 || CO > kTcMaxC) return 0;
    return (size_t)kPcBlocks * (CI * CO + CO) * sizeof(double);
}

extern "C" int trb_pointconv_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int CI, int CO, int D,
                                     int H, int W, int stride, void *stream)
{
    int rc = pc_validate(CI, CO, D, H, W, stride);
    if (rc) return rc;
    if (!x_dev || !w_dev || !y_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyToSymbolAsync(c_tc_w, w_dev, (size_t)CO * CI * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess && b_dev) e = cudaMemcpyToSymbolAsync(c_tc_b, b_dev, (size_t)CO * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return check_cuda(e, "cudaMemcpyToSymbolAsync(1x1 conv weights)");
    const int OD = (D - 1) / stride + 1, OH = (H - 1) / stride + 1, OW = (W - 1) / stride + 1;
    const size_t ovol = (size_t)OD * OH * OW;
    size_t nb = (ovol + 255) / 256;
    if (nb > 148 * 16) nb = 148 * 16;
    TC_DISPATCH(pointconv_fwd_kernel, <<<(unsigned)nb, 256, 0, s>>>(x_dev, y_dev, D, H, W, OD, OH, OW, stride, b_dev ? 1 : 0))
    return check_cuda(cudaGetLastError(), "pointconv_forward");
}

extern "C" int trb_pointconv_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev,
                                      float *gb_dev, int CI, int CO, int D, int H, int W, int stride, void *workspace_dev,
                                      size_t workspace_bytes, void *stream)
{
    int rc = pc_validate(CI, CO, D, H, W, stride);
    if (rc) return rc;
    if (!x_dev || !w_dev || !gy_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    const int OD = (D - 1) / stride + 1, OH = (H - 1) / stride + 1, OW = (W - 1) / stride + 1;
    if (gx_dev) {
        cudaError_t e = cudaMemcpyToSymbolAsync(c_tc_w, w_dev, (size_t)CO * CI * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) return check_cuda(e, "cudaMemcpyToSymbolAsync(1x1 conv weights)");
        size_t nb = ((size_t)D * H * W + 255) / 256;
        if (nb > 148 * 16) nb = 148 * 16;
        TC_DISPATCH(pointconv_dgrad_kernel, <<<(unsigned)nb, 256, 0, s>>>(gy_dev, gx_dev, D, H, W, OD, OH, OW, stride))
    }
    if (gw_dev) {
        if (!workspace_dev || workspace_bytes < trb_pointconv_workspace_bytes(CI, CO)) {
            set_error("workspace too small: need %zu bytes", trb_pointconv_workspace_bytes(CI, CO));
            return TRB_ERR_WORKSPACE;
        }
        double *part = (double *)workspace_dev;
        TC_DISPATCH(pointconv_wgrad_kernel, <<<kPcBlocks, 256, 0, s>>>(x_dev, gy_dev, D, H, W, OD, OH, OW, stride, part))
        pointconv_wgrad_final_kernel<<<CI * CO + CO, 32, 0, s>>>(part, kPcBlocks, CI, CO, gw_dev, gb_dev);
    }
    return check_cuda(cudaGetLastError(), "pointconv_backward");
}

// ---- 2x2x2 stride-2 transposed convolutions with few channels (the last up-sampling of the U-Net: utils.py:409-520) ---------
// y[co][2z+a][2y+b][2x+c] = bias[co] + sum_ci w[ci][co][a][b][c] * x[ci][z][y][x]: every output voxel has ONE source voxel, so
// this is a streaming kernel (C_in loads, 8 C_out stores per input voxel); cuDNN spends 1.5 ms each way on [4,118^3] -> [2,236^3].
namespace trb {

__constant__ float c_up_w[kTcMaxC * kTcMaxC * 8];

template <int CI, int CO>
__global__ void __launch_bounds__(256) upconv2_fwd_kernel(const float *__restrict__ x, float *__restrict__ y, int D, int H, int W, int has_bias)
{
    const size_t vol = (size_t)D * H * W, ovol = vol * 8;
    const int OW = 2 * W, OH = 2 * H;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < vol; i += (size_t)gridDim.x * 256) {
        const int ix = (int)(i % W);
        const size_t r = i / W;
        const int iy = (int)(r % H), iz = (int)(r / H);
        float v[CI];
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) v[ci] = __ldg(x + ci * vol + i);
#pragma unroll
        for (int co = 0; co < CO; ++co) {
            const float b = has_bias ? c_tc_b[co] : 0.f;
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int bb = 0; bb < 2; ++bb) {
                    float o0 = b, o1 = b;
#pragma unroll
                    for (int ci = 0; ci < CI; ++ci) {
                        o0 = fmaf(c_up_w[(ci * CO + co) * 8 + a * 4 + bb * 2], v[ci], o0);
                        o1 = fmaf(c_up_w[(ci * CO + co) * 8 + a * 4 + bb * 2 + 1], v[ci], o1);
                    }
                    float2 *dst = reinterpret_cast<float2 *>(y + co * ovol + ((size_t)(2 * iz + a) * OH + (2 * iy + bb)) * OW + 2 * ix);
                    __stcs(dst, make_float2(o0, o1));
                }
        }
    }
}

// gx[ci][v] = sum_{co,a,b,c} w[ci][co][a][b][c] * gy[co][2v + (a,b,c)]
template <int CI, int CO>
__global__ void __launch_bounds__(256) upconv2_dgrad_kernel(const float *__restrict__ gy, float *__restrict__ gx, int D, int H, int W)
{
    const size_t vol = (size_t)D * H * W, ovol = vol * 8;
    const int OW = 2 * W, OH = 2 * H;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < vol; i += (size_t)gridDim.x * 256) {
        const int ix = (int)(i % W);
        const size_t r = i / W;
        const int iy = (int)(r % H), iz = (int)(r / H);
        float acc[CI];
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) acc[ci] = 0.f;
#pragma unroll
        for (int co = 0; co < CO; ++co)
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int bb = 0; bb < 2; ++bb) {
                    const float2 g = __ldg(reinterpret_cast<const float2 *>(gy + co * ovol + ((size_t)(2 * iz + a) * OH + (2 * iy + bb)) * OW + 2 * ix));
#pragma unroll
                    for (int ci = 0; ci < CI; ++ci) {
                        acc[ci] = fmaf(c_up_w[(ci * CO + co) * 8 + a * 4 + bb * 2], g.x, acc[ci]);
                        acc[ci] = fmaf(c_up_w[(ci * CO + co) * 8 + a * 4 + bb * 2 + 1], g.y, acc[ci]);
                    }
                }
#pragma unroll
        for (int ci = 0; ci < CI; ++ci) gx[ci * vol + i] = acc[ci];
    }
}

// gw[ci][co][a][b][c] = sum_v x[ci][v] * gy[co][2v + (a,b,c)];  gb[co] = sum gy[co].  grid (blocks, CI): block partials in fp64
template <int CO>
__global__ void __launch_bounds__(256) upconv2_wgrad_kernel(const float *__restrict__ x, const float *__restrict__ gy, int D, int H, int W,
                                                             double *__restrict__ part)
{
    constexpr int NA = 8 * CO + CO;
    __shared__ double sh[kWarps][NA];
    const int ci = blockIdx.y;
    const size_t vol = (size_t)D * H * W, ovol = vol * 8;
    const int OW = 2 * W, OH = 2 * H;
    float acc[NA];
    double A[NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) { acc[k] = 0.f; A[k] = 0.0; }
    int since = 0;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < vol; i += (size_t)gridDim.x * 256) {
        const int ix = (int)(i % W);
        const size_t r = i / W;
        const int iy = (int)(r % H), iz = (int)(r / H);
        const float xv = __ldg(x + ci * vol + i);
#pragma unroll
        for (int co = 0; co < CO; ++co)
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int bb = 0; bb < 2; ++bb) {
                    const float2 g = __ldg(reinterpret_cast<const float2 *>(gy + co * ovol + ((size_t)(2 * iz + a) * OH + (2 * iy + bb)) * OW + 2 * ix));
                    acc[co * 8 + a * 4 + bb * 2] = fmaf(xv, g.x, acc[co * 8 + a * 4 + bb * 2]);
                    acc[co * 8 + a * 4 + bb * 2 + 1] = fmaf(xv, g.y, acc[co * 8 + a * 4 + bb * 2 + 1]);
                    acc[8 * CO + co] += g.x + g.y;
                }
        if (++since == 32) {
#pragma unroll
            for (int k = 0; k < NA; ++k) { A[k] += (double)acc[k]; acc[k] = 0.f; }
            since = 0;
        }
    }
#pragma unroll
    for (int k = 0; k < NA; ++k) A[k] += (double)acc[k];
    const double s = block_sum(A, sh);
    if (threadIdx.x < NA) part[((size_t)ci * gridDim.x + blockIdx.x) * NA + threadIdx.x] = s;
}

// one warp per entry: gw[ci][co][8] (k < 8*CO of group ci) and gb[co] (from group 0)
__global__ void upconv2_wgrad_final_kernel(const double *__restrict__ part, int blocks, int CI, int CO, float *__restrict__ gw, float *__restrict__ gb)
{
    const int NA = 8 * CO + CO, e = blockIdx.x;
    int ci, k;
    if (e < CI * CO * 8) { ci = e / (CO * 8); k = e - ci * CO * 8; }
    else { ci = 0; k = 8 * CO + (e - CI * CO * 8); }
    const double s = fold_blocks(part + (size_t)ci * blocks * NA, blocks, NA, k);
    if (threadIdx.x == 0) {
        if (e < CI * CO * 8) gw[e] = (float)s;          // [ci][co][a][b][c] is exactly e
        else if (gb) gb[e - CI * CO * 8] = (float)s;
    }
}

constexpr int kUpBlocks = 148 * 2;

static int up_upload(const float *w, const float *b, int CI, int CO, cudaStream_t s)
{
    cudaError_t e = cudaMemcpyToSymbolAsync(c_up_w, w, (size_t)CI * CO * 8 * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess && b) e = cudaMemcpyToSymbolAsync(c_tc_b, b, (size_t)CO * sizeof(float), 0, cudaMemcpyDeviceToDevice, s);
    return e == cudaSuccess ? TRB_OK : check_cuda(e, "cudaMemcpyToSymbolAsync(transposed conv weights)");
}

}  // namespace trb

extern "C" size_t trb_upconv2_workspace_bytes(int CI, int CO)
{
    if (CI < 1 || CI > kTcMaxC || CO < 1 || CO > kTcMaxC) return 0;
    return (size_t)CI * kUpBlocks * (8 * CO + CO) * sizeof(double);
}

extern "C" int trb_upconv2_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int CI, int CO, int D, int H,
                                   int W, void *stream)
{
    int rc = pc_validate(CI, CO, D, H, W, 1);
    if (rc) return rc;
    if (!x_dev || !w_dev || !y_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    rc = up_upload(w_dev, b_dev, CI, CO, s);
    if (rc) return rc;
    size_t nb = ((size_t)D * H * W + 255) / 256;
    if (nb > 148 * 16) nb = 148 * 16;
    TC_DISPATCH(upconv2_fwd_kernel, <<<(unsigned)nb, 256, 0, s>>>(x_dev, y_dev, D, H, W, b_dev ? 1 : 0))
    return check_cuda(cudaGetLastError(), "upconv2_forward");
}

extern "C" int trb_upconv2_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev, float *gb_dev,
                                    int CI, int CO, int D, int H, int W, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = pc_validate(CI, CO, D, H, W, 1);
    if (rc) return rc;
    if (!x_dev || !w_dev || !gy_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    if (gx_dev) {
        rc = up_upload(w_dev, nullptr, CI, CO, s);
        if (rc) return rc;
        size_t nb = ((size_t)D * H * W + 255) / 256;
        if (nb > 148 * 16) nb = 148 * 16;
        TC_DISPATCH(upconv2_dgrad_kernel, <<<(unsigned)nb, 256, 0, s>>>(gy_dev, gx_dev, D, H, W))
    }
    if (gw_dev) {
        if (!workspace_dev || workspace_bytes < trb_upconv2_workspace_bytes(CI, CO)) {
            set_error("workspace too small: need %zu bytes", trb_upconv2_workspace_bytes(CI, CO));
            return TRB_ERR_WORKSPACE;
        }
        double *part = (double *)workspace_dev;
        const dim3 grid(kUpBlocks, CI);
        switch (CO) {
        case 1: upconv2_wgrad_kernel<1><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, part); break;
        case 2: upconv2_wgrad_kernel<2><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, part); break;
        case 3: upconv2_wgrad_kernel<3><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, part); break;
        default: upconv2_wgrad_kernel<4><<<grid, 256, 0, s>>>(x_dev, gy_dev, D, H, W, part); break;
        }
        upconv2_wgrad_final_kernel<<<CI * CO * 8 + CO, 32, 0, s>>>(part, kUpBlocks, CI, CO, gw_dev, gb_dev);
    }
    return check_cuda(cudaGetLastError(), "upconv2_backward");
}
