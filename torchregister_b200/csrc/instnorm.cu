// instnorm.cu — SURVEY.md §8 f-3 (U-Net-side work of flow mode): InstanceNorm over [N*C] instances of S spatial elements,
// forward and backward, optionally fused with the ReLU that precedes every InstanceNorm of the reference's U-Net.
//
// Replaces, from the reference (paths relative to /root/reference/src/TorchRegister/):
//   nn.InstanceNorm3d / nn.InstanceNorm2d (affine=False, no running stats, eps 1e-5) in the conv -> ReLU -> InstanceNorm
//   blocks and the attention gates of Attention_UNet, utils.py:368-520, and autograd's backward of them.
//
// Why: PyTorch runs instance norm as batch norm over N*C "channels" and parallelises over channels only.  The flow U-Net
// at the reference's width divisor n = 32 has 2..32 channels, so at 256^3 its statistics / transform / backward kernels
// run on 2..32 thread blocks for 16.6 M elements per channel: 391 ms of a 492 ms epoch (torch.profiler,
// profiles/r02_unet_flow_profile.txt).  These kernels cut every instance into chunks over the whole grid (two-stage,
// fixed-order fp64 reduction: deterministic) and stream float4s: the layer becomes HBM bound.
//   forward : stats (sum, sum of squares of relu?(x))  ->  finalise (mean, rstd)  ->  y = (relu?(x) - mean) * rstd
//   backward: sums (sum dy, sum dy*y)                  ->  finalise               ->  dx = rstd * (dy - m1 - y*m2) [* (x > 0)]
#include "common.cuh"

namespace trb {

constexpr int kInChunkElems = 16384;          // elements per block of the reduction passes
constexpr int kInMaxChunks = 4096;            // chunks per instance

static int in_chunks(long long S)
{
    long long c = (S + kInChunkElems - 1) / kInChunkElems;
    if (c > kInMaxChunks) c = kInMaxChunks;
    if (c < 1) c = 1;
    return (int)c;
}

// grid (chunks, instances).  BWD = false: (sum v, sum v^2) of v = relu?(x);  BWD = true: (sum dy, sum dy*y), y from x and stats.
template <bool BWD, bool VEC>
__global__ void __launch_bounds__(256) instnorm_sums_kernel(const float *__restrict__ x, const float *__restrict__ gate,
                                                             const float *__restrict__ dy, long long S,
                                                             int relu, const float *__restrict__ stats, double *__restrict__ part)
{
    __shared__ double sh[kWarps][2];
    const int chunk = blockIdx.x, chunks = gridDim.x, inst = blockIdx.y;
    const long long i0 = S * chunk / chunks, i1 = S * (chunk + 1) / chunks;
    const float *xi = x + (size_t)inst * S;
    const float *di = BWD ? dy + (size_t)inst * S : nullptr;
    const float mean = BWD ? stats[2 * inst] : 0.f, rstd = BWD ? stats[2 * inst + 1] : 0.f;
    float a = 0.f, b = 0.f;
    double A = 0.0, B = 0.0;
    auto add = [&](float xv, float dv) {                  // xv: already multiplied by the gate, if any
        const float v = relu ? fmaxf(xv, 0.f) : xv;
        if (BWD) { const float y = (v - mean) * rstd; a += dv; b = fmaf(dv, y, b); }
        else { a += v; b = fmaf(v, v, b); }
    };
    if (VEC) {
        // S % 4 == 0 and 16-byte aligned bases: chunk borders are rounded to float4s
        const long long v0 = (i0 + 3) / 4, v1 = chunk + 1 == chunks ? S / 4 : (i1 + 3) / 4;
        const float4 *x4 = reinterpret_cast<const float4 *>(xi), *d4 = reinterpret_cast<const float4 *>(di);
        const float4 *g4 = reinterpret_cast<const float4 *>(gate);
        int n = 0;
        for (long long i = v0 + threadIdx.x; i < v1; i += 256) {
            float4 xv = __ldg(x4 + i);
            if (gate) { const float4 gv = __ldg(g4 + i); xv.x *= gv.x; xv.y *= gv.y; xv.z *= gv.z; xv.w *= gv.w; }
            float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (BWD) dv = __ldg(d4 + i);
            add(xv.x, dv.x); add(xv.y, dv.y); add(xv.z, dv.z); add(xv.w, dv.w);
            if (++n == 8) { A += (double)a; B += (double)b; a = b = 0.f; n = 0; }      // fp32 runs of 32 values, fp64 above
        }
    } else {
        int n = 0;
        for (long long i = i0 + threadIdx.x; i < i1; i += 256) {
            add(gate ? __ldg(xi + i) * __ldg(gate + i) : __ldg(xi + i), BWD ? __ldg(di + i) : 0.f);
            if (++n == 32) { A += (double)a; B += (double)b; a = b = 0.f; n = 0; }
        }
    }
    const double AB[2] = {A + (double)a, B + (double)b};
    const double t = block_sum(AB, sh);
    if (threadIdx.x < 2) __stcg(part + ((size_t)inst * chunks + chunk) * 2 + threadIdx.x, t);
}

// grid (instances).  FWD: stats[inst] = (mean, rstd).  BWD: coef[inst] = (mean dy, mean dy*y).
__global__ void __launch_bounds__(256) instnorm_finalise_kernel(const double *__restrict__ part, int chunks, long long S, float eps, int bwd,
                                                                 float *__restrict__ out)
{
    __shared__ double sh[kWarps][2];
    const int inst = blockIdx.x;
    const double *p = part + (size_t)inst * chunks * 2;
    double AB[2] = {0.0, 0.0};
    for (int c = threadIdx.x; c < chunks; c += 256) { AB[0] += p[2 * c]; AB[1] += p[2 * c + 1]; }
    block_sum_all(AB, sh);
    const double A = AB[0], B = AB[1];
    if (threadIdx.x == 0) {
        const double n = (double)S;
        if (bwd) { out[2 * inst] = (float)(A / n); out[2 * inst + 1] = (float)(B / n); }
        else {
            const double mean = A / n;
            double var = B / n - mean * mean;          // biased variance, fp64 sums of fp32 data
            if (var < 0.0) var = 0.0;
            out[2 * inst] = (float)mean;
            out[2 * inst + 1] = (float)(1.0 / sqrt(var + (double)eps));
        }
    }
}

// grid (blocks, instances).  FWD: y = (relu?(x) - mean) * rstd.  BWD: dx = rstd * (dy - m1 - y * m2), times (x > 0) with relu.
template <bool BWD, bool VEC>
__global__ void __launch_bounds__(256) instnorm_apply_kernel(const float *__restrict__ x, const float *__restrict__ gate,
                                                              const float *__restrict__ dy, long long S, int relu,
                                                              const float *__restrict__ stats, const float *__restrict__ coef,
                                                              float *__restrict__ out)
{
    const int inst = blockIdx.y;
    const float mean = stats[2 * inst], rstd = stats[2 * inst + 1];
    const float m1 = BWD ? coef[2 * inst] : 0.f, m2 = BWD ? coef[2 * inst + 1] : 0.f;
    const float *xi = x + (size_t)inst * S;
    const float *di = BWD ? dy + (size_t)inst * S : nullptr;
    float *oi = out + (size_t)inst * S;
    auto f = [&](float xv, float dv) {
        const float v = relu ? fmaxf(xv, 0.f) : xv;
        const float y = (v - mean) * rstd;
        if (!BWD) return y;
        const float g = rstd * (dv - m1 - y * m2);
        return (relu && !(xv > 0.f)) ? 0.f : g;
    };
    const long long stride = (long long)gridDim.x * 256;
    if (VEC) {
        const float4 *x4 = reinterpret_cast<const float4 *>(xi), *d4 = reinterpret_cast<const float4 *>(di);
        float4 *o4 = reinterpret_cast<float4 *>(oi);
        const float4 *g4 = reinterpret_cast<const float4 *>(gate);
        for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < S / 4; i += stride) {
            float4 xv = __ldg(x4 + i);
            if (gate) { const float4 gv = __ldg(g4 + i); xv.x *= gv.x; xv.y *= gv.y; xv.z *= gv.z; xv.w *= gv.w; }
            float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (BWD) dv = __ldg(d4 + i);
            o4[i] = make_float4(f(xv.x, dv.x), f(xv.y, dv.y), f(xv.z, dv.z), f(xv.w, dv.w));
        }
    } else {
        for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < S; i += stride)
            oi[i] = f(gate ? __ldg(xi + i) * __ldg(gate + i) : __ldg(xi + i), BWD ? __ldg(di + i) : 0.f);
    }
}

// Gated form y_c = IN(x_c * g) (the attention gate's `bnorm(x * w)`, utils.py:403-405; one sample, g shared by its channels):
// backward for ALL channels of a voxel in one thread: dv_c = rstd_c (dy_c - m1_c - y_c m2_c), dx_c = dv_c g, dg = sum_c dv_c x_c.
constexpr int kInMaxGatedC = 64;
__global__ void __launch_bounds__(256) instnorm_gated_bwd_kernel(const float *__restrict__ x, const float *__restrict__ gate,
                                                                  const float *__restrict__ dy, long long S, int C,
                                                                  const float *__restrict__ stats, const float *__restrict__ coef,
                                                                  float *__restrict__ dx, float *__restrict__ dgate)
{
    __shared__ float sc[kInMaxGatedC][4];
    for (int c = threadIdx.x; c < C; c += 256) {
        sc[c][0] = stats[2 * c]; sc[c][1] = stats[2 * c + 1]; sc[c][2] = coef[2 * c]; sc[c][3] = coef[2 * c + 1];
    }
    __syncthreads();
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < S; i += (long long)gridDim.x * 256) {
        const float g = __ldg(gate + i);
        float dg = 0.f;
        for (int c = 0; c < C; ++c) {
            const float xv = __ldg(x + (size_t)c * S + i);
            const float y = (xv * g - sc[c][0]) * sc[c][1];
            const float dv = sc[c][1] * (__ldg(dy + (size_t)c * S + i) - sc[c][2] - y * sc[c][3]);
            dx[(size_t)c * S + i] = dv * g;
            dg = fmaf(dv, xv, dg);
        }
        dgate[i] = dg;
    }
}

static int in_validate(const void *a, const void *b, int n_inst, long long S, const void *ws, size_t ws_bytes)
{
    if (!a || !b) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (n_inst < 1 || n_inst > 65535 || S < 1) { set_error("bad instance count %d / size %lld", n_inst, S); return TRB_ERR_ARG; }
    const size_t need = (size_t)n_inst * in_chunks(S) * 2 * sizeof(double);
    if (!ws || ws_bytes < need) { set_error("workspace too small: need %zu bytes", need); return TRB_ERR_WORKSPACE; }
    return TRB_OK;
}

static unsigned in_apply_blocks(long long S, int n_inst)
{
    long long nb = (S / 4 + 255) / 256;
    const long long cap = (148LL * 16 + n_inst - 1) / n_inst;
    if (nb > cap) nb = cap;
    if (nb < 1) nb = 1;
    return (unsigned)nb;
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_instnorm_workspace_bytes(int n_inst, long long S)
{
    if (n_inst < 1 || S < 1) return 0;
    return (size_t)n_inst * in_chunks(S) * 2 * sizeof(double);
}

extern "C" int trb_instnorm_forward(const float *x_dev, const float *gate_dev, float *y_dev, int n_inst, long long S, float eps, int relu,
                                    float *stats_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = in_validate(x_dev, y_dev, n_inst, S, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!stats_dev) { set_error("null stats"); return TRB_ERR_ARG; }
    if (gate_dev && relu) { set_error("the gated form has no ReLU"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    double *part = (double *)workspace_dev;
    const int chunks = in_chunks(S);
    const bool vec = S % 4 == 0 && (((uintptr_t)x_dev | (uintptr_t)y_dev | (uintptr_t)gate_dev) & 15) == 0;
    const dim3 gs(chunks, n_inst), ga(in_apply_blocks(S, n_inst), n_inst);
    if (vec) instnorm_sums_kernel<false, true><<<gs, 256, 0, s>>>(x_dev, gate_dev, nullptr, S, relu, nullptr, part);
    else instnorm_sums_kernel<false, false><<<gs, 256, 0, s>>>(x_dev, gate_dev, nullptr, S, relu, nullptr, part);
    instnorm_finalise_kernel<<<n_inst, 256, 0, s>>>(part, chunks, S, eps, 0, stats_dev);
    if (vec) instnorm_apply_kernel<false, true><<<ga, 256, 0, s>>>(x_dev, gate_dev, nullptr, S, relu, stats_dev, nullptr, y_dev);
    else instnorm_apply_kernel<false, false><<<ga, 256, 0, s>>>(x_dev, gate_dev, nullptr, S, relu, stats_dev, nullptr, y_dev);
    return check_cuda(cudaGetLastError(), "instnorm_forward");
}

extern "C" int trb_instnorm_backward(const float *x_dev, const float *gate_dev, const float *dy_dev, float *dx_dev, float *dgate_dev,
                                     int n_inst, long long S, int relu, const float *stats_dev, float *coef_dev, void *workspace_dev,
                                     size_t workspace_bytes, void *stream)
{
    int rc = in_validate(x_dev, dy_dev, n_inst, S, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!dx_dev || !stats_dev || !coef_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (gate_dev && (relu || !dgate_dev || n_inst > kInMaxGatedC)) { set_error("gated form: no ReLU, dgate required, <= %d channels", kInMaxGatedC); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    double *part = (double *)workspace_dev;
    const int chunks = in_chunks(S);
    const bool vec = S % 4 == 0 && (((uintptr_t)x_dev | (uintptr_t)dy_dev | (uintptr_t)dx_dev | (uintptr_t)gate_dev) & 15) == 0;
    const dim3 gs(chunks, n_inst), ga(in_apply_blocks(S, n_inst), n_inst);
    if (vec) instnorm_sums_kernel<true, true><<<gs, 256, 0, s>>>(x_dev, gate_dev, dy_dev, S, relu, stats_dev, part);
    else instnorm_sums_kernel<true, false><<<gs, 256, 0, s>>>(x_dev, gate_dev, dy_dev, S, relu, stats_dev, part);
    instnorm_finalise_kernel<<<n_inst, 256, 0, s>>>(part, chunks, S, 0.f, 1, coef_dev);
    if (gate_dev) {
        long long nb = (S + 255) / 256;
        if (nb > 148 * 16) nb = 148 * 16;
        instnorm_gated_bwd_kernel<<<(unsigned)nb, 256, 0, s>>>(x_dev, gate_dev, dy_dev, S, n_inst, stats_dev, coef_dev, dx_dev, dgate_dev);
    } else if (vec) instnorm_apply_kernel<true, true><<<ga, 256, 0, s>>>(x_dev, nullptr, dy_dev, S, relu, stats_dev, coef_dev, dx_dev);
    else instnorm_apply_kernel<true, false><<<ga, 256, 0, s>>>(x_dev, nullptr, dy_dev, S, relu, stats_dev, coef_dev, dx_dev);
    return check_cuda(cudaGetLastError(), "instnorm_backward");
}
