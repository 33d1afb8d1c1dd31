// flow.cu — flow-field warp, its VJP, and the fused warp+similarity+gradient node (sm_100a).
//
// Replaces, from the reference (paths relative to /root/reference/src/TorchRegister/):
//   SpatialTransformer.forward                         utils.py:350-365
//   the similarity forward + backward down to the flow warpings.py:213-215 (MSELoss, NCCLoss utils.py:197-205)
//   flow_register.deform / Register.__call__           warpings.py:238-242, torchregister.py:124-125
//
// Layout: src/target fp32 [D][H][W]; flow fp32 [ndim][D][H][W] (planar, channel i displaces
// spatial axis i).  One thread per output voxel, x fastest: flow/target/dflow/warped accesses are
// fully coalesced streams, the 8 (4) gathered corners hit neighbouring lines of `src`.
// Algorithmic traffic of the fused node: 32 B/voxel (moving 4 + target 4 + flow 12 read,
// dflow 12 written) + 20 B/voxel for the statistics pre-pass when the NCC term is on.
#include "common.cuh"

namespace trb {

// voxel (x,y,z) -> the sample position displaced by the flow
struct FlowAxes {
    AxisMap x, y, z;
};
__device__ __forceinline__ FlowAxes flow_axes(int D, int H, int W)
{
    FlowAxes a;
    a.x = axis_map(W); a.y = axis_map(H); a.z = axis_map(D > 1 ? D : 2);
    return a;
}
// DEVICE_GRID: the reference's grid as torch forms it on a CUDA device (flow_pos_rcp), else as on the CPU (flow_pos)
template <int NDIM, bool DEVICE_GRID = false>
__device__ __forceinline__ void flow_position(const float *__restrict__ flow, size_t vol, size_t idx, int x, int y, int z,
                                              const FlowAxes &ax, float &px, float &py, float &pz)
{
    const auto pos = [](const AxisMap &m, int i, float f) { return DEVICE_GRID ? flow_pos_rcp(m, i, f) : flow_pos(m, i, f); };
    if (NDIM == 3) {
        pz = pos(ax.z, z, ld_stream_f(flow + idx));
        py = pos(ax.y, y, ld_stream_f(flow + vol + idx));
        px = pos(ax.x, x, ld_stream_f(flow + 2 * vol + idx));
    } else {
        pz = 0.f;
        py = pos(ax.y, y, ld_stream_f(flow + idx));
        px = pos(ax.x, x, ld_stream_f(flow + vol + idx));
    }
}

template <int NDIM>
__global__ void __launch_bounds__(256, 4) warp_flow_kernel(const float *__restrict__ src, const float *__restrict__ flow,
                                                         float *__restrict__ out, int n_channels, int D, int H, int W)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    for_each_voxel<2>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        for (int c = 0; c < n_channels; ++c)
            out[(size_t)c * vol + idx] = sample_zero_pad<NDIM, false>(src + (size_t)c * vol, D, H, W, px, py, pz).val;
    });
}

// grid_sample(mode='nearest', align_corners=True) on the reference's grid as the device forms it: flow_position<.., true>
// reproduces that fp32 grid op for op and round_idx is torch's nearbyint, so the result is torch's on CUDA bit for bit
template <int NDIM>
__global__ void __launch_bounds__(256, 4) warp_flow_nearest_kernel(const float *__restrict__ src, const float *__restrict__ flow,
                                                                 float *__restrict__ out, int n_channels, int D, int H, int W)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    for_each_voxel<2>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM, true>(flow, vol, idx, x, y, z, ax, px, py, pz);
        long long o;
        const bool v = nearest_offset(NDIM == 3 ? D : 1, H, W, px, py, pz, o);
        for (int c = 0; c < n_channels; ++c) out[(size_t)c * vol + idx] = v ? __ldg(src + (size_t)c * vol + o) : 0.f;
    });
}

// dflow channel a (spatial axis a) receives the derivative along sampling coordinate NDIM-1-a
template <int NDIM>
__device__ __forceinline__ void store_dflow(float *__restrict__ dflow, size_t vol, size_t idx, float r, const float *g)
{
#pragma unroll
    for (int a = 0; a < NDIM; ++a) dflow[(size_t)a * vol + idx] = r * g[NDIM - 1 - a];
}

template <int NDIM>
__global__ void __launch_bounds__(256) warp_flow_vjp_kernel(const float *__restrict__ src, const float *__restrict__ flow,
                                                             const float *__restrict__ gout, float *__restrict__ dflow,
                                                             int D, int H, int W)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        const Sample<NDIM> s = sample_zero_pad<NDIM, true>(src, D, H, W, px, py, pz);
        store_dflow<NDIM>(dflow, vol, idx, ld_stream_f(gout + idx), s.g);
    });
}

// workspace layout (doubles): [0..3] cw, ct, c0, loss ; [4] ticket (as unsigned) ; [8..] partials[blocks][5]

template <int NDIM>
__global__ void __launch_bounds__(256) flow_stats_kernel(const float *__restrict__ moving, const float *__restrict__ target,
                                                          const float *__restrict__ flow, float *__restrict__ warped,
                                                          int D, int H, int W, double w_mse, double w_ncc,
                                                          double *ws, float *loss_out)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    // a thread sums ~50-60 voxels (grid = 8 CTAs per SM): fp32 partials are exact enough (values in [0,1],
    // relative error < 4e-6 worst case) and keep the register count low enough for full occupancy; everything
    // above the thread level is fp64
    float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        const float w = sample_zero_pad<NDIM, false, false>(moving, D, H, W, px, py, pz).val;
        const float t = ld_stream_f(target + idx);
        if (warped) warped[idx] = w;
        s[0] += t; s[1] += w;
        s[2] = fmaf(t, t, s[2]); s[3] = fmaf(w, w, s[3]); s[4] = fmaf(t, w, s[4]);
    });
    __shared__ double red[kWarps][5];
    if (!grid_sum(s, red, ws + 8, (unsigned *)(ws + 4)) || threadIdx.x != 0) return;
    const LossCoef lc = loss_coefficients((double)vol, red[0][0], red[0][1], red[0][2], red[0][3], red[0][4], w_mse, w_ncc);
    ws[0] = lc.cw; ws[1] = lc.ct; ws[2] = lc.c0; ws[3] = lc.loss;
    if (loss_out) *loss_out = (float)lc.loss;
}

template <int NDIM>
__global__ void __launch_bounds__(256) flow_grad_kernel(const float *__restrict__ moving, const float *__restrict__ target,
                                                         const float *__restrict__ flow, float *__restrict__ dflow,
                                                         int D, int H, int W, const double *__restrict__ ws)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    const float cw = (float)ws[0], ct = (float)ws[1], c0 = (float)ws[2];
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        const Sample<NDIM> s = sample_zero_pad<NDIM, true, false>(moving, D, H, W, px, py, pz);
        const float t = ld_stream_f(target + idx);
        const float r = fmaf(cw, s.val, fmaf(ct, t, c0));
        store_dflow<NDIM>(dflow, vol, idx, r, s.g);
    });
}

// MSE only (w_ncc == 0): dL/dw_v = 2 w_mse (w_v - t_v) / n needs no global moments, so the statistics pass is not needed —
// ONE pass samples, writes d loss / d flow (and optionally the warped volume) and reduces sum (w - t)^2 for the loss.
template <int NDIM>
__global__ void __launch_bounds__(256) flow_mse_fused_kernel(const float *__restrict__ moving, const float *__restrict__ target,
                                                              const float *__restrict__ flow, float *__restrict__ dflow,
                                                              float *__restrict__ warped, int D, int H, int W, double w_mse,
                                                              double *__restrict__ ws, float *__restrict__ loss_out)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W;
    const FlowAxes ax = flow_axes(D, H, W);
    const float gm = (float)(2.0 * w_mse / (double)vol);
    float sd[1] = {0.f};
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        const Sample<NDIM> s = sample_zero_pad<NDIM, true, false>(moving, D, H, W, px, py, pz);
        const float t = ld_stream_f(target + idx);
        const float d = s.val - t;
        if (warped) warped[idx] = s.val;
        sd[0] = fmaf(d, d, sd[0]);
        store_dflow<NDIM>(dflow, vol, idx, gm * d, s.g);
    });
    __shared__ double red[kWarps][1];
    if (!grid_sum(sd, red, ws + 8, (unsigned *)(ws + 4)) || threadIdx.x != 0) return;
    const double loss = w_mse * red[0][0] / (double)vol;
    ws[3] = loss;
    if (loss_out) *loss_out = (float)loss;
}

// ---- U-Net head fused with the node (SURVEY.md §8 f-3; reference utils.py:553-557) ---------------------------------
// The reference ends its U-Net with  y = padNd(y, x);  flow = out(y) (1x1 conv);  warp(x, flow).  Here the zero padding
// and the 1x1 convolution are evaluated inside the node's kernels: the forward pass forms flow_k(v) = b_k + sum_c
// W[k][c] * feat_c(v - lo) on the fly (feat: the decoder output, C <= 8 channels of the un-padded size), writes it once
// (Register.theta / deform need it) and accumulates the similarity moments; the backward pass turns d loss / d flow —
// kept in registers, never written — into d feat (cropped), d W and d b.  No padded copy, no separate conv / pad
// kernels and their autograd intermediates.
constexpr int kHeadMaxC = 8;
struct FlowHead {
    const float *feat;        // [C][fd][fh][fw]
    int C, fd, fh, fw;        // un-padded size (fd = 1 in 2-D)
    int lz, ly, lx;           // zeros in front of the data per axis (padNd: the larger half goes AFTER the data)
    const float *Wd, *bd;     // the 1x1 `out` convolution on the DEVICE: [ndim][C], [ndim] (read once per thread)
};
struct HeadWeights { float W[3 * kHeadMaxC]; float b[3]; };
template <int NDIM>
__device__ __forceinline__ HeadWeights head_weights(const FlowHead &h)
{
    HeadWeights w;
#pragma unroll
    for (int i = 0; i < 3 * kHeadMaxC; ++i) w.W[i] = i < NDIM * h.C ? __ldg(h.Wd + i) : 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) w.b[i] = (i < NDIM && h.bd) ? __ldg(h.bd + i) : 0.f;
    return w;
}
template <int NDIM>
__device__ __forceinline__ bool head_index(const FlowHead &h, int x, int y, int z, size_t &fi)
{
    const int fx = x - h.lx, fy = y - h.ly, fz = NDIM == 3 ? z - h.lz : 0;
    if ((unsigned)fx >= (unsigned)h.fw || (unsigned)fy >= (unsigned)h.fh || (unsigned)fz >= (unsigned)h.fd) return false;
    fi = ((size_t)fz * h.fh + fy) * h.fw + fx;
    return true;
}

template <int NDIM>
__global__ void __launch_bounds__(256) flow_head_forward_kernel(const float *__restrict__ moving, const float *__restrict__ target,
                                                                 const FlowHead h, float *__restrict__ flow, int D, int H, int W,
                                                                 double w_mse, double w_ncc, double *ws, float *loss_out)
{
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W, fvol = (size_t)h.fd * h.fh * h.fw;
    const FlowAxes ax = flow_axes(D, H, W);
    float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    const HeadWeights hw = head_weights<NDIM>(h);
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float f[NDIM];
#pragma unroll
        for (int k = 0; k < NDIM; ++k) f[k] = hw.b[k];
        size_t fi;
        if (head_index<NDIM>(h, x, y, z, fi)) {
            for (int c = 0; c < h.C; ++c) {
                const float v = __ldg(h.feat + (size_t)c * fvol + fi);
#pragma unroll
                for (int k = 0; k < NDIM; ++k) f[k] = fmaf(hw.W[k * h.C + c], v, f[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < NDIM; ++k) flow[(size_t)k * vol + idx] = f[k];
        float px, py, pz = 0.f;
        if (NDIM == 3) { pz = flow_pos(ax.z, z, f[0]); py = flow_pos(ax.y, y, f[1]); px = flow_pos(ax.x, x, f[2]); }
        else { py = flow_pos(ax.y, y, f[0]); px = flow_pos(ax.x, x, f[1]); }
        const float w = sample_zero_pad<NDIM, false, false>(moving, D, H, W, px, py, pz).val;
        const float t = ld_stream_f(target + idx);
        s[0] += t; s[1] += w;
        s[2] = fmaf(t, t, s[2]); s[3] = fmaf(w, w, s[3]); s[4] = fmaf(t, w, s[4]);
    });
    __shared__ double red[kWarps][5];
    if (!grid_sum(s, red, ws + 8, (unsigned *)(ws + 4)) || threadIdx.x != 0) return;
    const LossCoef lc = loss_coefficients((double)vol, red[0][0], red[0][1], red[0][2], red[0][3], red[0][4], w_mse, w_ncc);
    ws[0] = lc.cw; ws[1] = lc.ct; ws[2] = lc.c0; ws[3] = lc.loss;
    if (loss_out) *loss_out = (float)lc.loss;
}

// d loss / d flow (registers) -> d feat [C][fd][fh][fw], d W [ndim][C], d b [ndim] (dwb_out: ndim*(C+1) floats, W first)
template <int NDIM>
__global__ void __launch_bounds__(256) flow_head_backward_kernel(const float *__restrict__ moving, const float *__restrict__ target,
                                                                  const float *__restrict__ flow, const FlowHead h,
                                                                  float *__restrict__ dfeat, int D, int H, int W, double *ws,
                                                                  float *__restrict__ dwb_out)
{
    constexpr int NS = NDIM * (kHeadMaxC + 1);
    const size_t vol = (size_t)(NDIM == 3 ? D : 1) * H * W, fvol = (size_t)h.fd * h.fh * h.fw;
    const FlowAxes ax = flow_axes(D, H, W);
    const float cw = (float)ws[0], ct = (float)ws[1], c0 = (float)ws[2];
    float acc[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) acc[i] = 0.f;
    const HeadWeights hw = head_weights<NDIM>(h);
    for_each_voxel(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        float px, py, pz;
        flow_position<NDIM>(flow, vol, idx, x, y, z, ax, px, py, pz);
        const Sample<NDIM> sm = sample_zero_pad<NDIM, true, false>(moving, D, H, W, px, py, pz);
        const float t = ld_stream_f(target + idx);
        const float r = fmaf(cw, sm.val, fmaf(ct, t, c0));
        float df[NDIM];
#pragma unroll
        for (int a = 0; a < NDIM; ++a) df[a] = r * sm.g[NDIM - 1 - a];
#pragma unroll
        for (int a = 0; a < NDIM; ++a) acc[a * (kHeadMaxC + 1) + kHeadMaxC] += df[a];          // d b
        size_t fi;
        if (head_index<NDIM>(h, x, y, z, fi)) {
#pragma unroll
            for (int c = 0; c < kHeadMaxC; ++c) {
                if (c < h.C) {
                    const float v = __ldg(h.feat + (size_t)c * fvol + fi);
                    float g = 0.f;
#pragma unroll
                    for (int a = 0; a < NDIM; ++a) {
                        g = fmaf(hw.W[a * h.C + c], df[a], g);
                        acc[a * (kHeadMaxC + 1) + c] = fmaf(df[a], v, acc[a * (kHeadMaxC + 1) + c]);  // d W
                    }
                    dfeat[(size_t)c * fvol + fi] = g;
                }
            }
        }
    });
    // partials [blocks][NS]: the forward pass is done with the 5-wide rows
    __shared__ double red[kWarps][NS];
    if (!grid_sum(acc, red, ws + 8, (unsigned *)(ws + 4)) || threadIdx.x >= NS) return;
    const int i = threadIdx.x, a = i / (kHeadMaxC + 1), c = i - a * (kHeadMaxC + 1);
    if (c < h.C) dwb_out[a * h.C + c] = (float)red[0][i];
    else if (c == kHeadMaxC) dwb_out[NDIM * h.C + a] = (float)red[0][i];
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_flow_workspace_bytes(void) { return (size_t)(8 + kFlowMaxBlocks * 3 * (kHeadMaxC + 1)) * sizeof(double); }

extern "C" int trb_warp_flow(int ndim, const float *src_dev, const float *flow_dev, float *out_dev, int n_channels,
                             int D, int H, int W, void *stream)
{
    return trb_warp_flow_ex(ndim, src_dev, flow_dev, out_dev, n_channels, D, H, W, 0, stream);
}

extern "C" int trb_warp_flow_ex(int ndim, const float *src_dev, const float *flow_dev, float *out_dev, int n_channels,
                                int D, int H, int W, int flags, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (!src_dev || !flow_dev || !out_dev || n_channels < 1) { set_error("null pointer / n_channels"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (flags & TRB_FLAG_NEAREST) {
        if (ndim == 3) warp_flow_nearest_kernel<3><<<g, 256, 0, s>>>(src_dev, flow_dev, out_dev, n_channels, D, H, W);
        else warp_flow_nearest_kernel<2><<<g, 256, 0, s>>>(src_dev, flow_dev, out_dev, n_channels, 1, H, W);
    } else if (ndim == 3) {
        warp_flow_kernel<3><<<g, 256, 0, s>>>(src_dev, flow_dev, out_dev, n_channels, D, H, W);
    } else {
        warp_flow_kernel<2><<<g, 256, 0, s>>>(src_dev, flow_dev, out_dev, n_channels, 1, H, W);
    }
    return check_cuda(cudaGetLastError(), "warp_flow");
}

extern "C" int trb_warp_flow_vjp(int ndim, const float *src_dev, const float *flow_dev, const float *gout_dev,
                                 float *dflow_dev, int D, int H, int W, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (!src_dev || !flow_dev || !gout_dev || !dflow_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) warp_flow_vjp_kernel<3><<<g, 256, 0, s>>>(src_dev, flow_dev, gout_dev, dflow_dev, D, H, W);
    else warp_flow_vjp_kernel<2><<<g, 256, 0, s>>>(src_dev, flow_dev, gout_dev, dflow_dev, 1, H, W);
    return check_cuda(cudaGetLastError(), "warp_flow_vjp");
}

extern "C" int trb_flow_loss_grad(int ndim, const float *moving_dev, const float *target_dev, const float *flow_dev,
                                  int D, int H, int W, float w_mse, float w_ncc, float *loss_dev, float *dflow_dev,
                                  float *warped_dev_or_null, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (!moving_dev || !target_dev || !flow_dev || !loss_dev || !dflow_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_flow_workspace_bytes()) {
        set_error("workspace too small: need %zu bytes", trb_flow_workspace_bytes());
        return TRB_ERR_WORKSPACE;
    }
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    cudaStream_t s = (cudaStream_t)stream;
    double *ws = (double *)workspace_dev;
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    if (w_ncc == 0.f) {                 // no global moments needed: one fused pass (32 B/voxel instead of 52)
        if (ndim == 3) flow_mse_fused_kernel<3><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, dflow_dev, warped_dev_or_null, D, H, W, w_mse, ws, loss_dev);
        else flow_mse_fused_kernel<2><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, dflow_dev, warped_dev_or_null, 1, H, W, w_mse, ws, loss_dev);
        return check_cuda(cudaGetLastError(), "flow_loss_grad");
    }
    if (ndim == 3) {
        flow_stats_kernel<3><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, warped_dev_or_null, D, H, W, w_mse, w_ncc, ws, loss_dev);
        flow_grad_kernel<3><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, dflow_dev, D, H, W, ws);
    } else {
        flow_stats_kernel<2><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, warped_dev_or_null, 1, H, W, w_mse, w_ncc, ws, loss_dev);
        flow_grad_kernel<2><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, dflow_dev, 1, H, W, ws);
    }
    return check_cuda(cudaGetLastError(), "flow_loss_grad");
}

extern "C" int trb_flow_head_forward(int ndim, const float *moving_dev, const float *target_dev, const float *feat_dev, int C,
                                     int fd, int fh, int fw, const float *w_dev, const float *b_dev, int D, int H, int W,
                                     float w_mse, float w_ncc, float *loss_dev, float *flow_out_dev,
                                     void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (!moving_dev || !target_dev || !feat_dev || !w_dev || !b_dev || !loss_dev || !flow_out_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (C < 1 || C > kHeadMaxC) { set_error("the fused U-Net head handles 1..%d feature channels (got %d)", kHeadMaxC, C); return TRB_ERR_UNSUPPORTED; }
    if (fw > W || fh > H || (ndim == 3 && fd > D) || fw < 1 || fh < 1 || fd < 1) { set_error("feature map larger than the volume"); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_flow_workspace_bytes()) { set_error("workspace too small: need %zu bytes", trb_flow_workspace_bytes()); return TRB_ERR_WORKSPACE; }
    FlowHead h{};
    h.feat = feat_dev; h.C = C; h.fd = ndim == 3 ? fd : 1; h.fh = fh; h.fw = fw;
    // padNd (utils.py:271-277): delta = target - input, hi = ceil(delta / 2) zeros AFTER the data, the rest in front
    auto lo = [](int full, int part) { const int d = full - part; return d - (d + 1) / 2; };
    h.lz = ndim == 3 ? lo(D, fd) : 0; h.ly = lo(H, fh); h.lx = lo(W, fw);
    h.Wd = w_dev; h.bd = b_dev;
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) flow_head_forward_kernel<3><<<g, 256, 0, s>>>(moving_dev, target_dev, h, flow_out_dev, D, H, W, w_mse, w_ncc, (double *)workspace_dev, loss_dev);
    else flow_head_forward_kernel<2><<<g, 256, 0, s>>>(moving_dev, target_dev, h, flow_out_dev, 1, H, W, w_mse, w_ncc, (double *)workspace_dev, loss_dev);
    return check_cuda(cudaGetLastError(), "flow_head_forward");
}

extern "C" int trb_flow_head_backward(int ndim, const float *moving_dev, const float *target_dev, const float *flow_dev,
                                      const float *feat_dev, int C, int fd, int fh, int fw, const float *w_dev, int D, int H, int W,
                                      float *dfeat_dev, float *dwb_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = validate_flow(ndim, D, H, W);
    if (rc) return rc;
    if (!moving_dev || !target_dev || !flow_dev || !feat_dev || !w_dev || !dfeat_dev || !dwb_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (C < 1 || C > kHeadMaxC) { set_error("the fused U-Net head handles 1..%d feature channels (got %d)", kHeadMaxC, C); return TRB_ERR_UNSUPPORTED; }
    if (fw > W || fh > H || (ndim == 3 && fd > D) || fw < 1 || fh < 1 || fd < 1) { set_error("feature map larger than the volume"); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_flow_workspace_bytes()) { set_error("workspace too small"); return TRB_ERR_WORKSPACE; }
    FlowHead h{};
    h.feat = feat_dev; h.C = C; h.fd = ndim == 3 ? fd : 1; h.fh = fh; h.fw = fw;
    auto lo = [](int full, int part) { const int d = full - part; return d - (d + 1) / 2; };
    h.lz = ndim == 3 ? lo(D, fd) : 0; h.ly = lo(H, fh); h.lx = lo(W, fw);
    h.Wd = w_dev; h.bd = nullptr;
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    unsigned g;
    if ((rc = flow_grid(vol, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) flow_head_backward_kernel<3><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, h, dfeat_dev, D, H, W, (double *)workspace_dev, dwb_dev);
    else flow_head_backward_kernel<2><<<g, 256, 0, s>>>(moving_dev, target_dev, flow_dev, h, dfeat_dev, 1, H, W, (double *)workspace_dev, dwb_dev);
    return check_cuda(cudaGetLastError(), "flow_head_backward");
}
