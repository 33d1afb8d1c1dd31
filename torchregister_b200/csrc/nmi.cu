// nmi.cu — SURVEY.md §8 f-1: the NMI/KDE term of the reference's DEFAULT loss (weights .33/.33/.33) as CUDA
// kernels, forward and backward (sm_100a).
//
// Replaces, from the reference (paths relative to /root/reference/src/TorchRegister/):
//   K_gauss / PDF_xis / PDF / get_pdf / NMI            utils.py:18-79
//   NMILoss.forward (nearest resample to 200^n, 2^n chunks of 100^n, |NMI-1|*alpha)   utils.py:224-259
//   and autograd's backward of all of it down to the warped volume.
//
// Semantics kept (all of them quirks of the reference, see oracle/torch_port.py:nmi_loss):
//   * both images are nearest-resampled to 200^n and VIEWED as K = 2^n chunks of P = 100^n consecutive values;
//   * the 256 bin centres are linspace(max, min) (swapped, descending), the range taken over ALL chunks with
//     .item(), i.e. detached; the "joint" density is a 1-D KDE of the concatenation (target chunk, warped chunk)
//     over the joint range, not a 2-D histogram;
//   * kernel exp(-((s-c)/h)^2/2) (its 1/(2 pi), 1/h and 1/P factors cancel in p = pdf/sum(pdf));
//   * E = sum p*log2(p + 1e-10) (negative entropy), MI = E1+E2-EJ, NMI = 2*MI/(E1+E2), loss = alpha*mean|NMI-1|.
//
// Work per epoch (3-D): 8e6 resampled values x 256 bins x (warped: own + joint range, target: joint range) =
// 6.1e9 Gaussians forward + 4.1e9 backward.  That is MUFU.EX2 work (16 lanes/clk/SM -> 4.65e12/s on 148 SMs):
// the roofline of this term is the special-function unit, ~2.2 ms per epoch, not HBM (the three resampled
// arrays are 96 MB).  The target's own marginal is constant over the epochs and computed once (prepare).
// Histograms are reduced in a fixed order (tile partials -> fp64), min/max by order-independent integer
// atomics: results are deterministic.

#include "nmi_shared.cuh"

namespace trb {

constexpr int kTile = 2000;                  // values per histogram block: divides 100^2 and 100^3, 16-byte rows

struct NmiLayout {
    int ndim, K, P, N, tiles;
    size_t off_rs_t, off_rs_w, off_grs, off_part, off_hist, off_gtab, off_range, off_tabs, off_scal, total;
    int S[3];                                // source extent per axis (x, y, z)
};

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static NmiLayout nmi_layout(int ndim, int D, int H, int W)
{
    NmiLayout L{};
    L.ndim = ndim;
    L.K = ndim == 3 ? 8 : 4;
    L.P = ndim == 3 ? kPatch * kPatch * kPatch : kPatch * kPatch;
    L.N = L.K * L.P;
    L.tiles = L.P / kTile;
    L.S[0] = W; L.S[1] = H; L.S[2] = ndim == 3 ? D : 1;
    size_t o = 0;
    L.off_rs_t = o; o = align256(o + (size_t)L.N * 4);
    L.off_rs_w = o; o = align256(o + (size_t)L.N * 4);
    L.off_grs = o; o = align256(o + (size_t)L.N * 4);
    L.off_part = o; o = align256(o + (size_t)3 * L.K * L.tiles * kBins * 4);      // streams: (w,W) (w,J) (t,J|T)
    L.off_hist = o; o = align256(o + (size_t)4 * L.K * kBins * 8);                // fp64: T marginal, W, J(w), J(t)
    L.off_gtab = o; o = align256(o + (size_t)L.K * kBins * 24);                   // [cW|gW|hW|cJ|gJ|hJ][256] per chunk
    L.off_range = o; o = align256(o + 4 * sizeof(int));                           // keys: t_min t_max w_min w_max
    L.off_tabs = o; o = align256(o + (size_t)2 * ((size_t)W + H + (ndim == 3 ? D : 1)) * sizeof(int));
    L.off_scal = o; o = align256(o + 16 * sizeof(double));              // K chunk terms + ticket
    L.total = o;
    return L;
}

__global__ void nmi_reset_kernel(int *keys2)
{
    if (threadIdx.x == 0) { keys2[0] = INT_MAX; keys2[1] = INT_MIN; }
}

// per axis: the range [lo, hi) of resampled indices that read source index x (empty: lo = hi = 0)
__global__ void nmi_tables_kernel(int S, float scale, int *__restrict__ lo, int *__restrict__ hi)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= S) return;
    int l = kRes, h = 0;
    for (int i = 0; i < kRes; ++i)
        if (nearest_src(i, scale, S) == x) { l = min(l, i); h = max(h, i + 1); }
    if (h == 0) l = 0;
    lo[x] = l; hi[x] = h;
}

// F.interpolate(mode='nearest', size=200^n) + global min/max of the resampled values (utils.py:238-250, :45-46)
template <int NDIM>
__global__ void __launch_bounds__(256) nmi_resample_kernel(const float *__restrict__ src, int D, int H, int W, float sz, float sy,
                                                            float sx, float *__restrict__ rs, int *__restrict__ keys2)
{
    const int N = NDIM == 3 ? kRes * kRes * kRes : kRes * kRes;
    float mn = INFINITY, mx = -INFINITY;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < N; i += gridDim.x * 256) {
        const int ix = i % kRes, r = i / kRes;
        const int iy = r % kRes, iz = r / kRes;
        const int x = nearest_src(ix, sx, W), y = nearest_src(iy, sy, H);
        const int z = NDIM == 3 ? nearest_src(iz, sz, D) : 0;
        const float v = __ldg(src + ((size_t)z * H + y) * W + x);
        rs[i] = v;
        mn = fminf(mn, v); mx = fmaxf(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(kFull, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(keys2, float_key(mn));
        atomicMax(keys2 + 1, float_key(mx));
    }
}

// One block = one tile of kTile values of chunk k.  NSETS bin ranges are evaluated on the same staged values (the
// warped stream needs its own range and the joint one).  part[set][(k*tiles+tile)*256 + b].
// Grouped path: lane l of every warp owns bins 8l..8l+7, the 8 warps split the tile's values, partial histograms
// are folded over the warps in a fixed order.  Direct path: thread b owns bin b and walks all values.
template <int NSETS>
__global__ void __launch_bounds__(256) nmi_hist_kernel(const float *__restrict__ rs, int P, int tiles, const int *__restrict__ keys,
                                                        int range0, int range1, float kappa, float h, float *__restrict__ part0,
                                                        float *__restrict__ part1)
{
    __shared__ float4 vals[kTile / 4];
    __shared__ float red[NSETS][8][kBins];
    const int k = blockIdx.x / tiles, tile = blockIdx.x - k * tiles;
    const float4 *g = reinterpret_cast<const float4 *>(rs + (size_t)k * P + (size_t)tile * kTile);
    for (int i = threadIdx.x; i < kTile / 4; i += 256) vals[i] = g[i];
    float s0, e0, s1 = 0.f, e1 = 0.f;
    bin_range(keys, range0, s0, e0);
    if (NSETS == 2) bin_range(keys, range1, s1, e1);
    const float d0 = bin_delta(keys, range0, kappa), d1 = NSETS == 2 ? bin_delta(keys, range1, kappa) : 0.f;
    const size_t o = (size_t)blockIdx.x * kBins + threadIdx.x;
    __syncthreads();
    if (moment_ok(keys, NSETS == 2 ? range1 : range0, h)) {        // range1 (joint) contains range0
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const float m0 = 0.5f * (s0 + e0), m1 = 0.5f * (s1 + e1), inv_h = 1.f / h;
        float a0[kMom], a1[kMom];
#pragma unroll
        for (int m = 0; m < kMom; ++m) { a0[m] = 0.f; a1[m] = 0.f; }
        const float *v = reinterpret_cast<const float *>(vals);
        for (int i = threadIdx.x; i < kTile; i += 256) {
            hermite_chain<kMom>(v[i], m0, inv_h, [&](int m, float x) { a0[m] += x; });
            if (NSETS == 2) hermite_chain<kMom>(v[i], m1, inv_h, [&](int m, float x) { a1[m] += x; });
        }
#pragma unroll
        for (int m = 0; m < kMom; ++m) {
            const float x0 = warp_sum(a0[m]), x1 = NSETS == 2 ? warp_sum(a1[m]) : 0.f;
            if (lane == 0) { red[0][warp][m] = x0; if (NSETS == 2) red[1][warp][m] = x1; }
        }
        __syncthreads();
        float h0 = 0.f, h1 = 0.f;
        if (threadIdx.x < kMom) {
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                h0 += red[0][w][threadIdx.x];
                if (NSETS == 2) h1 += red[1][w][threadIdx.x];
            }
        }
        part0[o] = h0;                                               // columns >= kMom stay 0
        if (NSETS == 2) part1[o] = h1;
        return;
    }
    if (group_ok(d0) && group_ok(d1)) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const float c0 = bin_centre(s0, e0, kGroup * lane), c1 = NSETS == 2 ? bin_centre(s1, e1, kGroup * lane) : 0.f;
        float w0[kGroup], w1[kGroup], a0[kGroup], a1[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) {
            w0[j] = ex2_approx(-(float)(j * j) * d0 * d0);
            w1[j] = ex2_approx(-(float)(j * j) * d1 * d1);
            a0[j] = 0.f; a1[j] = 0.f;
        }
        const float r0 = 2.f * d0, r1 = 2.f * d1;
        for (int i = warp; i < kTile / 4; i += 8) {
            const float4 v = vals[i];
            const float sv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                {
                    const float t0 = (sv[q] - c0) * kappa;          // subtract first: s*kappa - c*kappa loses the low bits for 12/16-bit data
                    float pw = ex2_approx(-t0 * t0);
                    const float rho = ex2_approx(fminf(t0 * r0, 60.f));
                    a0[0] += pw;
#pragma unroll
                    for (int j = 1; j < kGroup; ++j) { pw *= rho; a0[j] = fmaf(pw, w0[j], a0[j]); }
                }
                if (NSETS == 2) {
                    const float t1 = (sv[q] - c1) * kappa;
                    float pw = ex2_approx(-t1 * t1);
                    const float rho = ex2_approx(fminf(t1 * r1, 60.f));
                    a1[0] += pw;
#pragma unroll
                    for (int j = 1; j < kGroup; ++j) { pw *= rho; a1[j] = fmaf(pw, w1[j], a1[j]); }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kGroup; ++j) {
            red[0][warp][kGroup * lane + j] = a0[j];
            if (NSETS == 2) red[1][warp][kGroup * lane + j] = a1[j];
        }
        __syncthreads();
        float h0 = 0.f, h1 = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            h0 += red[0][w][threadIdx.x];
            if (NSETS == 2) h1 += red[1][w][threadIdx.x];
        }
        part0[o] = h0;
        if (NSETS == 2) part1[o] = h1;
        return;
    }
    const float c0 = bin_centre(s0, e0, threadIdx.x);
    const float c1 = NSETS == 2 ? bin_centre(s1, e1, threadIdx.x) : 0.f;
    float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int i = 0; i < kTile / 4; ++i) {
        const float4 v = vals[i];
        const float sv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float t0 = (sv[j] - c0) * kappa;
            a0[j] += ex2_approx(-t0 * t0);
            if (NSETS == 2) {
                const float t1 = (sv[j] - c1) * kappa;
                a1[j] += ex2_approx(-t1 * t1);
            }
        }
    }
    part0[o] = (a0[0] + a0[1]) + (a0[2] + a0[3]);
    if (NSETS == 2) part1[o] = (a1[0] + a1[1]) + (a1[2] + a1[3]);
}

// hist[k][b] = sum over tiles, fixed order, fp64.  grid = (K, n_streams).  16 columns x 16 tile lanes at a time;
// slots in moment form only carry kMom columns.
__global__ void __launch_bounds__(256) nmi_reduce_kernel(const float *__restrict__ part, int tiles, size_t stream_stride,
                                                          double *__restrict__ hist, size_t hist_stride,
                                                          const int *__restrict__ keys, int range_first, int range_rest, float h)
{
    __shared__ double sh[16][17];
    const int k = blockIdx.x;
    const int cols = moment_ok(keys, blockIdx.y == 0 ? range_first : range_rest, h) ? 16 : kBins;
    const float *p = part + (size_t)blockIdx.y * stream_stride + (size_t)k * tiles * kBins;
    double *out = hist + (size_t)blockIdx.y * hist_stride + (size_t)k * kBins;
    const int col = threadIdx.x & 15, lane = threadIdx.x >> 4;
    for (int c0 = 0; c0 < cols; c0 += 16) {
        double acc = 0.0;
        for (int t = lane; t < tiles; t += 16) acc += (double)p[(size_t)t * kBins + c0 + col];
        sh[lane][col] = acc;
        __syncthreads();
        if (threadIdx.x < 16) {
            double v = 0.0;
#pragma unroll
            for (int l = 0; l < 16; ++l) v += sh[l][threadIdx.x];
            out[c0 + threadIdx.x] = v;
        }
        __syncthreads();
    }
}

// Entropies, NMI, loss and the table the backward needs.  One block per chunk, thread b = bin b; the last block to
// finish adds the K chunk terms in order.
// hist layout: [0] target marginal (prepare), [1] warped marginal, [2] joint (warped half), [3] joint (target half);
// a slot computed in moment form holds M_0..M_11 in its first columns and is expanded to bins here (fp64, with the
// exact fp32 bin centres of torch.linspace).
__global__ void __launch_bounds__(256) nmi_epilogue_kernel(const double *__restrict__ hist, int K, const int *__restrict__ keys,
                                                            float kappa, float h, double alpha, double weight,
                                                            float *__restrict__ gtab, double *__restrict__ scal,
                                                            double *__restrict__ loss_out)
{
    __shared__ double sh[kWarps][1];
    const int b = threadIdx.x, k = blockIdx.x;
    const size_t hs = (size_t)K * kBins;
    const double eps = 1e-10, ln2 = 0.6931471805599453;
    float sT, eT, sW, eW, sJ, eJ;
    bin_range(keys, kRangeT, sT, eT);
    bin_range(keys, kRangeW, sW, eW);
    bin_range(keys, kRangeJ, sJ, eJ);
    const float cT = bin_centre(sT, eT, b), cW = bin_centre(sW, eW, b), cJ = bin_centre(sJ, eJ, b);
    const bool momT = moment_ok(keys, kRangeT, h), momWJ = moment_ok(keys, kRangeJ, h);
    const float midT = range_mid(keys, kRangeT), midW = range_mid(keys, kRangeW), midJ = range_mid(keys, kRangeJ);
    const double yT = ((double)cT - (double)midT) / (double)h, yW = ((double)cW - (double)midW) / (double)h;
    const double yJ = ((double)cJ - (double)midJ) / (double)h;
    // grouped backward: the constant 2^-(j d)^2 of bin b = b0 + j rides in the coefficient
    const float dW = bin_delta(keys, kRangeW, kappa), dJ = bin_delta(keys, kRangeJ, kappa);
    const int j = b & (kGroup - 1);
    const double wW = group_ok(dW) ? exp2(-(double)(j * j) * (double)dW * (double)dW) : 1.0;
    const double wJ = group_ok(dJ) ? exp2(-(double)(j * j) * (double)dJ * (double)dJ) : 1.0;
    const double *r1 = hist + (size_t)k * kBins, *r2 = hist + hs + (size_t)k * kBins;
    const double *r3 = hist + 2 * hs + (size_t)k * kBins, *r4 = hist + 3 * hs + (size_t)k * kBins;
    const double H1 = momT ? expand_moments(r1, yT) : r1[b];
    const double H2 = momWJ ? expand_moments(r2, yW) : r2[b];
    const double HJ = momWJ ? expand_moments(r3, yJ) + expand_moments(r4, yJ) : r3[b] + r4[b];
    const double S1 = block_sum_all(H1, sh), S2 = block_sum_all(H2, sh), SJ = block_sum_all(HJ, sh);
    const double p1 = H1 / S1, p2 = H2 / S2, pj = HJ / SJ;
    const double l2 = log2(p2 + eps), lj = log2(pj + eps);
    const double E1 = block_sum_all(p1 * log2(p1 + eps), sh);
    const double E2 = block_sum_all(p2 * l2, sh), EJ = block_sum_all(pj * lj, sh);
    const double d2 = l2 + p2 / ((p2 + eps) * ln2), dj = lj + pj / ((pj + eps) * ln2);      // dE/dp_b
    const double A2 = block_sum_all(p2 * d2, sh), AJ = block_sum_all(pj * dj, sh);
    const double den = E1 + E2, mi = den - EJ;
    const double nmi = 2.0 * mi / den;
    const double dev = nmi - 1.0;
    const double dl = weight * alpha / (double)K * (dev > 0.0 ? 1.0 : (dev < 0.0 ? -1.0 : 0.0));
    const double dn_e2 = 2.0 / den - 2.0 * mi / (den * den), dn_ej = -2.0 / den;
    // dL/dH_b = dl * dn * (dE/dp_b - sum_c p_c dE/dp_c) / S
    const double G2 = dl * dn_e2 * (d2 - A2) / S2, GJ = dl * dn_ej * (dj - AJ) / SJ;
    float *tab = gtab + (size_t)k * 6 * kBins;       // [cW | gW | hW | cJ | gJ | hJ][256]
    if (momWJ) {
        // Gamma_m = sum_b G_b y_b^m / m!, stored as -Gamma_m/h in gW[m] / gJ[m]; the range centres in cW[0] / cJ[0]
        double tw = G2, tj = GJ;
        for (int m = 0; m < kMom; ++m) {
            const double gw = block_sum_all(tw, sh), gj = block_sum_all(tj, sh);
            if (b == 0) { tab[kBins + m] = (float)(-gw / (double)h); tab[4 * kBins + m] = (float)(-gj / (double)h); }
            tw *= yW / (double)(m + 1); tj *= yJ / (double)(m + 1);
        }
        if (b == 0) { tab[0] = midW; tab[3 * kBins] = midJ; }
    } else {
        // dH_b/ds = exp(-u^2/2) * (-u/h), u = t/(kappa*h);  h-arrays: j*g for the grouped form
        const double to_s = -1.0 / ((double)kappa * (double)h * (double)h);
        const double g2 = G2 * to_s, gj = GJ * to_s;
        tab[b] = cW; tab[kBins + b] = (float)(g2 * wW); tab[2 * kBins + b] = (float)((double)j * g2 * wW);
        tab[3 * kBins + b] = cJ; tab[4 * kBins + b] = (float)(gj * wJ); tab[5 * kBins + b] = (float)((double)j * gj * wJ);
    }
    // chunk term -> scal[k]; the last block adds them in chunk order
    unsigned *ticket = reinterpret_cast<unsigned *>(scal + 8);
    if (b == 0) __stcg(scal + k, fabs(dev));
    if (last_to_arrive(ticket, K) && b == 0) {
        double loss = 0.0;
        for (int c = 0; c < K; ++c) loss += __ldcg(scal + c);
        *loss_out = weight * alpha * loss / (double)K;
        *ticket = 0u;
    }
}

// d loss / d (resampled warped value): 2 x 256 Gaussians per value, grouped like the histogram when the bin spacing
// allows (see kGroup).  grid = (ceil(P/256), K)
__device__ __forceinline__ float nmi_grad_set(const float *__restrict__ c, const float *__restrict__ gw, const float *__restrict__ hw,
                                              float s, float kappa, float d, bool grouped)
{
    float acc = 0.f;
    if (grouped) {
        // sum_j g_j t_j P_j with t_j = t0 - j d  =  t0 * sum_j g_j P_j - d * sum_j (j g_j) P_j: 3 operations per bin
        const float r = 2.f * d;
#pragma unroll 2
        for (int b0 = 0; b0 < kBins; b0 += kGroup) {
            const float t = (s - c[b0]) * kappa;
            float pw = ex2_approx(-t * t);
            const float rho = ex2_approx(fminf(t * r, 60.f));
            const float4 ga = *reinterpret_cast<const float4 *>(gw + b0), gb = *reinterpret_cast<const float4 *>(gw + b0 + 4);
            const float4 ha = *reinterpret_cast<const float4 *>(hw + b0), hb = *reinterpret_cast<const float4 *>(hw + b0 + 4);
            const float gq[kGroup] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
            const float hq[kGroup] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
            float A = gq[0] * pw, B = 0.f;
#pragma unroll
            for (int j = 1; j < kGroup; ++j) {
                pw *= rho;
                A = fmaf(gq[j], pw, A);
                B = fmaf(hq[j], pw, B);
            }
            acc = fmaf(t, A, fmaf(-d, B, acc));
        }
    } else {
#pragma unroll 4
        for (int b = 0; b < kBins; ++b) {
            const float t = (s - c[b]) * kappa;
            acc = fmaf(gw[b] * t, ex2_approx(-t * t), acc);
        }
    }
    return acc;
}

__global__ void __launch_bounds__(256) nmi_grad_kernel(const float *__restrict__ rs_w, int P, const float *__restrict__ gtab,
                                                        const int *__restrict__ keys, float kappa, float h, float *__restrict__ grs)
{
    __shared__ __align__(16) float tab[6 * kBins];
    const int k = blockIdx.y;
    const bool mom = moment_ok(keys, kRangeJ, h);
    const float *gt = gtab + (size_t)k * 6 * kBins;
    if (mom) {                                   // 2 x (centre + kMom coefficients) instead of the 6 KB table
        if (threadIdx.x <= kMom) { tab[kBins - 1 + threadIdx.x] = gt[kBins - 1 + threadIdx.x]; tab[4 * kBins - 1 + threadIdx.x] = gt[4 * kBins - 1 + threadIdx.x]; }
        if (threadIdx.x == 0) { tab[0] = gt[0]; tab[3 * kBins] = gt[3 * kBins]; }
    } else {
        for (int i = threadIdx.x; i < 6 * kBins; i += 256) tab[i] = gt[i];
    }
    const float dW = bin_delta(keys, kRangeW, kappa), dJ = bin_delta(keys, kRangeJ, kappa);
    __syncthreads();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= P) return;
    const float s = rs_w[(size_t)k * P + i];
    if (mom) {
        float acc = 0.f;
        const float inv_h = 1.f / h;
        hermite_chain<kMom + 1>(s, tab[0], inv_h, [&](int m, float x) { if (m > 0) acc = fmaf(tab[kBins + m - 1], x, acc); });
        hermite_chain<kMom + 1>(s, tab[3 * kBins], inv_h, [&](int m, float x) { if (m > 0) acc = fmaf(tab[4 * kBins + m - 1], x, acc); });
        grs[(size_t)k * P + i] = acc;
        return;
    }
    grs[(size_t)k * P + i] = nmi_grad_set(tab, tab + kBins, tab + 2 * kBins, s, kappa, dW, group_ok(dW)) +
                             nmi_grad_set(tab + 3 * kBins, tab + 4 * kBins, tab + 5 * kBins, s, kappa, dJ, group_ok(dJ));
}

// backward of the nearest resample: every source voxel sums the resampled positions that read it (fixed order)
template <int NDIM>
__global__ void __launch_bounds__(256) nmi_scatter_kernel(const float *__restrict__ grs, int D, int H, int W,
                                                           const int *__restrict__ tabs, float *__restrict__ gout)
{
    const int *xlo = tabs, *xhi = tabs + W, *ylo = tabs + 2 * W, *yhi = tabs + 2 * W + H;
    const int *zlo = tabs + 2 * W + 2 * H, *zhi = zlo + (NDIM == 3 ? D : 1);
    for_each_voxel<1>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        const int x0 = xlo[x], x1 = xhi[x], y0 = ylo[y], y1 = yhi[y];
        const int z0 = NDIM == 3 ? zlo[z] : 0, z1 = NDIM == 3 ? zhi[z] : 1;
        float acc = 0.f;
        for (int iz = z0; iz < z1; ++iz)
            for (int iy = y0; iy < y1; ++iy)
                for (int ix = x0; ix < x1; ++ix) acc += grs[((size_t)iz * kRes + iy) * kRes + ix];
        gout[idx] = acc;
    });
}

static int nmi_validate(int ndim, int D, int H, int W, const void *ws, size_t ws_bytes)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (H < 1 || W < 1 || (ndim == 3 && D < 1)) { set_error("bad volume shape %dx%dx%d", D, H, W); return TRB_ERR_ARG; }
    if ((unsigned long long)(ndim == 3 ? D : 1) * H * W >= (1ull << 31)) { set_error("volume too large"); return TRB_ERR_UNSUPPORTED; }
    const NmiLayout L = nmi_layout(ndim, D, H, W);
    if (!ws || ws_bytes < L.total) { set_error("workspace too small: need %zu bytes", L.total); return TRB_ERR_WORKSPACE; }
    return TRB_OK;
}

static float nmi_kappa(float h) { return (float)(sqrt(0.5 * 1.4426950408889634) / (double)h); }   // exp(-u^2/2) = 2^-(kappa*(s-c))^2

template <int NDIM>
static void nmi_resample(const float *src, int D, int H, int W, float *rs, int *keys2, cudaStream_t s)
{
    const int N = NDIM == 3 ? kRes * kRes * kRes : kRes * kRes;
    // torch computes the scale in fp32 as input_size / output_size (UpSample.h compute_scales_value)
    const float sz = (float)(NDIM == 3 ? D : 1) / (float)kRes, sy = (float)H / (float)kRes, sx = (float)W / (float)kRes;
    int nb = (N + 255) / 256;
    if (nb > 148 * 16) nb = 148 * 16;
    nmi_reset_kernel<<<1, 32, 0, s>>>(keys2);
    nmi_resample_kernel<NDIM><<<nb, 256, 0, s>>>(src, D, H, W, sz, sy, sx, rs, keys2);
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_nmi_workspace_bytes(int ndim, int D, int H, int W)
{
    if ((ndim != 2 && ndim != 3) || H < 1 || W < 1 || (ndim == 3 && D < 1)) return 0;
    return nmi_layout(ndim, D, H, W).total;
}

extern "C" int trb_nmi_prepare(int ndim, const float *target_dev, int D, int H, int W, float bandwidth,
                               void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = nmi_validate(ndim, D, H, W, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!target_dev) { set_error("null target"); return TRB_ERR_ARG; }
    if (!(bandwidth > 0.f)) { set_error("bandwidth must be positive"); return TRB_ERR_ARG; }
    const NmiLayout L = nmi_layout(ndim, D, H, W);
    char *ws = (char *)workspace_dev;
    float *rs_t = (float *)(ws + L.off_rs_t), *part = (float *)(ws + L.off_part);
    double *hist = (double *)(ws + L.off_hist);
    int *keys = (int *)(ws + L.off_range), *tabs = (int *)(ws + L.off_tabs);
    cudaStream_t s = (cudaStream_t)stream;
    // resampled-index ranges per source index, axis order x, y, z
    int *t = tabs;
    for (int a = 0; a < ndim; ++a) {
        const int S = L.S[a];
        nmi_tables_kernel<<<(S + 127) / 128, 128, 0, s>>>(S, (float)S / (float)kRes, t, t + S);
        t += 2 * S;
    }
    if (ndim == 3) nmi_resample<3>(target_dev, D, H, W, rs_t, keys, s);
    else nmi_resample<2>(target_dev, 1, H, W, rs_t, keys, s);
    // the target's own marginal (range = target range): constant over the epochs
    const size_t stream_stride = (size_t)L.K * L.tiles * kBins;
    nmi_hist_kernel<1><<<L.K * L.tiles, 256, 0, s>>>(rs_t, L.P, L.tiles, keys, kRangeT, kRangeT, nmi_kappa(bandwidth), bandwidth,
                                                     part + 2 * stream_stride, nullptr);
    cudaMemsetAsync(ws + L.off_scal, 0, 16 * sizeof(double), s);        // chunk terms + the epilogue's ticket
    nmi_reduce_kernel<<<dim3(L.K, 1), 256, 0, s>>>(part + 2 * stream_stride, L.tiles, stream_stride, hist, (size_t)L.K * kBins, keys,
                                                 kRangeT, kRangeT, bandwidth);
    return check_cuda(cudaGetLastError(), "nmi_prepare");
}

extern "C" int trb_nmi_loss_grad(int ndim, const float *warped_dev, int D, int H, int W, float bandwidth, float alpha,
                                 float weight, double *loss_dev, float *gout_dev, void *workspace_dev,
                                 size_t workspace_bytes, void *stream)
{
    int rc = nmi_validate(ndim, D, H, W, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!warped_dev || !loss_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (!(bandwidth > 0.f)) { set_error("bandwidth must be positive"); return TRB_ERR_ARG; }
    const NmiLayout L = nmi_layout(ndim, D, H, W);
    char *ws = (char *)workspace_dev;
    float *rs_t = (float *)(ws + L.off_rs_t), *rs_w = (float *)(ws + L.off_rs_w), *grs = (float *)(ws + L.off_grs);
    float *part = (float *)(ws + L.off_part);
    double *hist = (double *)(ws + L.off_hist);
    float *gtab = (float *)(ws + L.off_gtab);
    int *keys = (int *)(ws + L.off_range), *tabs = (int *)(ws + L.off_tabs);
    cudaStream_t s = (cudaStream_t)stream;
    const float kappa = nmi_kappa(bandwidth);
    const size_t stream_stride = (size_t)L.K * L.tiles * kBins, hs = (size_t)L.K * kBins;
    if (ndim == 3) nmi_resample<3>(warped_dev, D, H, W, rs_w, keys + 2, s);
    else nmi_resample<2>(warped_dev, 1, H, W, rs_w, keys + 2, s);
    nmi_hist_kernel<2><<<L.K * L.tiles, 256, 0, s>>>(rs_w, L.P, L.tiles, keys, kRangeW, kRangeJ, kappa, bandwidth, part, part + stream_stride);
    nmi_hist_kernel<1><<<L.K * L.tiles, 256, 0, s>>>(rs_t, L.P, L.tiles, keys, kRangeJ, kRangeJ, kappa, bandwidth, part + 2 * stream_stride, nullptr);
    nmi_reduce_kernel<<<dim3(L.K, 3), 256, 0, s>>>(part, L.tiles, stream_stride, hist + hs, hs, keys, kRangeJ, kRangeJ, bandwidth);
    nmi_epilogue_kernel<<<L.K, 256, 0, s>>>(hist, L.K, keys, kappa, bandwidth, (double)alpha, (double)weight, gtab,
                                           (double *)(ws + L.off_scal), loss_dev);
    if (gout_dev) {
        nmi_grad_kernel<<<dim3((L.P + 255) / 256, L.K), 256, 0, s>>>(rs_w, L.P, gtab, keys, kappa, bandwidth, grs);
        const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
        size_t nb = (vol + 255) / 256;
        if (nb > 148 * 16) nb = 148 * 16;
        if (ndim == 3) nmi_scatter_kernel<3><<<(unsigned)nb, 256, 0, s>>>(grs, D, H, W, tabs, gout_dev);
        else nmi_scatter_kernel<2><<<(unsigned)nb, 256, 0, s>>>(grs, 1, H, W, tabs, gout_dev);
    }
    return check_cuda(cudaGetLastError(), "nmi_loss_grad");
}
