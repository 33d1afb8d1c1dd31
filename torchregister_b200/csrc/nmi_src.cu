// nmi_src.cu — SURVEY.md §8 f-1, second evaluation of the NMI/KDE term of the reference's DEFAULT loss: in SOURCE-voxel
// space, batched over pairs, plus the default-loss epoch loop as ONE C-ABI call (no host code per epoch).
//
// Replaces, from the reference (paths relative to /root/reference/src/TorchRegister/):
//   NMILoss.forward / NMI / get_pdf                     utils.py:18-79, 224-259   (and autograd's backward of it)
//   the epoch loop with the default criterions          warpings.py:123-159 (affine), :60-93 (rigid)
//
// nmi.cu materialises the nearest-resampled 200^3 arrays (3 x 32 MB per pair) and walks them four times per epoch
// (resample, moments, gradient, scatter: 0.24 ms).  When the value range is narrow against the bandwidth (<= 0.6 h — images
// normalised to [0,1] with the default bandwidth 3, as the README does; nmi.cu's "moment" regime) none of that is needed:
//   * the nearest resample reads source voxel (x,y,z) exactly mx(x)*my(y)*mz(z) times, and the chunk of a resampled
//     value only depends on its slice: a chunk's KDE is a sum over SOURCE voxels weighted by mx*my*mz_k(z);
//   * with u = (s - mid)/h and y = (c - mid)/h:  exp(-(u-y)^2/2) = e^{-y^2/2} e^{-u^2/2} sum_m (u y)^m / m!, so the KDE at
//     ANY bin centre is e^{-y^2/2} sum_m (y^m/m!) N_m with N_m = sum w e^{-u^2/2} u^m: ONE set of 8 moments per chunk about
//     a FIXED centre `mid` serves the warped marginal (own range), the joint range and — for the target, whose moments
//     are then constant over the epochs — both of its ranges.  |u|,|y| <= 0.3: the series is cut at (0.09)^8/8! = 1e-13;
//   * the backward is a pointwise function of the warped value: (1/h) e^{-u^2/2} sum_m c_m u^m, one polynomial per chunk.
// Per epoch and pair: one pass over the warped volume (8 moments per chunk piece, fp64 partials, fixed order), one small
// block per chunk (entropies, NMI, loss, polynomial — the arithmetic of nmi_epilogue_kernel), one pass writing
// d loss / d warped.  The caller supplies value bounds [lo, hi] that hold for both volumes and every warp of the moving
// one (trilinear samples with zero padding are convex combinations of voxel values and 0); the loss is NaN if a
// value ever leaves them.  Results equal nmi.cu's moment form up to both truncations (2e-11) and summation order.
#include "nmi_shared.cuh"
#include "affine_shared.cuh"

namespace trb {

constexpr int kMomPad = 16;                  // moment rows are padded to 16 columns
constexpr int kPow = 8;                      // power moments per chunk (series in u*y, |u*y| <= 0.09: (0.09)^8/8! = 1e-13)
constexpr int kMaxChunks = 8;                // 3-D: 200^3 viewed as 8 chunks of 100^3 = 25 slices of 200x200 each;
                                             // 2-D: 200^2 as 4 chunks of 100^2 = 50 rows of 200 each
// A 2-D image [H][W] is handled as the volume [H][1][W]: the chunks cut its rows like they cut the slices of a volume, and
// the 200 resampled copies of the single "row" of a slice multiply every weight by the same constant, which cancels in the
// normalised histograms and in the gradient.
struct SrcDims { int K, D, H, W; };
static SrcDims src_dims(int ndim, int D, int H, int W)
{
    return ndim == 3 ? SrcDims{8, D, H, W} : SrcDims{4, H, 1, W};
}

struct SrcLayout {
    int B;                                   // blocks (partial rows) per chunk in the moments pass
    int GB;                                  // blocks per slice in the gradient pass
    size_t off_keys, off_tabs, off_mxy, off_momT, off_part, off_gtab, off_scal, off_mom, off_mom2, off_extra, off_theta, total;
};

constexpr int kMaxChunkSlices = 256;         // source slices (rows in 2-D) one chunk can read
constexpr int kMomBlocks = 74;               // 8 chunks x 74 = 592 = 4 blocks on each of the 148 SMs: one wave per pair
constexpr int kBatch = 8;                    // values per thread whose loads are in flight together
constexpr int kGradSeg = 256 * kBatch * 2;   // voxels per block of the gradient pass

static size_t align256s(size_t v) { return (v + 255) & ~(size_t)255; }

static SrcLayout src_layout(int n_pairs, int K, int D, int H, int W)
{
    SrcLayout L{};
    const size_t vol = (size_t)D * H * W, hw = (size_t)H * W;
    L.B = (int)(vol / K / (256 * kBatch));
    if (L.B < 1) L.B = 1;
    if (L.B > kMomBlocks) L.B = kMomBlocks;
    L.GB = (int)((hw + kGradSeg - 1) / kGradSeg);
    size_t o = 0;
    const size_t n = (size_t)n_pairs;
    L.off_keys = o; o = align256s(o + n * 4 * sizeof(int));                                   // t_min t_max w_min w_max
    L.off_tabs = o; o = align256s(o + ((size_t)W + H + 2 * (size_t)D) * sizeof(int));        // mulx | muly | zlo | zhi
    L.off_mxy = o; o = align256s(o + hw * sizeof(unsigned short));                            // mulx * muly per (y, x)
    L.off_momT = o; o = align256s(o + n * kMaxChunks * kMomPad * sizeof(double));
    L.off_part = o; o = align256s(o + n * kMaxChunks * (size_t)L.B * kMomPad * sizeof(double));
    L.off_gtab = o; o = align256s(o + n * kMaxChunks * kMomPad * sizeof(float));
    L.off_scal = o; o = align256s(o + n * 16 * sizeof(double));                               // K chunk terms + ticket
    L.off_mom = o; o = align256s(o + n * TRB_MOMENTS * sizeof(double));
    L.off_mom2 = o; o = align256s(o + n * TRB_MOMENTS * sizeof(double));
    L.off_extra = o; o = align256s(o + n * 13 * sizeof(double));
    L.off_theta = o; o = align256s(o + n * 12 * sizeof(float));
    L.total = o;
    return L;
}

// how many resampled indices read source index i of each axis; for z also the range itself (chunks cut it)
__global__ void nmi_src_tables_kernel(int W, int H, int D, int *__restrict__ tabs)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W + H + D) return;
    const int axis = i < W ? 0 : (i < W + H ? 1 : 2);
    const int S = axis == 0 ? W : (axis == 1 ? H : D), x = axis == 0 ? i : (axis == 1 ? i - W : i - W - H);
    const float scale = (float)S / (float)kRes;     // torch computes the scale in fp32 as input_size / output_size
    int l = kRes, h = 0;
    for (int j = 0; j < kRes; ++j)
        if (nearest_src(j, scale, S) == x) { l = min(l, j); h = max(h, j + 1); }
    if (h == 0) l = 0;
    if (axis < 2) tabs[i] = h - l;                  // the indices reading x are consecutive (the map is monotone)
    else { tabs[W + H + x] = l; tabs[W + H + D + x] = h; }
}

__global__ void nmi_src_plane_kernel(int W, int H, const int *__restrict__ tabs, unsigned short *__restrict__ mxy)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < W * H) mxy[i] = (unsigned short)(tabs[i % W] * tabs[W + i / W]);      // <= 200 * 200
}

__device__ __forceinline__ int chunk_overlap(int zl, int zh, int k, int cs)
{
    return max(0, min(zh, (k + 1) * cs) - max(zl, k * cs));
}

__global__ void nmi_src_reset_kernel(int *keys, int n_pairs, int off)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pairs) { keys[4 * i + off] = INT_MAX; keys[4 * i + off + 1] = INT_MIN; }
}

// source slices [zf, zl] read by chunk k's 25 resampled slices (the resample map is monotone)
__device__ __forceinline__ void chunk_slices(int k, int cs, int D, int &zf, int &zl)
{
    const float sz = (float)D / (float)kRes;
    zf = nearest_src(k * cs, sz, D);
    zl = nearest_src((k + 1) * cs - 1, sz, D);
}

// i = q * hw + r, 0 <= r < hw, for 0 <= i < 2^31 (float estimate, corrected)
__device__ __forceinline__ void divmod_hw(int i, int hw, float inv_hw, int &q, int &r)
{
    q = (int)((float)i * inv_hw);
    r = i - q * hw;
    if (r < 0) { --q; r += hw; }
    else if (r >= hw) { ++q; r -= hw; }
}

// weighted power moments of one value: a[m] += w * e^{-u^2/2} * u^m, m < kPow
__device__ __forceinline__ void power_chain(float v, float fm, float inv_h, float c0, float (&a)[kPow])
{
    const float u = fmaf(v, inv_h, c0);                        // (v - mid) / h
    float pw = fm * ex2_approx(-0.72134752f * u * u);          // w * exp(-u^2/2)
    a[0] += pw;
#pragma unroll
    for (int m = 1; m < kPow; ++m) { pw *= u; a[m] += pw; }
}

// grid (B, K, pairs): the slices of chunk k are one contiguous run of memory, cut evenly over the B blocks; every voxel
// enters with weight mx*my*mz_k(z).  part[pair][k][b][0..kPow) in fp64, folded in a fixed order.  VEC: H*W % 4 == 0 and
// 16-byte aligned volumes — four voxels per load.
template <bool VEC>
__global__ void __launch_bounds__(256) nmi_src_moments_kernel(const float *__restrict__ vol, long long pair_stride, int D, int H, int W,
                                                               const int *__restrict__ tabs, const unsigned short *__restrict__ mxy,
                                                               float mid, float inv_h, double *__restrict__ part,
                                                               int *__restrict__ keys, int key_off)
{
    __shared__ double red[kWarps][kPow];
    __shared__ float rmn[8], rmx[8];
    __shared__ int mzk[kMaxChunkSlices];
    const int b = blockIdx.x, B = gridDim.x, k = blockIdx.y, K = gridDim.y, cs = kRes / K, pair = blockIdx.z;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int *zlo = tabs + W + H, *zhi = zlo + D;
    int zf, zl;
    chunk_slices(k, cs, D, zf, zl);
    for (int z = zf + threadIdx.x; z <= zl; z += 256) mzk[z - zf] = chunk_overlap(zlo[z], zhi[z], k, cs);
    __syncthreads();
    constexpr int V = VEC ? 4 : 1, U = VEC ? 2 : 8;            // voxels per item, items per thread in flight
    const int hw = H * W / V;                                   // items per slice
    const float inv_hw = 1.f / (float)hw;
    const long long n = (long long)(zl - zf + 1) * hw;
    const int i0 = (int)(n * b / B), i1 = (int)(n * (b + 1) / B);
    const float *src = vol + (size_t)pair * pair_stride + (size_t)zf * hw * V;
    const float c0 = -mid * inv_h;
    float a[kPow];
#pragma unroll
    for (int m = 0; m < kPow; ++m) a[m] = 0.f;
    float mn = INFINITY, mx = -INFINITY;
    for (int base = i0 + threadIdx.x; base < i1; base += 256 * U) {
        float v[U][V], fm[U][V];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int i = min(base + 256 * j, i1 - 1);
            const bool live = base + 256 * j < i1;
            int q, r;
            divmod_hw(i, hw, inv_hw, q, r);
            const int mz = live ? mzk[q] : 0;
            if (VEC) {
                const ushort4 m4 = *reinterpret_cast<const ushort4 *>(mxy + 4 * r);
                const float4 v4 = __ldg(reinterpret_cast<const float4 *>(src) + i);
                fm[j][0] = (float)(m4.x * mz); fm[j][1 % V] = (float)(m4.y * mz); fm[j][2 % V] = (float)(m4.z * mz); fm[j][3 % V] = (float)(m4.w * mz);
                v[j][0] = v4.x; v[j][1 % V] = v4.y; v[j][2 % V] = v4.z; v[j][3 % V] = v4.w;
            } else {
                fm[j][0] = (float)((int)mxy[r] * mz);
                v[j][0] = __ldg(src + i);
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j)
#pragma unroll
            for (int c = 0; c < V; ++c) {
                const bool used = fm[j][c] != 0.f;
                mn = fminf(mn, used ? v[j][c] : INFINITY);
                mx = fmaxf(mx, used ? v[j][c] : -INFINITY);
                power_chain(v[j][c], fm[j][c], inv_h, c0, a);
            }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(kFull, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    }
    if (lane == 0) { rmn[warp] = mn; rmx[warp] = mx; }
    const double sm = block_sum(a, red);                        // its barrier also publishes rmn / rmx
    if (threadIdx.x < kMomPad) part[(((size_t)pair * K + k) * B + b) * kMomPad + threadIdx.x] = sm;
    if (threadIdx.x == 32) {
#pragma unroll
        for (int w = 0; w < 8; ++w) { mn = fminf(mn, rmn[w]); mx = fmaxf(mx, rmx[w]); }
        if (mn <= mx) {
            atomicMin(keys + 4 * pair + key_off, float_key(mn));
            atomicMax(keys + 4 * pair + key_off + 1, float_key(mx));
        }
    }
}

// grid (K, pairs), 256 threads, thread b = bin b.  Chunk moments = sum of the B partial rows (fp64, fixed order).
// PREPARE: store them (target).  Otherwise: histograms H_b = e^{-y_b^2/2} sum_m N_m y_b^m/m! of the warped marginal (own
// range), the joint range (warped + target moments) and the target marginal; entropies, NMI, loss term as in
// nmi_epilogue_kernel; and the backward's polynomial c_m = (m+1) L_{m+1} - L_{m-1}, L_m = sum_b dL/dH_b e^{-y_b^2/2} y_b^m/m!
// (both warped bin sets), stored as c_m / h.  The last block of a pair adds the chunk terms in order and re-arms the
// warped range for the next call.
template <bool PREPARE>
__global__ void __launch_bounds__(256) nmi_src_epilogue_kernel(const double *__restrict__ part, int B, double *__restrict__ momT,
                                                                int *__restrict__ keys_all, float mid, float lo, float hi, float h,
                                                                double alpha, double weight, float *__restrict__ gtab,
                                                                double *__restrict__ scal_all, double *__restrict__ loss_out,
                                                                int loss_stride)
{
    __shared__ double fold[16][kMomPad + 1];
    __shared__ double rowW[kMomPad];
    __shared__ double sh[kWarps][kPow + 1];
    const int b = threadIdx.x, k = blockIdx.x, pair = blockIdx.y, K = gridDim.x;
    {
        const int col = b & 15, ln = b >> 4;
        const double *p = part + ((size_t)pair * K + k) * B * kMomPad;
        double acc = 0.0;
        for (int item = ln; item < B; item += 16) acc += p[(size_t)item * kMomPad + col];
        fold[ln][col] = acc;
        __syncthreads();
        if (b < kMomPad) {
            double v = 0.0;
#pragma unroll
            for (int l = 0; l < 16; ++l) v += fold[l][b];
            rowW[b] = v;
            if (PREPARE) momT[((size_t)pair * K + k) * kMomPad + b] = v;
        }
        __syncthreads();
    }
    if (PREPARE) return;
    int *keys = keys_all + 4 * pair;
    double *scal = scal_all + (size_t)pair * 16;
    const double eps = 1e-10, ln2 = 0.6931471805599453;
    float sT, eT, sW, eW, sJ, eJ;
    bin_range(keys, kRangeT, sT, eT);
    bin_range(keys, kRangeW, sW, eW);
    bin_range(keys, kRangeJ, sJ, eJ);
    const float vmin = fminf(eT, eW), vmax = fmaxf(sT, sW);
    const float cT = bin_centre(sT, eT, b), cW = bin_centre(sW, eW, b), cJ = bin_centre(sJ, eJ, b);
    const double yT = ((double)cT - (double)mid) / (double)h, yW = ((double)cW - (double)mid) / (double)h;
    const double yJ = ((double)cJ - (double)mid) / (double)h;
    const double gT = exp(-0.5 * yT * yT), gW = exp(-0.5 * yW * yW), gJ = exp(-0.5 * yJ * yJ);
    const double *rT = momT + ((size_t)pair * K + k) * kMomPad;
    double pW[kPow + 1], pJ[kPow + 1];                         // e^{-y^2/2} y^m / m!
    double hs[3] = {0.0, 0.0, 0.0};
    {
        double tT = gT, tW = gW, tJ = gJ;
#pragma unroll
        for (int m = 0; m <= kPow; ++m) {
            pW[m] = tW; pJ[m] = tJ;
            if (m < kPow) {
                const double mt = rT[m], mw = rowW[m];
                hs[0] += mt * tT; hs[1] += mw * tW; hs[2] += (mw + mt) * tJ;
            }
            const double inv = 1.0 / (double)(m + 1);          // compile-time constant
            tT *= yT * inv; tW *= yW * inv; tJ *= yJ * inv;
        }
    }
    const double H1 = hs[0], H2 = hs[1], HJ = hs[2];
    block_sum_all(hs, sh);
    const double S1 = hs[0], S2 = hs[1], SJ = hs[2];
    const double p1 = H1 / S1, p2 = H2 / S2, pj = HJ / SJ;
    const double l2 = log2(p2 + eps), lj = log2(pj + eps);
    const double d2 = l2 + p2 / ((p2 + eps) * ln2), dj = lj + pj / ((pj + eps) * ln2);      // dE/dp_b
    double es[5] = {p1 * log2(p1 + eps), p2 * l2, pj * lj, p2 * d2, pj * dj};
    block_sum_all(es, sh);
    const double E1 = es[0], E2 = es[1], EJ = es[2], A2 = es[3], AJ = es[4];
    const double den = E1 + E2, mi = den - EJ;
    const double nmi = 2.0 * mi / den;
    const double dev = nmi - 1.0;
    const double dl = weight * alpha / (double)K * (dev > 0.0 ? 1.0 : (dev < 0.0 ? -1.0 : 0.0));
    const double dn_e2 = 2.0 / den - 2.0 * mi / (den * den), dn_ej = -2.0 / den;
    // dL/dH_b = dl * dn * (dE/dp_b - sum_c p_c dE/dp_c) / S
    const double G2 = dl * dn_e2 * (d2 - A2) / S2, GJ = dl * dn_ej * (dj - AJ) / SJ;
    double lm[kPow + 1];
#pragma unroll
    for (int m = 0; m <= kPow; ++m) lm[m] = G2 * pW[m] + GJ * pJ[m];
    block_sum_all(lm, sh);
    if (b == 0) {
        float *tab = gtab + ((size_t)pair * K + k) * kMomPad;
#pragma unroll
        for (int m = 0; m < kPow; ++m) tab[m] = (float)(((double)(m + 1) * lm[m + 1] - (m > 0 ? lm[m - 1] : 0.0)) / (double)h);
    }
    // chunk term -> scal[k]; the last block of the pair adds them in chunk order
    unsigned *ticket = reinterpret_cast<unsigned *>(scal + 8);
    if (b == 0) __stcg(scal + k, fabs(dev));
    if (last_to_arrive(ticket, K) && b == 0) {
        double loss = 0.0;
        for (int c = 0; c < K; ++c) loss += __ldcg(scal + c);
        loss = weight * alpha * loss / (double)K;
        // the caller's value bounds are what makes the truncated series valid: refuse to report a number outside them
        if (!(vmin >= lo && vmax <= hi)) loss = __longlong_as_double(0x7ff8000000000000ll);
        loss_out[(size_t)pair * loss_stride] = loss;
        *ticket = 0u;
        keys[2] = INT_MAX; keys[3] = INT_MIN;          // every block of the pair has read the range by now
    }
}

// grid (GB, D, pairs): d loss / d warped voxel = mx*my * e^{-u^2/2} * sum_m u^m * sum_k mz_k(z) c_m^k / h
template <bool VEC>
__global__ void __launch_bounds__(256) nmi_src_grad_kernel(const float *__restrict__ vol, long long pair_stride, int D, int H, int W,
                                                            const int *__restrict__ tabs, const unsigned short *__restrict__ mxy,
                                                            const float *__restrict__ gtab, int K, float mid, float inv_h,
                                                            float *__restrict__ gout)
{
    __shared__ float coef[kMomPad];
    const int z = blockIdx.y, pair = blockIdx.z;
    const int *zlo = tabs + W + H, *zhi = zlo + D;
    const int zl = zlo[z], zh = zhi[z];
    if (threadIdx.x < kMomPad) {
        float c = 0.f;
        if (threadIdx.x < kPow)
            for (int k = 0; k < K; ++k) {
                const int w = chunk_overlap(zl, zh, k, kRes / K);
                if (w) c = fmaf((float)w, gtab[((size_t)pair * K + k) * kMomPad + threadIdx.x], c);
            }
        coef[threadIdx.x] = c;
    }
    __syncthreads();
    float cf[kPow];
#pragma unroll
    for (int m = 0; m < kPow; ++m) cf[m] = coef[m];
    constexpr int V = VEC ? 4 : 1, U = VEC ? 2 : 8;
    const int hw = H * W / V;
    const int i0 = blockIdx.x * (kGradSeg / V), i1 = min(hw, i0 + kGradSeg / V);
    const size_t base = (size_t)pair * pair_stride + (size_t)z * hw * V;
    const float c0 = -mid * inv_h;
    const bool read = zh > zl;
    for (int b0 = i0 + threadIdx.x; b0 < i1; b0 += 256 * U) {
        float v[U][V], fm[U][V];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int i = min(b0 + 256 * j, i1 - 1);
            if (VEC) {
                const ushort4 m4 = *reinterpret_cast<const ushort4 *>(mxy + 4 * i);
                const float4 v4 = __ldg(reinterpret_cast<const float4 *>(vol + base) + i);
                fm[j][0] = (float)m4.x; fm[j][1 % V] = (float)m4.y; fm[j][2 % V] = (float)m4.z; fm[j][3 % V] = (float)m4.w;
                v[j][0] = v4.x; v[j][1 % V] = v4.y; v[j][2 % V] = v4.z; v[j][3 % V] = v4.w;
            } else {
                fm[j][0] = (float)mxy[i];
                v[j][0] = __ldg(vol + base + i);
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            float g[V];
#pragma unroll
            for (int c = 0; c < V; ++c) {
                const float u = fmaf(v[j][c], inv_h, c0);
                float acc = cf[kPow - 1];
#pragma unroll
                for (int m = kPow - 2; m >= 0; --m) acc = fmaf(acc, u, cf[m]);
                g[c] = read ? fm[j][c] * ex2_approx(-0.72134752f * u * u) * acc : 0.f;
            }
            const int i = b0 + 256 * j;
            if (i < i1) {
                if (VEC) reinterpret_cast<float4 *>(gout + base)[i] = make_float4(g[0], g[1 % V], g[2 % V], g[3 % V]);
                else gout[base + i] = g[0];
            }
        }
    }
}

__global__ void nmi_src_theta_kernel(const float *__restrict__ state, float *__restrict__ theta, int n_pairs, int nt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pairs * nt) theta[i] = state[(size_t)(i / nt) * TRB_STATE_FLOATS + TRB_STATE_THETA + i % nt];
}

// d term / d theta from the moments pass run with d term / d warped in the target slot (block [17..28] = sum gout * J)
__global__ void nmi_src_extract_kernel(const double *__restrict__ mom2, double *__restrict__ extra, int n_pairs, int ndim, int D, int H, int W)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int nc = ndim + 1, nt = ndim * nc;
    if (i >= n_pairs * nt) return;
    const int pair = i / nt, j = i % nt, r = j / nc;
    const double scale = r == 0 ? 0.5 * W : (r == 1 ? 0.5 * H : 0.5 * D);
    extra[(size_t)pair * 13 + 1 + j] = mom2[(size_t)pair * TRB_MOMENTS + 17 + j] * scale;
}

static int src_validate(int ndim, int n_pairs, int D, int H, int W, float bandwidth, float lo, float hi, const void *ws, size_t ws_bytes)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (n_pairs < 1 || n_pairs > 65535) { set_error("n_pairs must be in 1..65535 (got %d)", n_pairs); return TRB_ERR_ARG; }
    if (H < 1 || W < 1 || (ndim == 3 && D < 1)) { set_error("bad volume shape %dx%dx%d", D, H, W); return TRB_ERR_ARG; }
    const SrcDims d = src_dims(ndim, D, H, W);
    if ((long long)d.D * (kRes / d.K) / kRes + 2 > kMaxChunkSlices || d.D > 65535) {
        set_error("source-space NMI: %d slices / rows is too many for one chunk table", d.D); return TRB_ERR_UNSUPPORTED;
    }
    if ((unsigned long long)d.D * d.H * d.W >= (1ull << 31)) { set_error("volume too large"); return TRB_ERR_UNSUPPORTED; }
    if (!(bandwidth > 0.f)) { set_error("bandwidth must be positive"); return TRB_ERR_ARG; }
    if (!(lo <= hi)) { set_error("value bounds must satisfy lo <= hi"); return TRB_ERR_ARG; }
    if (hi - lo > 0.6f * bandwidth) {
        set_error("source-space NMI needs a value range <= 0.6 bandwidths (got %g for bandwidth %g): use trb_nmi_loss_grad",
                  (double)(hi - lo), (double)bandwidth);
        return TRB_ERR_UNSUPPORTED;
    }
    const SrcLayout L = src_layout(n_pairs, d.K, d.D, d.H, d.W);
    if (!ws || ws_bytes < L.total) { set_error("workspace too small: need %zu bytes", L.total); return TRB_ERR_WORKSPACE; }
    return TRB_OK;
}

static bool src_vec_ok(const float *p, long long pair_stride, int H, int W)
{
    return ((size_t)H * W) % 4 == 0 && pair_stride % 4 == 0 && ((uintptr_t)p & 15) == 0;
}

static int src_loss_grad(const float *warped, long long pair_stride, int n_pairs, const SrcDims &d, float bandwidth, float alpha,
                         float weight, float lo, float hi, double *loss_dev, int loss_stride, float *gout, char *ws, cudaStream_t s)
{
    const int K = d.K, D = d.D, H = d.H, W = d.W;
    const SrcLayout L = src_layout(n_pairs, K, D, H, W);
    int *keys = (int *)(ws + L.off_keys), *tabs = (int *)(ws + L.off_tabs);
    const unsigned short *mxy = (const unsigned short *)(ws + L.off_mxy);
    double *momT = (double *)(ws + L.off_momT), *part = (double *)(ws + L.off_part), *scal = (double *)(ws + L.off_scal);
    float *gtab = (float *)(ws + L.off_gtab);
    const float mid = 0.5f * (lo + hi), inv_h = 1.f / bandwidth;
    const bool vec = src_vec_ok(warped, pair_stride, H, W) && (!gout || src_vec_ok(gout, pair_stride, H, W));
    if (vec) nmi_src_moments_kernel<true><<<dim3(L.B, K, n_pairs), 256, 0, s>>>(warped, pair_stride, D, H, W, tabs, mxy, mid, inv_h, part, keys, 2);
    else nmi_src_moments_kernel<false><<<dim3(L.B, K, n_pairs), 256, 0, s>>>(warped, pair_stride, D, H, W, tabs, mxy, mid, inv_h, part, keys, 2);
    nmi_src_epilogue_kernel<false><<<dim3(K, n_pairs), 256, 0, s>>>(part, L.B, momT, keys, mid, lo, hi, bandwidth, (double)alpha,
                                                                    (double)weight, gtab, scal, loss_dev, loss_stride);
    if (gout && vec) nmi_src_grad_kernel<true><<<dim3(L.GB, D, n_pairs), 256, 0, s>>>(warped, pair_stride, D, H, W, tabs, mxy, gtab, K, mid, inv_h, gout);
    else if (gout) nmi_src_grad_kernel<false><<<dim3(L.GB, D, n_pairs), 256, 0, s>>>(warped, pair_stride, D, H, W, tabs, mxy, gtab, K, mid, inv_h, gout);
    return check_cuda(cudaGetLastError(), "nmi_src_loss_grad");
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_nmi_src_workspace_bytes(int ndim, int n_pairs, int D, int H, int W)
{
    if ((ndim != 2 && ndim != 3) || n_pairs < 1 || H < 1 || W < 1 || (ndim == 3 && D < 1)) return 0;
    const SrcDims d = src_dims(ndim, D, H, W);
    return src_layout(n_pairs, d.K, d.D, d.H, d.W).total;
}

extern "C" int trb_nmi_src_prepare(int ndim, const float *target_dev, long long pair_stride, int n_pairs, int D, int H, int W,
                                   float bandwidth, float lo, float hi, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = src_validate(ndim, n_pairs, D, H, W, bandwidth, lo, hi, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!target_dev) { set_error("null target"); return TRB_ERR_ARG; }
    const SrcDims d = src_dims(ndim, D, H, W);
    const SrcLayout L = src_layout(n_pairs, d.K, d.D, d.H, d.W);
    char *ws = (char *)workspace_dev;
    int *keys = (int *)(ws + L.off_keys), *tabs = (int *)(ws + L.off_tabs);
    unsigned short *mxy = (unsigned short *)(ws + L.off_mxy);
    double *momT = (double *)(ws + L.off_momT), *part = (double *)(ws + L.off_part);
    cudaStream_t s = (cudaStream_t)stream;
    const float mid = 0.5f * (lo + hi), inv_h = 1.f / bandwidth;
    nmi_src_tables_kernel<<<(d.W + d.H + d.D + 127) / 128, 128, 0, s>>>(d.W, d.H, d.D, tabs);
    nmi_src_plane_kernel<<<(d.W * d.H + 255) / 256, 256, 0, s>>>(d.W, d.H, tabs, mxy);
    nmi_src_reset_kernel<<<(n_pairs + 127) / 128, 128, 0, s>>>(keys, n_pairs, 0);
    nmi_src_reset_kernel<<<(n_pairs + 127) / 128, 128, 0, s>>>(keys, n_pairs, 2);
    cudaMemsetAsync(ws + L.off_scal, 0, (size_t)n_pairs * 16 * sizeof(double), s);      // chunk terms + the epilogue's tickets
    if (src_vec_ok(target_dev, pair_stride, d.H, d.W))
        nmi_src_moments_kernel<true><<<dim3(L.B, d.K, n_pairs), 256, 0, s>>>(target_dev, pair_stride, d.D, d.H, d.W, tabs, mxy, mid, inv_h, part, keys, 0);
    else
        nmi_src_moments_kernel<false><<<dim3(L.B, d.K, n_pairs), 256, 0, s>>>(target_dev, pair_stride, d.D, d.H, d.W, tabs, mxy, mid, inv_h, part, keys, 0);
    nmi_src_epilogue_kernel<true><<<dim3(d.K, n_pairs), 256, 0, s>>>(part, L.B, momT, keys, mid, lo, hi, bandwidth, 0.0, 0.0, nullptr,
                                                                     nullptr, nullptr, 0);
    return check_cuda(cudaGetLastError(), "nmi_src_prepare");
}

extern "C" int trb_nmi_src_loss_grad(int ndim, const float *warped_dev, long long pair_stride, int n_pairs, int D, int H, int W,
                                     float bandwidth, float alpha, float weight, float lo, float hi, double *loss_dev,
                                     int loss_stride, float *gout_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = src_validate(ndim, n_pairs, D, H, W, bandwidth, lo, hi, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!warped_dev || !loss_dev || loss_stride < 1) { set_error("null pointer / loss stride"); return TRB_ERR_ARG; }
    return src_loss_grad(warped_dev, pair_stride, n_pairs, src_dims(ndim, D, H, W), bandwidth, alpha, weight, lo, hi, loss_dev, loss_stride,
                         gout_dev, (char *)workspace_dev, (cudaStream_t)stream);
}

// The reference's loop with its DEFAULT criterions [MSE, NCC, NMI] (warpings.py:36-40,123-159), every epoch enqueued from
// here: MSE/NCC moments (all pairs; the 3-D TMA pass also stores the warped volumes) -> NMI term and d term / d warped ->
// chained to theta by a second moments pass (d term / d warped in the target slot) -> update, best-theta and loss
// bookkeeping on the device.
extern "C" int trb_affine_optim_nmi(int ndim, int mode, const float *moving_dev, const float *target_dev, int n_pairs, int D, int H, int W,
                                    const float *xb_dev, const float *yb_dev, const float *zb_dev, float *state_dev,
                                    float *loss_log_dev, int log_stride, int epoch0, int n_epochs, float w_mse, float w_ncc,
                                    float w_nmi, float lr, int optimiser, float beta1, float beta2, float adam_eps, int flags,
                                    float bandwidth, float alpha, float lo, float hi, float *warped_scratch_dev,
                                    float *gout_scratch_dev, void *nmi_workspace_dev, size_t nmi_workspace_bytes,
                                    void *workspace_dev, size_t workspace_bytes, void *stream)
{
    int rc = src_validate(ndim, n_pairs, D, H, W, bandwidth, lo, hi, nmi_workspace_dev, nmi_workspace_bytes);
    if (rc) return rc;
    if (!moving_dev || !target_dev || !state_dev || !warped_scratch_dev || !gout_scratch_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (loss_log_dev && epoch0 + n_epochs > log_stride) { set_error("loss log too short"); return TRB_ERR_ARG; }
    const SrcDims d = src_dims(ndim, D, H, W);
    const SrcLayout L = src_layout(n_pairs, d.K, d.D, d.H, d.W);
    char *ws = (char *)nmi_workspace_dev;
    double *mom = (double *)(ws + L.off_mom), *mom2 = (double *)(ws + L.off_mom2), *extra = (double *)(ws + L.off_extra);
    float *theta = (float *)(ws + L.off_theta);
    const int Dn = ndim == 3 ? D : 1, slices = ndim == 3 ? D : H, nt = ndim * (ndim + 1);
    const long long vol = (long long)Dn * H * W;
    cudaStream_t s = (cudaStream_t)stream;
    const int nb = (n_pairs * nt + 127) / 128;
    for (int e = 0; e < n_epochs; ++e) {
        bool have_warped = false;
        rc = affine_moments_impl(ndim, moving_dev, target_dev, vol, n_pairs, Dn, H, W, 0, slices, xb_dev, yb_dev, zb_dev, state_dev, mom, flags,
                                 e == 0 ? 3 : 2, warped_scratch_dev, &have_warped, workspace_dev, workspace_bytes, stream);
        if (rc) return rc;
        if (!have_warped) {             // the pass ran on a kernel without the by-product (2-D / shape / rotation): separate warp
            nmi_src_theta_kernel<<<nb, 128, 0, s>>>(state_dev, theta, n_pairs, nt);
            rc = trb_warp_affine_batch(ndim, moving_dev, warped_scratch_dev, n_pairs, 1, Dn, H, W, theta, xb_dev, yb_dev, zb_dev, flags, stream);
            if (rc) return rc;
        }
        rc = src_loss_grad(warped_scratch_dev, vol, n_pairs, d, bandwidth, alpha, w_nmi, lo, hi, extra, 13, gout_scratch_dev, ws, s);
        if (rc) return rc;
        rc = affine_moments_impl(ndim, moving_dev, gout_scratch_dev, vol, n_pairs, Dn, H, W, 0, slices, xb_dev, yb_dev, zb_dev, state_dev, mom2,
                                 flags, 0, nullptr, nullptr, workspace_dev, workspace_bytes, stream);
        if (rc) return rc;
        nmi_src_extract_kernel<<<nb, 128, 0, s>>>(mom2, extra, n_pairs, ndim, Dn, H, W);
        rc = trb_affine_apply(ndim, mode, mom, n_pairs, Dn, H, W, state_dev, loss_log_dev, log_stride, epoch0 + e, w_mse, w_ncc, lr, optimiser,
                              beta1, beta2, adam_eps, extra, stream);
        if (rc) return rc;
    }
    return check_cuda(cudaGetLastError(), "affine_optim_nmi");
}
