// nmi_shared.cuh — device helpers shared by the two evaluations of the NMI/KDE term (nmi.cu: on the resampled 200^n
// arrays, all bin regimes; nmi_src.cu: in source-voxel space, Hermite-moment regime).  See nmi.cu for the semantics.
#pragma once
#include "common.cuh"
#include <limits.h>

namespace trb {

constexpr int kBins = 256, kRes = 200, kPatch = 100;

// monotone float <-> int key so min/max can use integer atomics (order independent = deterministic)
__device__ __forceinline__ int float_key(float f)
{
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__device__ __forceinline__ float ex2_approx(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// torch 'nearest' source index (UpSample.h nearest_neighbor_compute_source_index): floor(dst * scale), clamped
__device__ __forceinline__ int nearest_src(int i, float scale, int S) { return min((int)floorf((float)i * scale), S - 1); }

// bin centre b of torch.linspace(start, end, 256) in fp32 (RangeFactories: symmetric evaluation from both ends)
__device__ __forceinline__ float bin_centre(float start, float end, int b)
{
    const float step = (end - start) / (float)(kBins - 1);
    return b < kBins / 2 ? start + step * (float)b : end - step * (float)(kBins - 1 - b);
}

enum { kRangeT = 0, kRangeW = 1, kRangeJ = 2 };
// (start, end) = (max, min): the reference swaps them (utils.py:45-46)
__device__ __forceinline__ void bin_range(const int *__restrict__ keys, int which, float &start, float &end)
{
    const float tmin = key_float(keys[0]), tmax = key_float(keys[1]), wmin = key_float(keys[2]), wmax = key_float(keys[3]);
    if (which == kRangeT) { start = tmax; end = tmin; }
    else if (which == kRangeW) { start = wmax; end = wmin; }
    else { start = fmaxf(tmax, wmax); end = fminf(tmin, wmin); }
}

// Bins are equally spaced, so inside a group of kGroup bins anchored at bin b0
//   2^-(t0 - j*d)^2 = 2^-(t0^2) * (2^(2*d*t0))^j * 2^-(j*d)^2,    t0 = (s - c_b0)*kappa, d = step*kappa:
// two MUFU.EX2 per value and group, then one multiply (running power) and one FMA (times the constant 2^-(j d)^2)
// per bin instead of one MUFU per bin — 3.4x fewer issue cycles on the quarter-rate unit.  Valid while the
// running power cannot overflow before the Gaussian itself underflows: (kGroup-1)^2 * d^2 < 100, i.e. bin spacing
// below ~1.7 bandwidths (always for normalised or 8-bit data with the default bandwidth 3); wider spacings take
// the direct one-exponential-per-bin path.  Error: <= (j+1) roundings, j < 8.
constexpr int kGroup = 8;
__device__ __forceinline__ float bin_delta(const int *__restrict__ keys, int which, float kappa)
{
    float s, e;
    bin_range(keys, which, s, e);
    return (e - s) / (float)(kBins - 1) * kappa;
}
__device__ __forceinline__ bool group_ok(float d) { return (float)((kGroup - 1) * (kGroup - 1)) * d * d < 100.f; }

// Third form, for bin ranges narrow against the bandwidth (normalised images with the default bandwidth 3: the
// whole range spans 1/3 of a bandwidth).  With u = (s - mid)/h and y_b = (c_b - mid)/h,
//   exp(-(u - y)^2/2) = exp(-u^2/2) * sum_m He_m(u) y^m / m!        (generating function of the Hermite polynomials)
// so every histogram is H_b = sum_m (y_b^m/m!) M_m with kMom moments M_m = sum_p exp(-u_p^2/2) He_m(u_p) per chunk —
// 12 recurrence steps per value instead of 256 bins — and its backward is -(1/h) exp(-u^2/2) sum_m He_{m+1}(u) Gamma_m
// with Gamma_m = sum_b (dL/dH_b) y_b^m/m!.  Truncation for |y|,|u| <= 0.3: 0.3^12/sqrt(12!) = 2e-11.
constexpr int kMom = 12;
__device__ __forceinline__ bool moment_ok(const int *__restrict__ keys, int which, float h)
{
    float s, e;
    bin_range(keys, which, s, e);
    return fabsf(s - e) <= 0.6f * h;
}
__device__ __forceinline__ float range_mid(const int *__restrict__ keys, int which)
{
    float s, e;
    bin_range(keys, which, s, e);
    return 0.5f * (s + e);
}
// e * He_m(u) for m = 0..kMom accumulated against coefficients: f(m, value)
template <int COUNT, typename F>
__device__ __forceinline__ void hermite_chain(float s, float mid, float inv_h, F f)
{
    const float u = (s - mid) * inv_h;
    float hm1 = ex2_approx(-0.72134752f * u * u), hm = u * hm1;       // exp(-u^2/2)
    f(0, hm1);
    f(1, hm);
#pragma unroll
    for (int m = 1; m + 1 < COUNT; ++m) {
        const float hn = fmaf(u, hm, -(float)m * hm1);
        f(m + 1, hn);
        hm1 = hm; hm = hn;
    }
}

// a histogram kept in moment form (M_0..M_11) evaluated at the bin with reduced centre y = (c_b - mid)/h, in fp64
__device__ __forceinline__ double expand_moments(const double *__restrict__ row, double y)
{
    double acc = 0.0, term = 1.0;
#pragma unroll
    for (int m = 0; m < kMom; ++m) { acc += row[m] * term; term *= y / (double)(m + 1); }
    return acc;
}

}  // namespace trb
