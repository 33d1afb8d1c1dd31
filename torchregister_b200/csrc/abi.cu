// abi.cu — error plumbing and version entry points of the C ABI (include/trb.h).
#include "common.cuh"
#include <stdarg.h>
#include <stdio.h>

namespace trb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return TRB_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return (int)e;
}

// grid sizes follow the SM count; launchers ask on every call, so the answer is cached per device ordinal
static int g_sm_count[64] = {};

int sm_count(int &n)
{
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice");
    if (rc) return rc;
    int &c = g_sm_count[dev & 63];
    if (c == 0) rc = check_cuda(cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, dev), "SM count");
    n = c;
    return rc;
}

int check_fast_floor_axes(int ndim, int D, int H, int W)
{
    if (W <= kMaxFastFloorAxis && H <= kMaxFastFloorAxis && (ndim != 3 || D <= kMaxFastFloorAxis)) return TRB_OK;
    set_error("every spatial axis must be at most 2^22 = %d voxels long (got %dx%dx%d): the sampling kernels' fast floor "
              "indexes exactly only up to there", kMaxFastFloorAxis, ndim == 3 ? D : 1, H, W);
    return TRB_ERR_UNSUPPORTED;
}

int validate_flow(int ndim, int D, int H, int W)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (H < 2 || W < 2 || (ndim == 3 && D < 2)) { set_error("flow warp needs every axis >= 2 (got %dx%dx%d)", D, H, W); return TRB_ERR_ARG; }
    if ((unsigned long long)(ndim == 3 ? D : 1) * H * W >= (1ull << 31)) { set_error("flow kernels index volumes with 32 bits: D*H*W must stay below 2^31"); return TRB_ERR_ARG; }
    return check_fast_floor_axes(ndim, D, H, W);
}

int flow_grid(size_t vol, unsigned &grid)
{
    int sms;
    if (int rc = sm_count(sms)) return rc;
    size_t nb = (vol + 255) / 256;      // enough CTAs for every SM to hold 8; each strides over row pairs
    const size_t cap = (size_t)sms * 8;
    if (nb > cap) nb = cap;
    if (nb > kFlowMaxBlocks) nb = kFlowMaxBlocks;
    grid = (unsigned)(nb < 1 ? 1 : nb);
    return TRB_OK;
}

}  // namespace trb

extern "C" int trb_abi_version(void) { return TRB_ABI_VERSION; }
extern "C" const char *trb_last_error(void) { return trb::g_err; }
