// capi.cu -- the C ABI of include/wrfb200.h: device-resident patch state, stream-ordered launcher,
// CUDA-graph replay, and the reference-compatible 48-argument entry point.
//
// Replaces the reference CUDA host layer /root/reference/advance_mu_t_no_async.cu:35-424, which on
// EVERY call cudaMallocs 29 buffers per GPU (:178-244), copies every field host->device (:245-306),
// launches (:329-353), blocks (:354-357), copies 8 fields back (:366-390) and frees (:392-423).
// Here allocation happens once per patch, copies happen only when the caller asks (per RK sub-step,
// not per acoustic step), launches are asynchronous on a caller-visible stream, and errors are
// returned instead of exit() (:22-32).
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <tuple>
#include <type_traits>

#include "amt_params.h"
#include "capi_internal.h"

// -------------------------------------------------------------------------------------------------
// errors
// -------------------------------------------------------------------------------------------------
namespace {

thread_local char g_err[512] = "";

#define fail wrfb200_fail

#define CU(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return fail(WRFB200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),    \
                        __FILE__, __LINE__);                                                         \
    } while (0)

inline bool is3d(int f) { return f >= WRFB200_WW && f <= WRFB200_FT; }
inline bool is2d(int f) { return f >= WRFB200_MU && f <= WRFB200_MSFTY; }
inline bool is1d(int f) { return f >= WRFB200_DNW && f <= WRFB200_RDNW; }

inline long round_up(long x, long m) { return (x + m - 1) / m * m; }

}  // namespace

namespace {

int check_domain(const wrfb200_domain &d)
{
    if (d.ime < d.ims || d.jme < d.jms || d.kme < d.kms)
        return fail(WRFB200_ERR_INVALID_ARG, "empty memory extents");
    if (d.kms > 1) return fail(WRFB200_ERR_UNSUPPORTED, "kms=%d > 1: the routine addresses level 1 literally", d.kms);
    if (d.kme < d.kde) return fail(WRFB200_ERR_INVALID_ARG, "kme=%d < kde=%d", d.kme, d.kde);
    return WRFB200_OK;
}

}  // namespace

namespace {

// Build the kernel argument block for the tile its:ite x jts:jte.  Returns >0 status on error,
// sets *empty when the index sets are empty (legal: nothing to do).  P = AmtParams or AmtParamsR8, matching
// the handle's element size (the callers check it).
template <class P>
int make_params(const wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte, P *out, bool *empty)
{
    using T = std::remove_pointer_t<decltype(P::ww)>;
    const wrfb200_domain &d = h->dom;
    if (kts != 1) return fail(WRFB200_ERR_UNSUPPORTED, "kts=%d: the routine addresses levels 1 and 2 literally (module_small_step_em.f90:159,168,209)", kts);
    if (kte != d.kde) return fail(WRFB200_ERR_UNSUPPORTED, "kte=%d != kde=%d: wdtn(kde) is the top boundary flux (module_small_step_em.f90:221)", kte, d.kde);
    if (kte > d.kme) return fail(WRFB200_ERR_INVALID_ARG, "kte=%d > kme=%d", kte, d.kme);
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   its, ite, jts, jte, kts, kte, &is, &ie, &js, &je, &ks, &ke);
    *empty = (is > ie || js > je || ks > ke);
    if (*empty) return WRFB200_OK;
    if (is - 1 < d.ims || ie + 1 > d.ime || js - 1 < d.jms || je + 1 > d.jme)
        return fail(WRFB200_ERR_INVALID_ARG,
                    "computed range i=%d..%d j=%d..%d needs a one-cell ring inside memory i=%d..%d j=%d..%d",
                    is, ie, js, je, d.ims, d.ime, d.jms, d.jme);
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f)
        if (!h->d[f]) return fail(WRFB200_ERR_STATE, "field %d has no device buffer (allocate or bind it)", f);
    if (!h->scalars_set)
        return fail(WRFB200_ERR_STATE, "rdx/rdy/dts/epssm not set (wrfb200_set_scalars%s)", sizeof(T) == 8 ? "_r8" : "");

    auto F = [h](int f) { return reinterpret_cast<T *>(h->d[f]); };
    P p{};
    p.ww = F(WRFB200_WW);       p.ww_1 = F(WRFB200_WW_1);
    p.u = F(WRFB200_U);         p.u_1 = F(WRFB200_U_1);
    p.v = F(WRFB200_V);         p.v_1 = F(WRFB200_V_1);
    p.t = F(WRFB200_T);         p.t_1 = F(WRFB200_T_1);
    p.t_ave = F(WRFB200_T_AVE); p.ft = F(WRFB200_FT);
    p.mu = F(WRFB200_MU);       p.mut = F(WRFB200_MUT);
    p.muave = F(WRFB200_MUAVE); p.muts = F(WRFB200_MUTS);
    p.muu = F(WRFB200_MUU);     p.muv = F(WRFB200_MUV);
    p.mudf = F(WRFB200_MUDF);   p.mu_tend = F(WRFB200_MU_TEND);
    p.msfuy = F(WRFB200_MSFUY); p.msfvx_inv = F(WRFB200_MSFVX_INV);
    p.msftx = F(WRFB200_MSFTX); p.msfty = F(WRFB200_MSFTY);
    p.dnw = F(WRFB200_DNW);     p.fnm = F(WRFB200_FNM);
    p.fnp = F(WRFB200_FNP);     p.rdnw = F(WRFB200_RDNW);
    p.rdx = (T)h->rdx; p.rdy = (T)h->rdy; p.dts = (T)h->dts; p.epssm = (T)h->epssm;   // exact: stored from a T
    p.pitch = h->pitch3;
    p.jstride = h->pitch3 * (long long)h->kdim;
    p.pitch2 = h->pitch2;
    p.i0 = is - d.ims; p.i1 = ie - d.ims;
    p.j0 = js - d.jms; p.j1 = je - d.jms;
    p.k0 = ks - d.kms;
    p.nk = ke - ks + 1;
    p.kdim = h->kdim;
    p.jdim = h->jdim;
    *out = p;
    return WRFB200_OK;
}

}  // namespace

int wrfb200_make_params(const wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                AmtParams *out, bool *empty)
{
    return make_params(h, its, ite, jts, jte, kts, kte, out, empty);
}

namespace {

// Tuning override for the pipelined kernel: WRFB200_PIPE_CFG = TJ*10 + STAGES (0 / unset = automatic).
int pipe_cfg()
{
    static const int cfg = [] { const char *e = getenv("WRFB200_PIPE_CFG"); return e ? atoi(e) : 0; }();
    return cfg;
}

int launch(wrfb200_handle *h, const AmtParams &p, cudaStream_t s, int kernel)
{
    cudaError_t e;
    int ran = kernel;
    if (kernel == WRFB200_KERNEL_COLUMN) {
        e = amt_launch_column(p, s);
    } else if (kernel == WRFB200_KERNEL_TILE) {
        if (!amt_tile_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "tile kernel needs 16-byte aligned fields and pitches that are multiples of 4");
        e = amt_launch_tile(p, s);
    } else if (kernel == WRFB200_KERNEL_PIPE) {
        if (!amt_pipe_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "pipe kernel needs 16-byte aligned fields and pitches that are multiples of 4");
        if (!amt_build_tma_maps(p, &h->maps)) return fail(WRFB200_ERR_CUDA, "cuTensorMapEncodeTiled failed");
        e = amt_launch_pipe(p, h->maps, s, pipe_cfg());
    } else {
        // AUTO: the TMA-pipelined tile kernel wherever the layout allows it; tiles narrower than a warp
        // of columns (e.g. the one-column strips behind an east halo) would stage 128-wide rows for
        // nothing, and unaligned caller layouts cannot be bulk-copied: those take the column kernel.
        const bool wide = (p.i1 - p.i0 + 1) >= 32;
        if (wide && amt_pipe_supported(p) && amt_build_tma_maps(p, &h->maps)) {
            e = amt_launch_pipe(p, h->maps, s, pipe_cfg());
            ran = WRFB200_KERNEL_PIPE;
        } else {
            e = amt_launch_column(p, s);
            ran = WRFB200_KERNEL_COLUMN;
        }
    }
    if (e != cudaSuccess) return fail(WRFB200_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    h->last_kernel = ran;
    return WRFB200_OK;
}

// real*8: the double2 tile kernel where the layout allows it, else the any-layout column kernel.  The TMA pipe
// kernel is binary32 only.
int launch(wrfb200_handle *h, const AmtParamsR8 &p, cudaStream_t s, int kernel)
{
    cudaError_t e;
    int ran = kernel;
    if (kernel == WRFB200_KERNEL_PIPE) {
        return fail(WRFB200_ERR_UNSUPPORTED, "the pipe kernel is binary32 only; a real*8 handle runs the tile or column kernel");
    } else if (kernel == WRFB200_KERNEL_COLUMN) {
        e = amt_launch_column(p, s);
    } else if (kernel == WRFB200_KERNEL_TILE) {
        if (!amt_tile_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "real*8 tile kernel needs 16-byte aligned fields, pitches of an even "
                                                 "number of doubles and at most 220 levels (nk=%d)", p.nk);
        e = amt_launch_tile(p, s);
    } else {
        // AUTO: tiles narrower than a warp of columns take the column kernel, as for binary32
        const bool wide = (p.i1 - p.i0 + 1) >= 32;
        if (wide && amt_tile_supported(p)) {
            e = amt_launch_tile(p, s);
            ran = WRFB200_KERNEL_TILE;
        } else {
            e = amt_launch_column(p, s);
            ran = WRFB200_KERNEL_COLUMN;
        }
    }
    if (e != cudaSuccess) return fail(WRFB200_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    h->last_kernel = ran;
    return WRFB200_OK;
}

// validate the tile and launch one step on `s` in the handle's precision
int step_on(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte, cudaStream_t s, int kernel)
{
    bool empty = false;
    if (h->esize == 8) {
        AmtParamsR8 p;
        if (int rc = make_params(h, its, ite, jts, jte, kts, kte, &p, &empty)) return rc;
        return empty ? WRFB200_OK : launch(h, p, s, kernel);
    }
    AmtParams p;
    if (int rc = make_params(h, its, ite, jts, jte, kts, kte, &p, &empty)) return rc;
    return empty ? WRFB200_OK : launch(h, p, s, kernel);
}

// A verb typed for one precision applied to a handle of the other.
int wrong_precision(const wrfb200_handle *h, const char *verb)
{
    return fail(WRFB200_ERR_STATE, "%s: this is a %s handle (created by %s); use the %s verbs", verb,
                h->esize == 8 ? "real*8" : "real*4", h->esize == 8 ? "wrfb200_create_r8" : "wrfb200_create",
                h->esize == 8 ? "_r8" : "binary32 (no _r8 suffix)");
}

}  // namespace

int wrfb200_require_r4(const wrfb200_handle *h, const char *what)
{
    if (h->esize == 4) return WRFB200_OK;
    return fail(WRFB200_ERR_UNSUPPORTED, "%s is binary32 only and not available on a real*8 handle", what);
}

int wrfb200_launch_params(wrfb200_handle *h, const AmtParams &p, cudaStream_t s, int kernel)
{
    return launch(h, p, s, kernel);
}

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define GUARD(h)                                                                                     \
    if (!(h)) return fail(WRFB200_ERR_INVALID_ARG, "null handle");                                   \
    DeviceGuard guard_((h)->device);                                                                 \
    if (!guard_.ok) return fail(WRFB200_ERR_CUDA, "cannot select CUDA device %d", (h)->device)

// Copy a Fortran-numbered sub-box between a dense host array and the (pitched) device mirror, in elements of
// the handle's size (4 or 8 bytes).
int copy_range(wrfb200_handle *h, int field, const void *host_src, void *host_dst,
               int i0, int i1, int k0, int k1, int j0, int j1)
{
    const wrfb200_domain &d = h->dom;
    if (field < 0 || field >= WRFB200_NUM_FIELDS) return fail(WRFB200_ERR_INVALID_ARG, "bad field id %d", field);
    if (!h->d[field]) return fail(WRFB200_ERR_STATE, "field %d has no device buffer", field);
    const bool to_dev = host_src != nullptr;
    const cudaMemcpyKind kind = to_dev ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    const size_t es = (size_t)h->esize;
    char *dev = reinterpret_cast<char *>(h->d[field]);
    char *host = to_dev ? const_cast<char *>(static_cast<const char *>(host_src)) : static_cast<char *>(host_dst);
    if (is1d(field)) {
        if (k0 < d.kms || k1 > d.kme || k0 > k1) return fail(WRFB200_ERR_INVALID_ARG, "bad k range %d..%d", k0, k1);
        const size_t off = (size_t)(k0 - d.kms) * es, n = (size_t)(k1 - k0 + 1) * es;
        if (to_dev) CU(cudaMemcpyAsync(dev + off, host + off, n, kind, h->stream));
        else        CU(cudaMemcpyAsync(host + off, dev + off, n, kind, h->stream));
        return WRFB200_OK;
    }
    if (i0 < d.ims || i1 > d.ime || i0 > i1 || j0 < d.jms || j1 > d.jme || j0 > j1)
        return fail(WRFB200_ERR_INVALID_ARG, "bad i/j range %d..%d, %d..%d", i0, i1, j0, j1);
    const size_t w = (size_t)(i1 - i0 + 1) * es;
    if (is2d(field)) {
        const size_t hoff = ((size_t)(j0 - d.jms) * h->idim + (size_t)(i0 - d.ims)) * es;
        const size_t doff = ((size_t)(j0 - d.jms) * h->pitch2 + (size_t)(i0 - d.ims)) * es;
        const size_t rows = (size_t)(j1 - j0 + 1);
        if (to_dev)
            CU(cudaMemcpy2DAsync(dev + doff, h->pitch2 * es, host + hoff, h->idim * es, w, rows, kind, h->stream));
        else
            CU(cudaMemcpy2DAsync(host + hoff, h->idim * es, dev + doff, h->pitch2 * es, w, rows, kind, h->stream));
        return WRFB200_OK;
    }
    if (k0 < d.kms || k1 > d.kme || k0 > k1) return fail(WRFB200_ERR_INVALID_ARG, "bad k range %d..%d", k0, k1);
    const size_t nkc = (size_t)(k1 - k0 + 1), njc = (size_t)(j1 - j0 + 1);
    const size_t hoff = (((size_t)(j0 - d.jms) * h->kdim + (size_t)(k0 - d.kms)) * h->idim + (size_t)(i0 - d.ims)) * es;
    const size_t doff = (((size_t)(j0 - d.jms) * h->kdim + (size_t)(k0 - d.kms)) * h->pitch3 + (size_t)(i0 - d.ims)) * es;
    if (nkc == (size_t)h->kdim) {
        // whole columns: rows of one field are equally spaced across k AND j -> a single 2-D copy
        const size_t rows = nkc * njc;
        if (to_dev)
            CU(cudaMemcpy2DAsync(dev + doff, h->pitch3 * es, host + hoff, h->idim * es, w, rows, kind, h->stream));
        else
            CU(cudaMemcpy2DAsync(host + hoff, h->idim * es, dev + doff, h->pitch3 * es, w, rows, kind, h->stream));
        return WRFB200_OK;
    }
    cudaMemcpy3DParms cp{};
    cudaPitchedPtr hostp = make_cudaPitchedPtr(host + hoff, h->idim * es, h->idim * es, h->kdim);
    cudaPitchedPtr devp = make_cudaPitchedPtr(dev + doff, h->pitch3 * es, h->pitch3 * es, h->kdim);
    cp.srcPtr = to_dev ? hostp : devp;
    cp.dstPtr = to_dev ? devp : hostp;
    cp.extent = make_cudaExtent(w, nkc, njc);
    cp.kind = kind;
    CU(cudaMemcpy3DAsync(&cp, h->stream));
    return WRFB200_OK;
}

// whole-field copy
int copy_field(wrfb200_handle *h, int field, const void *host_src, void *host_dst)
{
    const wrfb200_domain &d = h->dom;
    return copy_range(h, field, host_src, host_dst, d.ims, d.ime, d.kms, d.kme, d.jms, d.jme);
}

}  // namespace

// -------------------------------------------------------------------------------------------------
// exported: misc
// -------------------------------------------------------------------------------------------------
int wrfb200_fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

extern "C" const char *wrfb200_last_error(void) { return g_err; }
extern "C" int wrfb200_version(void) { return WRFB200_VERSION; }

extern "C" int wrfb200_bounds(int periodic_x, int specified, int nested,
                              int ids, int ide, int jds, int jde,
                              int its, int ite, int jts, int jte, int kts, int kte,
                              int *i_start, int *i_end, int *j_start, int *j_end, int *k_start, int *k_end)
{
    // module_small_step_em.f90:91-106
    int is = its, ie = ite < ide - 1 ? ite : ide - 1;
    int js = jts, je = jte < jde - 1 ? jte : jde - 1;
    const bool spec = specified || nested;
    if (!periodic_x && spec) {
        is = its > ids + 1 ? its : ids + 1;
        ie = ite < ide - 2 ? ite : ide - 2;
    }
    if (spec) {
        js = jts > jds + 1 ? jts : jds + 1;
        je = jte < jde - 2 ? jte : jde - 2;
    }
    if (i_start) *i_start = is;
    if (i_end) *i_end = ie;
    if (j_start) *j_start = js;
    if (j_end) *j_end = je;
    if (k_start) *k_start = kts;
    if (k_end) *k_end = kte - 1;
    return WRFB200_OK;
}

// -------------------------------------------------------------------------------------------------
// exported: handle life cycle
// -------------------------------------------------------------------------------------------------
namespace {

int create(wrfb200_handle **out, const wrfb200_domain *dom, int device, int allocate, int esize)
{
    if (!out || !dom) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    *out = nullptr;
    if (int rc = check_domain(*dom)) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(WRFB200_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    if (device < 0) CU(cudaGetDevice(&device));
    if (device >= ndev) return fail(WRFB200_ERR_INVALID_ARG, "device %d out of range (%d devices)", device, ndev);
    wrfb200_handle *h = new (std::nothrow) wrfb200_handle();
    if (!h) return fail(WRFB200_ERR_NOMEM, "out of host memory");
    h->dom = *dom;
    h->device = device;
    h->esize = esize;
    h->idim = dom->ime - dom->ims + 1;
    h->jdim = dom->jme - dom->jms + 1;
    h->kdim = dom->kme - dom->kms + 1;
    if (allocate) {
        DeviceGuard g(device);
        if (!g.ok) { delete h; return fail(WRFB200_ERR_CUDA, "cannot select CUDA device %d", device); }
        h->pitch3 = h->pitch2 = round_up(h->idim, 128 / esize);  // 128-byte rows
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) {
            size_t n = is3d(f) ? (size_t)h->pitch3 * h->kdim * h->jdim
                     : is2d(f) ? (size_t)h->pitch2 * h->jdim
                               : (size_t)h->kdim;
            cudaError_t e = cudaMalloc(&h->d[f], n * esize);
            if (e == cudaSuccess) e = cudaMemsetAsync(h->d[f], 0, n * esize, nullptr);
            if (e != cudaSuccess) {
                for (int q = 0; q < f; ++q) cudaFree(h->d[q]);
                delete h;
                return fail(e == cudaErrorMemoryAllocation ? WRFB200_ERR_NOMEM : WRFB200_ERR_CUDA,
                            "cudaMalloc of field %d (%zu bytes) failed: %s", f, n * esize, cudaGetErrorString(e));
            }
            h->owned[f] = true;
        }
        cudaStreamSynchronize(nullptr);
    }
    *out = h;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_create(wrfb200_handle **out, const wrfb200_domain *dom, int device, int allocate)
{
    return create(out, dom, device, allocate, 4);
}

extern "C" int wrfb200_create_r8(wrfb200_handle **out, const wrfb200_domain *dom, int device, int allocate)
{
    return create(out, dom, device, allocate, 8);
}

extern "C" int wrfb200_destroy(wrfb200_handle *h)
{
    if (!h) return WRFB200_OK;
    DeviceGuard g(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream); else cudaDeviceSynchronize();
    wrfb200_comm_release(h);
    for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second);
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f)
        if (h->owned[f] && h->d[f]) cudaFree(h->d[f]);
    delete h;
    return WRFB200_OK;
}

extern "C" int wrfb200_set_stream(wrfb200_handle *h, void *cuda_stream)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    h->stream = (cudaStream_t)cuda_stream;
    return WRFB200_OK;
}

namespace {

int set_scalars(wrfb200_handle *h, double rdx, double rdy, double dts, double epssm)
{
    if (h->scalars_set && (rdx != h->rdx || rdy != h->rdy || dts != h->dts || epssm != h->epssm)) {
        for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second);     // captured kernels hold the old values
        h->graphs.clear();
    }
    h->rdx = rdx; h->rdy = rdy; h->dts = dts; h->epssm = epssm;
    h->scalars_set = true;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_set_scalars(wrfb200_handle *h, float rdx, float rdy, float dts, float epssm)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 4) return wrong_precision(h, "wrfb200_set_scalars");
    return set_scalars(h, rdx, rdy, dts, epssm);
}

extern "C" int wrfb200_set_scalars_r8(wrfb200_handle *h, double rdx, double rdy, double dts, double epssm)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 8) return wrong_precision(h, "wrfb200_set_scalars_r8");
    return set_scalars(h, rdx, rdy, dts, epssm);
}

extern "C" int wrfb200_set_kernel(wrfb200_handle *h, int kernel)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (kernel < WRFB200_KERNEL_AUTO || kernel > WRFB200_KERNEL_PIPE)
        return fail(WRFB200_ERR_INVALID_ARG, "bad kernel id %d", kernel);
    h->kernel = kernel;
    return WRFB200_OK;
}

namespace {

int bind_device(wrfb200_handle *h, int field, void *device_ptr, long pitch)
{
    if (field < 0 || field >= WRFB200_NUM_FIELDS) return fail(WRFB200_ERR_INVALID_ARG, "bad field id %d", field);
    if (!device_ptr) return fail(WRFB200_ERR_INVALID_ARG, "null device pointer");
    if (!is1d(field)) {
        if (pitch < h->idim) return fail(WRFB200_ERR_INVALID_ARG, "pitch %ld < row length %d", pitch, h->idim);
        long &ref = is3d(field) ? h->pitch3 : h->pitch2;
        bool other_bound = false;
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f)
            if (f != field && h->d[f] && (is3d(f) == is3d(field)) && !is1d(f)) other_bound = true;
        if (other_bound && ref != pitch)
            return fail(WRFB200_ERR_INVALID_ARG, "all %s fields of a patch must share one pitch (%ld vs %ld)",
                        is3d(field) ? "3-D" : "2-D", ref, pitch);
        ref = pitch;
    }
    if (h->owned[field] && h->d[field]) {
        DeviceGuard g(h->device);
        cudaFree(h->d[field]);
    }
    h->owned[field] = false;
    h->d[field] = static_cast<float *>(device_ptr);
    for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second);
    h->graphs.clear();
    return WRFB200_OK;
}

int device_ptr(wrfb200_handle *h, int field, void **ptr, long *pitch)
{
    if (field < 0 || field >= WRFB200_NUM_FIELDS) return fail(WRFB200_ERR_INVALID_ARG, "bad field id %d", field);
    if (ptr) *ptr = h->d[field];
    if (pitch) *pitch = is3d(field) ? h->pitch3 : is2d(field) ? h->pitch2 : h->kdim;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_bind_device(wrfb200_handle *h, int field, float *device_ptr, long pitch)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 4) return wrong_precision(h, "wrfb200_bind_device");
    return bind_device(h, field, device_ptr, pitch);
}

extern "C" int wrfb200_bind_device_r8(wrfb200_handle *h, int field, double *device_ptr, long pitch)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 8) return wrong_precision(h, "wrfb200_bind_device_r8");
    return bind_device(h, field, device_ptr, pitch);
}

extern "C" int wrfb200_device_ptr(wrfb200_handle *h, int field, float **ptr, long *pitch)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 4) return wrong_precision(h, "wrfb200_device_ptr");
    void *p = nullptr;
    const int rc = device_ptr(h, field, &p, pitch);
    if (ptr) *ptr = static_cast<float *>(p);
    return rc;
}

extern "C" int wrfb200_device_ptr_r8(wrfb200_handle *h, int field, double **ptr, long *pitch)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (h->esize != 8) return wrong_precision(h, "wrfb200_device_ptr_r8");
    void *p = nullptr;
    const int rc = device_ptr(h, field, &p, pitch);
    if (ptr) *ptr = static_cast<double *>(p);
    return rc;
}

// -------------------------------------------------------------------------------------------------
// exported: copies
// -------------------------------------------------------------------------------------------------
// Every copy verb checks the handle's precision against its own and then runs the one copy_range.
namespace {

int copy_verb(wrfb200_handle *h, int esize, const char *verb, int field, const void *src, void *dst,
              int i0, int i1, int k0, int k1, int j0, int j1)
{
    GUARD(h);
    if (h->esize != esize) return wrong_precision(h, verb);
    if (!src && !dst) return fail(WRFB200_ERR_INVALID_ARG, "null host pointer");
    return copy_range(h, field, src, dst, i0, i1, k0, k1, j0, j1);
}

int copy_verb_all(wrfb200_handle *h, int esize, const char *verb, int field, const void *src, void *dst)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    const wrfb200_domain &d = h->dom;
    return copy_verb(h, esize, verb, field, src, dst, d.ims, d.ime, d.kms, d.kme, d.jms, d.jme);
}

}  // namespace

extern "C" int wrfb200_upload_range(wrfb200_handle *h, int field, const float *host,
                                    int i0, int i1, int k0, int k1, int j0, int j1)
{
    return copy_verb(h, 4, "wrfb200_upload_range", field, host, nullptr, i0, i1, k0, k1, j0, j1);
}

extern "C" int wrfb200_download_range(wrfb200_handle *h, int field, float *host,
                                      int i0, int i1, int k0, int k1, int j0, int j1)
{
    return copy_verb(h, 4, "wrfb200_download_range", field, nullptr, host, i0, i1, k0, k1, j0, j1);
}

extern "C" int wrfb200_upload(wrfb200_handle *h, int field, const float *host)
{
    return copy_verb_all(h, 4, "wrfb200_upload", field, host, nullptr);
}

extern "C" int wrfb200_download(wrfb200_handle *h, int field, float *host)
{
    return copy_verb_all(h, 4, "wrfb200_download", field, nullptr, host);
}

extern "C" int wrfb200_upload_range_r8(wrfb200_handle *h, int field, const double *host,
                                       int i0, int i1, int k0, int k1, int j0, int j1)
{
    return copy_verb(h, 8, "wrfb200_upload_range_r8", field, host, nullptr, i0, i1, k0, k1, j0, j1);
}

extern "C" int wrfb200_download_range_r8(wrfb200_handle *h, int field, double *host,
                                         int i0, int i1, int k0, int k1, int j0, int j1)
{
    return copy_verb(h, 8, "wrfb200_download_range_r8", field, nullptr, host, i0, i1, k0, k1, j0, j1);
}

extern "C" int wrfb200_upload_r8(wrfb200_handle *h, int field, const double *host)
{
    return copy_verb_all(h, 8, "wrfb200_upload_r8", field, host, nullptr);
}

extern "C" int wrfb200_download_r8(wrfb200_handle *h, int field, double *host)
{
    return copy_verb_all(h, 8, "wrfb200_download_r8", field, nullptr, host);
}

// Resident-state verbs (SURVEY.md section 8b): the groups of arrays a host-resident caller moves at the three
// cadences of the acoustic loop.  A null pointer skips that array.  Replaces the per-call copies of every field,
// advance_mu_t_no_async.cu:245-306 (H2D) and :366-390 (D2H).
extern "C" int wrfb200_upload_constants(
    wrfb200_handle *h, const float *ww_1, const float *u_1, const float *v_1, const float *t_1, const float *ft,
    const float *mut, const float *muu, const float *muv, const float *mu_tend,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (int rc = wrfb200_require_r4(h, "wrfb200_upload_constants")) return rc;
    const int ids[] = {WRFB200_WW_1, WRFB200_U_1, WRFB200_V_1, WRFB200_T_1, WRFB200_FT, WRFB200_MUT, WRFB200_MUU,
                       WRFB200_MUV, WRFB200_MU_TEND, WRFB200_MSFUY, WRFB200_MSFVX_INV, WRFB200_MSFTX, WRFB200_MSFTY,
                       WRFB200_DNW, WRFB200_FNM, WRFB200_FNP, WRFB200_RDNW};
    const float *ptr[] = {ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend, msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw};
    for (int x = 0; x < 17; ++x)
        if (ptr[x]) if (int rc = wrfb200_upload(h, ids[x], ptr[x])) return rc;
    return WRFB200_OK;
}

extern "C" int wrfb200_upload_state(wrfb200_handle *h, const float *ww, const float *t, const float *mu)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (int rc = wrfb200_require_r4(h, "wrfb200_upload_state")) return rc;
    if (ww) if (int rc = wrfb200_upload(h, WRFB200_WW, ww)) return rc;
    if (t) if (int rc = wrfb200_upload(h, WRFB200_T, t)) return rc;
    if (mu) if (int rc = wrfb200_upload(h, WRFB200_MU, mu)) return rc;
    return WRFB200_OK;
}

extern "C" int wrfb200_set_uv(wrfb200_handle *h, const float *u, const float *v)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (int rc = wrfb200_require_r4(h, "wrfb200_set_uv")) return rc;
    if (u) if (int rc = wrfb200_upload(h, WRFB200_U, u)) return rc;
    if (v) if (int rc = wrfb200_upload(h, WRFB200_V, v)) return rc;
    return WRFB200_OK;
}

// Downloads exactly the cells the routine writes for the tile its:ite x jts:jte (everything else in the
// caller's arrays keeps its bytes, as with the Fortran).
extern "C" int wrfb200_download_outputs(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                                        float *ww, float *t, float *t_ave, float *mu, float *muave, float *muts, float *mudf)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (int rc = wrfb200_require_r4(h, "wrfb200_download_outputs")) return rc;
    const wrfb200_domain &d = h->dom;
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   its, ite, jts, jte, kts, kte, &is, &ie, &js, &je, &ks, &ke);
    if (is > ie || js > je || ks > ke) return WRFB200_OK;
    const int ids[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE, WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF};
    float *ptr[] = {ww, t, t_ave, mu, muave, muts, mudf};
    for (int x = 0; x < 7; ++x)
        if (ptr[x]) if (int rc = wrfb200_download_range(h, ids[x], ptr[x], is, ie, ks, ke, js, je)) return rc;
    return WRFB200_OK;
}

// -------------------------------------------------------------------------------------------------
// exported: stepping
// -------------------------------------------------------------------------------------------------
extern "C" int wrfb200_step(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte)
{
    GUARD(h);
    return step_on(h, its, ite, jts, jte, kts, kte, h->stream, h->kernel);
}

extern "C" int wrfb200_step_graph(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte, int nsteps)
{
    GUARD(h);
    if (nsteps <= 0) return WRFB200_OK;
    AmtParams p;
    AmtParamsR8 p8;
    bool empty = false;
    const int rc0 = h->esize == 8 ? make_params(h, its, ite, jts, jte, kts, kte, &p8, &empty)
                                  : make_params(h, its, ite, jts, jte, kts, kte, &p, &empty);
    if (rc0) return rc0;
    if (empty) return WRFB200_OK;
    const auto key = std::make_tuple(its, ite, jts, jte, kte, nsteps, h->kernel);
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
        // capture on a private stream so the caller's stream state is untouched
        cudaStream_t cs;
        CU(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        int rc = WRFB200_OK;
        if (e == cudaSuccess) {
            for (int s = 0; s < nsteps && rc == WRFB200_OK; ++s)
                rc = h->esize == 8 ? launch(h, p8, cs, h->kernel) : launch(h, p, cs, h->kernel);
            h->launches -= nsteps;                      // counted again on every replay below
            e = cudaStreamEndCapture(cs, &graph);
        }
        cudaStreamDestroy(cs);
        if (rc != WRFB200_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) return fail(WRFB200_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
        cudaGraphExec_t exec = nullptr;
        e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return fail(WRFB200_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
        it = h->graphs.emplace(key, exec).first;
    }
    CU(cudaGraphLaunch(it->second, h->stream));
    h->launches += nsteps;
    return WRFB200_OK;
}

extern "C" int wrfb200_sync(wrfb200_handle *h)
{
    GUARD(h);
    CU(cudaStreamSynchronize(h->stream));
    return WRFB200_OK;
}

extern "C" int wrfb200_launch_count(wrfb200_handle *h, long *count)
{
    if (!h || !count) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    *count = h->launches;
    return WRFB200_OK;
}

// -------------------------------------------------------------------------------------------------
// exported: the reference-compatible entry point (module_small_step_em.f90:7-18)
// -------------------------------------------------------------------------------------------------
namespace {

thread_local cudaStream_t g_default_stream = nullptr;
thread_local int g_default_kernel = WRFB200_KERNEL_AUTO;

constexpr int kMaxSlabs = 16;

struct Args {
    void *f[WRFB200_NUM_FIELDS];       // float or double arrays (the entry point's precision)
    double rdx, rdy, dts, epssm;
    wrfb200_domain dom;
    int its, ite, jts, jte, kts, kte;
};

// Per-thread cache of device mirrors for host-pointer callers (the reference allocates and frees
// 29 buffers on every call; we allocate once per distinct memory shape).
struct CompatCache {
    wrfb200_handle *h = nullptr;
    cudaStream_t up = nullptr, comp = nullptr, down = nullptr;      // upload / compute / download lanes
    cudaEvent_t ev_up[kMaxSlabs] = {}, ev_comp[kMaxSlabs] = {};
    void *stage[2] = {nullptr, nullptr};                            // dense landing buffers for H2D slabs
    size_t stage_bytes = 0;
    // acoustic-loop residency (wrfb200_acoustic_loop_begin/end): after the first call of a loop the device
    // mirrors hold everything; later calls with the SAME arrays and index sets move only u, v up
    bool loop_active = false, primed = false;
    Args primed_args{};
    void release()
    {
        primed = false;
        if (h) {
            DeviceGuard g(h->device);
            h->stream = nullptr;               // never synchronise on one of the lanes destroyed below
            wrfb200_destroy(h);                // device-wide sync, frees the mirrors
            h = nullptr;
            for (void *&b : stage) if (b) { cudaFree(b); b = nullptr; }
            stage_bytes = 0;
            for (cudaEvent_t &e : ev_up) if (e) { cudaEventDestroy(e); e = nullptr; }
            for (cudaEvent_t &e : ev_comp) if (e) { cudaEventDestroy(e); e = nullptr; }
            for (cudaStream_t *st : {&up, &comp, &down}) if (*st) { cudaStreamDestroy(*st); *st = nullptr; }
            (void)cudaGetLastError();
        }
    }
    ~CompatCache() { release(); }
};
thread_local CompatCache g_cache[2];        // [0]: binary32 calls, [1]: real*8 calls

// Device-pointer callers: the handle that wraps the caller's arrays (and its six TMA tensor maps) is kept
// between calls and re-used while the pointers and extents stay the same -- a 25-830 us step must not pay
// six cuTensorMapEncodeTiled and 26 cudaPointerGetAttributes every time.
struct DeviceCallCache {
    wrfb200_handle h;
    void *ptrs[WRFB200_NUM_FIELDS] = {};
    wrfb200_domain dom{};
    bool valid = false;
};
thread_local DeviceCallCache g_devcall[2];   // indexed like g_cache
thread_local int g_last_prec = 0;              // which of the two the most recent call used

bool same_shape(const wrfb200_domain &a, const wrfb200_domain &b)
{
    return a.ims == b.ims && a.ime == b.ime && a.jms == b.jms && a.jme == b.jme && a.kms == b.kms && a.kme == b.kme;
}
bool same_domain(const wrfb200_domain &a, const wrfb200_domain &b) { return std::memcmp(&a, &b, sizeof(a)) == 0; }

enum PtrKind { PTR_HOST, PTR_DEVICE, PTR_BAD };
PtrKind classify(const void *p, bool *pinned = nullptr)
{
    if (!p) return PTR_BAD;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return PTR_HOST; }
    if (pinned) *pinned = (a.type == cudaMemoryTypeHost);
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? PTR_DEVICE : PTR_HOST;
}

// ---- page-locking of caller arrays (opt-in) -------------------------------------------------------
// Pageable host memory reaches the GPU at a fraction of the link rate (the driver stages it through its own
// pinned buffer).  With pinning enabled, every host array of a compat call is cudaHostRegister'ed the first
// time it is seen and stays registered until wrfb200_release_cache() / wrfb200_host_unregister_all().
// OPT-IN because the caller must keep those arrays allocated for as long as they are registered: a freed and
// re-mapped virtual range with a stale registration would be DMA'd from the wrong pages.
std::mutex g_pin_mutex;
std::map<const void *, size_t> g_pinned;
int g_pin_mode = -1;                     // -1: read WRFB200_PIN_HOST on first use; 0 off; 1 on

bool pin_enabled()
{
    if (g_pin_mode < 0) { const char *e = getenv("WRFB200_PIN_HOST"); g_pin_mode = (e && atoi(e) > 0) ? 1 : 0; }
    return g_pin_mode == 1;
}

int pin_host(const void *p, size_t bytes)
{
    if (!p || bytes == 0) return WRFB200_OK;
    std::lock_guard<std::mutex> lock(g_pin_mutex);
    auto it = g_pinned.find(p);
    if (it != g_pinned.end() && it->second >= bytes) return WRFB200_OK;
    bool already = false;
    if (classify(p, &already) != PTR_HOST || already) return WRFB200_OK;       // already page-locked by the caller
    if (it != g_pinned.end()) { cudaHostUnregister(const_cast<void *>(p)); g_pinned.erase(it); }
    cudaError_t e = cudaHostRegister(const_cast<void *>(p), bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return WRFB200_OK; }     // stays pageable: slower, still correct
    g_pinned[p] = bytes;
    return WRFB200_OK;
}

void unpin_all()
{
    std::lock_guard<std::mutex> lock(g_pin_mutex);
    for (auto &kv : g_pinned) cudaHostUnregister(const_cast<void *>(kv.first));
    g_pinned.clear();
    (void)cudaGetLastError();
}

size_t field_bytes(const wrfb200_handle *h, int f)
{
    const size_t n = is3d(f) ? (size_t)h->idim * h->kdim * h->jdim : is2d(f) ? (size_t)h->idim * h->jdim : (size_t)h->kdim;
    return n * h->esize;
}

int run_device_in_place(const Args &a, int prec)
{
    // Caller-owned device arrays in the dense Fortran layout, wrapped in a (cached) handle.
    if (int rc = check_domain(a.dom)) return rc;
    DeviceCallCache &c = g_devcall[prec];
    int dev = 0;
    CU(cudaGetDevice(&dev));
    const bool hit = c.valid && c.h.device == dev && same_domain(c.dom, a.dom) &&
                     std::memcmp(c.ptrs, a.f, sizeof(c.ptrs)) == 0;
    if (!hit) {
        c.valid = false;
        c.h.dom = a.dom;
        c.h.device = dev;
        c.h.idim = a.dom.ime - a.dom.ims + 1;
        c.h.jdim = a.dom.jme - a.dom.jms + 1;
        c.h.kdim = a.dom.kme - a.dom.kms + 1;
        c.h.pitch3 = c.h.pitch2 = c.h.idim;
        c.h.esize = prec ? 8 : 4;
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) c.h.d[f] = static_cast<float *>(a.f[f]);
        c.h.maps.valid = 0;
        std::memcpy(c.ptrs, a.f, sizeof(c.ptrs));
        c.dom = a.dom;
        c.valid = true;
    }
    c.h.rdx = a.rdx; c.h.rdy = a.rdy; c.h.dts = a.dts; c.h.epssm = a.epssm; c.h.scalars_set = true;
    return step_on(&c.h, a.its, a.ite, a.jts, a.jte, a.kts, a.kte, g_default_stream, g_default_kernel);
}

// Host-pointer form of the operator.  The reference does alloc -> 26 blocking H2D copies -> launch ->
// sync -> 8 blocking D2H copies -> free on every call (advance_mu_t_no_async.cu:178-423).  Here the device
// mirrors are cached, and the call is software-pipelined over j-slabs on three streams: while slab s is
// being computed (all `nsteps` steps), slab s+1's inputs are in flight host->device and slab s-1's outputs
// device->host, so the PCIe link is busy in both directions.  Slabs are independent for this routine:
// every column needs only its own state plus the read-only one-row ring of u,v,t_1 etc. (SURVEY.md 8e),
// and the caller's u,v do not change between the steps of one call.
//
// Inside wrfb200_acoustic_loop_begin/end the first call uploads everything and later calls with the same
// arrays upload only u and v (what advance_uv changed; everything else on the device is this routine's own
// previous output or a loop constant) -- the per-small-step drop-in pattern of a host-resident model:
// 0.76 GB up and 1.15 GB down per step on 1800x1060x50 instead of 3.2 GB up.
int run_host_compat_body(const Args &a, int nsteps, wrfb200_handle *h, CompatCache &cc)
{
    const wrfb200_domain &d = a.dom;
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   a.its, a.ite, a.jts, a.jte, a.kts, a.kte, &is, &ie, &js, &je, &ks, &ke);
    if (is > ie || js > je || ks > ke) return WRFB200_OK;
    if (is - 1 < d.ims || ie + 1 > d.ime || js - 1 < d.jms || je + 1 > d.jme)
        return fail(WRFB200_ERR_INVALID_ARG,
                    "computed range i=%d..%d j=%d..%d needs a one-cell ring inside memory i=%d..%d j=%d..%d",
                    is, ie, js, je, d.ims, d.ime, d.jms, d.jme);
    CU(cudaStreamSynchronize(g_default_stream));          // the caller's earlier work on its stream is done

    static const int in3_all[] = {WRFB200_WW_1, WRFB200_U, WRFB200_U_1, WRFB200_V, WRFB200_V_1,
                                  WRFB200_T, WRFB200_T_1, WRFB200_FT};
    static const int in3_uv[] = {WRFB200_U, WRFB200_V};
    static const int in2[] = {WRFB200_MU, WRFB200_MUT, WRFB200_MUU, WRFB200_MUV, WRFB200_MU_TEND,
                              WRFB200_MSFUY, WRFB200_MSFVX_INV, WRFB200_MSFTX, WRFB200_MSFTY};
    static const int in1[] = {WRFB200_DNW, WRFB200_FNM, WRFB200_FNP, WRFB200_RDNW};
    static const int out3[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE};
    static const int out2[] = {WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF};

    // resident step: same arrays, same index sets, same scalars as the call that primed the mirrors
    const bool resident = cc.loop_active && cc.primed && std::memcmp(cc.primed_args.f, a.f, sizeof(a.f)) == 0 &&
                          same_domain(cc.primed_args.dom, a.dom) && cc.primed_args.its == a.its &&
                          cc.primed_args.ite == a.ite && cc.primed_args.jts == a.jts && cc.primed_args.jte == a.jte &&
                          cc.primed_args.kts == a.kts && cc.primed_args.kte == a.kte &&
                          cc.primed_args.rdx == a.rdx && cc.primed_args.rdy == a.rdy &&
                          cc.primed_args.dts == a.dts && cc.primed_args.epssm == a.epssm;
    cc.primed = false;                                    // until this call has completed
    const int *in3 = resident ? in3_uv : in3_all;
    const int n_in3 = resident ? 2 : 8;

    if (pin_enabled())
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) pin_host(a.f[f], field_bytes(h, f));

    // small operands first: 2-D and 1-D inputs, and ww at level 1 (the only level of ww the routine
    // reads, module_small_step_em.f90:159-161)
    h->stream = cc.up;
    if (!resident) {
        for (int f : in2) if (int rc = copy_field(h, f, a.f[f], nullptr)) return rc;
        for (int f : in1) if (int rc = copy_field(h, f, a.f[f], nullptr)) return rc;
        if (int rc = copy_range(h, WRFB200_WW, a.f[WRFB200_WW], nullptr, d.ims, d.ime, a.kts, a.kts, d.jms, d.jme)) return rc;
    }

    const int nj = je - js + 1;
    const size_t es = (size_t)h->esize;
    const size_t bytes3 = (size_t)h->idim * h->kdim * h->jdim * es;
    int nslab = 1;
    if (bytes3 >= ((size_t)16 << 20) && nj >= 32) nslab = nj / 16 < kMaxSlabs ? nj / 16 : kMaxSlabs;
    if (nslab > kMaxSlabs) nslab = kMaxSlabs;             // one event pair per slab
    int next_row = js - 1;                                // first row of the 3-D inputs not yet uploaded
    // A row-pitched (2-D) host->device copy runs ~18 % below a contiguous one on this link (40 vs 49 GB/s
    // measured, tools/pcie_probe.py).  When the mirror is padded, land each slab densely in a staging buffer
    // with ONE contiguous copy and re-pitch it on the device (HBM speed, negligible).
    const bool staged = (h->pitch3 != h->idim) && nslab > 1;
    const size_t slab_bytes = (size_t)(nj / nslab + 3) * h->kdim * h->idim * es;
    if (staged && cc.stage_bytes < slab_bytes) {
        for (void *&b : cc.stage) { if (b) cudaFree(b); b = nullptr; }
        cc.stage_bytes = 0;
        for (void *&b : cc.stage) CU(cudaMalloc(&b, slab_bytes));
        cc.stage_bytes = slab_bytes;
    }
    const int fpe = h->esize / (int)sizeof(float);         // the re-pitch kernel moves 4-byte words
    int flip = 0;
    for (int s = 0; s < nslab; ++s) {
        const int ja = js + (int)((long long)nj * s / nslab);
        const int jb = js + (int)((long long)nj * (s + 1) / nslab) - 1;
        // inputs through row jb+1 (the ring row the slab's last row reads)
        h->stream = cc.up;
        const int hi = jb + 1;
        if (next_row <= hi) {
            const long long nrows = (long long)(hi - next_row + 1) * h->kdim;
            const size_t hoff = (size_t)(next_row - d.jms) * h->kdim * h->idim;
            const size_t doff = (size_t)(next_row - d.jms) * h->kdim * h->pitch3;
            for (int x = 0; x < n_in3; ++x) {
                const int f = in3[x];
                if (!staged) {
                    if (int rc = copy_range(h, f, a.f[f], nullptr, d.ims, d.ime, d.kms, d.kme, next_row, hi)) return rc;
                    continue;
                }
                float *st = static_cast<float *>(cc.stage[flip]);
                flip ^= 1;
                CU(cudaMemcpyAsync(st, static_cast<const char *>(a.f[f]) + hoff * es, (size_t)nrows * h->idim * es,
                                   cudaMemcpyHostToDevice, cc.up));
                CU(wrfb200_repitch_rows(h->d[f] + doff * fpe, st, h->pitch3 * fpe, h->idim * fpe, nrows, cc.up));
                h->launches += 1;
            }
            next_row = hi + 1;
        }
        CU(cudaEventRecord(cc.ev_up[s], cc.up));
        // all steps of this slab
        CU(cudaStreamWaitEvent(cc.comp, cc.ev_up[s], 0));
        h->stream = cc.comp;
        for (int step = 0; step < nsteps; ++step)
            if (int rc = wrfb200_step(h, a.its, a.ite, ja, jb, a.kts, a.kte)) return rc;
        CU(cudaEventRecord(cc.ev_comp[s], cc.comp));
        // outputs: exactly the cells the Fortran writes
        CU(cudaStreamWaitEvent(cc.down, cc.ev_comp[s], 0));
        h->stream = cc.down;
        for (int f : out3) if (int rc = copy_range(h, f, nullptr, a.f[f], is, ie, ks, ke, ja, jb)) return rc;
        for (int f : out2) if (int rc = copy_range(h, f, nullptr, a.f[f], is, ie, 0, 0, ja, jb)) return rc;
    }
    CU(cudaStreamSynchronize(cc.up));
    CU(cudaStreamSynchronize(cc.comp));
    CU(cudaStreamSynchronize(cc.down));
    if (cc.loop_active) { cc.primed = true; cc.primed_args = a; }
    return WRFB200_OK;
}

int run_host_compat(const Args &a, int nsteps, int prec)
{
    if (int rc = check_domain(a.dom)) return rc;
    CompatCache &cc = g_cache[prec];
    if (cc.h && !same_shape(cc.h->dom, a.dom)) cc.release();
    if (!cc.h) {
        if (int rc = create(&cc.h, &a.dom, -1, 1, prec ? 8 : 4)) return rc;
        DeviceGuard g(cc.h->device);
        for (cudaStream_t *st : {&cc.up, &cc.comp, &cc.down})
            CU(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
        for (int i = 0; i < kMaxSlabs; ++i) {
            CU(cudaEventCreateWithFlags(&cc.ev_up[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&cc.ev_comp[i], cudaEventDisableTiming));
        }
    }
    wrfb200_handle *h = cc.h;
    GUARD(h);
    h->dom = a.dom;                       // same extents; domain dims / flags may differ between calls
    h->kernel = g_default_kernel;
    set_scalars(h, a.rdx, a.rdy, a.dts, a.epssm);
    const int rc = run_host_compat_body(a, nsteps, h, cc);
    if (rc != WRFB200_OK) {
        // an early return must not leave copies on the caller's arrays in flight, nor the cached handle
        // pointing at one of the internal lanes
        const std::string msg = wrfb200_last_error();
        for (cudaStream_t st : {cc.up, cc.comp, cc.down}) if (st) cudaStreamSynchronize(st);
        (void)cudaGetLastError();
        cc.primed = false;
        wrfb200_fail(rc, "%s", msg.c_str());
    }
    h->stream = g_default_stream;
    return rc;
}

// prec: 0 = binary32 entry points, 1 = real*8 entry points
int dispatch(Args &a, int nsteps, bool allow_device, int prec)
{
    g_last_prec = prec;
    DeviceCallCache &dc = g_devcall[prec];
    // device-pointer fast path: the very same arrays as the previous call need no re-classification
    if (allow_device && nsteps == 1 && dc.valid && std::memcmp(dc.ptrs, a.f, sizeof(a.f)) == 0)
        return run_device_in_place(a, prec);
    PtrKind kind = classify(a.f[0]);
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) {
        PtrKind k = classify(a.f[f]);
        if (k == PTR_BAD) return fail(WRFB200_ERR_INVALID_ARG, "field %d: null pointer", f);
        if (k != kind) return fail(WRFB200_ERR_INVALID_ARG, "field %d: host and device pointers mixed in one call", f);
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(WRFB200_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    if (kind == PTR_DEVICE) {
        if (!allow_device || nsteps != 1)
            return fail(WRFB200_ERR_INVALID_ARG, "this entry point takes host pointers; device-resident callers use wrfb200_step");
        return run_device_in_place(a, prec);
    }
    dc.valid = false;
    return run_host_compat(a, nsteps, prec);
}

}  // namespace

#define WRFB200_PACK_ARGS(a)                                                                              \
    Args a{};                                                                                             \
    a.f[WRFB200_WW] = (void *)ww;            a.f[WRFB200_WW_1] = (void *)ww_1;                            \
    a.f[WRFB200_U] = (void *)u;       a.f[WRFB200_U_1] = (void *)u_1;                                     \
    a.f[WRFB200_V] = (void *)v;       a.f[WRFB200_V_1] = (void *)v_1;                                     \
    a.f[WRFB200_T] = (void *)t;              a.f[WRFB200_T_1] = (void *)t_1;                              \
    a.f[WRFB200_T_AVE] = (void *)t_ave;      a.f[WRFB200_FT] = (void *)ft;                                \
    a.f[WRFB200_MU] = (void *)mu;            a.f[WRFB200_MUT] = (void *)mut;                              \
    a.f[WRFB200_MUAVE] = (void *)muave;      a.f[WRFB200_MUTS] = (void *)muts;                            \
    a.f[WRFB200_MUU] = (void *)muu;   a.f[WRFB200_MUV] = (void *)muv;                                     \
    a.f[WRFB200_MUDF] = (void *)mudf;        a.f[WRFB200_MU_TEND] = (void *)mu_tend;                      \
    a.f[WRFB200_MSFUY] = (void *)msfuy;                                                                   \
    a.f[WRFB200_MSFVX_INV] = (void *)msfvx_inv;                                                           \
    a.f[WRFB200_MSFTX] = (void *)msftx;                                                                   \
    a.f[WRFB200_MSFTY] = (void *)msfty;                                                                   \
    a.f[WRFB200_DNW] = (void *)dnw;   a.f[WRFB200_FNM] = (void *)fnm;                                     \
    a.f[WRFB200_FNP] = (void *)fnp;   a.f[WRFB200_RDNW] = (void *)rdnw;                                   \
    a.rdx = rdx; a.rdy = rdy; a.dts = dts; a.epssm = epssm;                                               \
    a.dom.ids = ids; a.dom.ide = ide; a.dom.jds = jds; a.dom.jde = jde; a.dom.kde = kde;                  \
    a.dom.ims = ims; a.dom.ime = ime; a.dom.jms = jms; a.dom.jme = jme; a.dom.kms = kms; a.dom.kme = kme; \
    a.dom.periodic_x = periodic_x; a.dom.specified = specified; a.dom.nested = nested;                    \
    a.its = its; a.ite = ite; a.jts = jts; a.jte = jte; a.kts = kts; a.kte = kte

extern "C" int wrfb200_advance_mu_t(
    float *ww, const float *ww_1, const float *u, const float *u_1, const float *v, const float *v_1,
    float *mu, const float *mut, float *muave, float *muts, const float *muu, const float *muv,
    float *mudf, float *t, const float *t_1, float *t_ave, const float *ft, const float *mu_tend,
    float rdx, float rdy, float dts, float epssm,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte)
{
    WRFB200_PACK_ARGS(a);
    return dispatch(a, 1, true, 0);
}

extern "C" int wrfb200_advance_mu_t_loop(
    float *ww, const float *ww_1, const float *u, const float *u_1, const float *v, const float *v_1,
    float *mu, const float *mut, float *muave, float *muts, const float *muu, const float *muv,
    float *mudf, float *t, const float *t_1, float *t_ave, const float *ft, const float *mu_tend,
    float rdx, float rdy, float dts, float epssm,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte,
    int nsteps)
{
    if (nsteps < 1) return fail(WRFB200_ERR_INVALID_ARG, "nsteps=%d", nsteps);
    WRFB200_PACK_ARGS(a);
    return dispatch(a, nsteps, false, 0);
}

// The same two entry points for WRF built with -r8 (default REAL = 8 bytes): double arrays and scalars,
// evaluated in binary64 by the real*8 kernels.
extern "C" int wrfb200_advance_mu_t_r8(
    double *ww, const double *ww_1, const double *u, const double *u_1, const double *v, const double *v_1,
    double *mu, const double *mut, double *muave, double *muts, const double *muu, const double *muv,
    double *mudf, double *t, const double *t_1, double *t_ave, const double *ft, const double *mu_tend,
    double rdx, double rdy, double dts, double epssm,
    const double *dnw, const double *fnm, const double *fnp, const double *rdnw,
    const double *msfuy, const double *msfvx_inv, const double *msftx, const double *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte)
{
    WRFB200_PACK_ARGS(a);
    return dispatch(a, 1, true, 1);
}

extern "C" int wrfb200_advance_mu_t_loop_r8(
    double *ww, const double *ww_1, const double *u, const double *u_1, const double *v, const double *v_1,
    double *mu, const double *mut, double *muave, double *muts, const double *muu, const double *muv,
    double *mudf, double *t, const double *t_1, double *t_ave, const double *ft, const double *mu_tend,
    double rdx, double rdy, double dts, double epssm,
    const double *dnw, const double *fnm, const double *fnp, const double *rdnw,
    const double *msfuy, const double *msfvx_inv, const double *msftx, const double *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte,
    int nsteps)
{
    if (nsteps < 1) return fail(WRFB200_ERR_INVALID_ARG, "nsteps=%d", nsteps);
    WRFB200_PACK_ARGS(a);
    return dispatch(a, nsteps, false, 1);
}

extern "C" int wrfb200_set_default_stream(void *cuda_stream)
{
    g_default_stream = (cudaStream_t)cuda_stream;
    return WRFB200_OK;
}

extern "C" int wrfb200_set_default_kernel(int kernel)
{
    if (kernel < WRFB200_KERNEL_AUTO || kernel > WRFB200_KERNEL_PIPE)
        return fail(WRFB200_ERR_INVALID_ARG, "bad kernel id %d", kernel);
    g_default_kernel = kernel;
    return WRFB200_OK;
}

extern "C" int wrfb200_release_cache(void)
{
    for (CompatCache &c : g_cache) c.release();
    for (DeviceCallCache &c : g_devcall) c.valid = false;
    unpin_all();
    return WRFB200_OK;
}

extern "C" int wrfb200_acoustic_loop_begin(void)
{
    for (CompatCache &c : g_cache) { c.loop_active = true; c.primed = false; }
    return WRFB200_OK;
}

extern "C" int wrfb200_acoustic_loop_end(void)
{
    for (CompatCache &c : g_cache) { c.loop_active = false; c.primed = false; }
    return WRFB200_OK;
}

extern "C" int wrfb200_set_host_pinning(int enable)
{
    g_pin_mode = enable ? 1 : 0;
    if (!enable) unpin_all();
    return WRFB200_OK;
}

extern "C" int wrfb200_host_register(const float *host, size_t bytes)
{
    if (!host) return fail(WRFB200_ERR_INVALID_ARG, "null host pointer");
    return pin_host(host, bytes);
}

extern "C" int wrfb200_host_unregister_all(void)
{
    unpin_all();
    return WRFB200_OK;
}

extern "C" int wrfb200_pipe_plan(const wrfb200_domain *dom, int its, int ite, int jts, int jte, int kts, int kte,
                                 int resident_blocks, long long *plan10)
{
    if (!dom || !plan10) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (int rc = check_domain(*dom)) return rc;
    if (kts != 1 || kte != dom->kde) return fail(WRFB200_ERR_UNSUPPORTED, "kts must be 1 and kte must equal kde");
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(dom->periodic_x, dom->specified, dom->nested, dom->ids, dom->ide, dom->jds, dom->jde,
                   its, ite, jts, jte, kts, kte, &is, &ie, &js, &je, &ks, &ke);
    AmtParams p{};
    p.i0 = is - dom->ims; p.i1 = ie - dom->ims;
    p.j0 = js - dom->jms; p.j1 = je - dom->jms;
    p.k0 = ks - dom->kms; p.nk = ke - ks + 1;
    if (!amt_pipe_plan(p, 0, resident_blocks > 0 ? resident_blocks : 2 * 148, plan10))
        return fail(WRFB200_ERR_INVALID_ARG, "empty index sets or no launch shape");
    return WRFB200_OK;
}

extern "C" int wrfb200_selftest_division(long long *mismatches, long long *checked, int dividends_per_divisor)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(WRFB200_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    if (dividends_per_divisor < 1) dividends_per_divisor = 1;
    unsigned long long bad = 0, n = 0;
    CU(amt_division_selftest(&bad, &n, dividends_per_divisor));
    if (mismatches) *mismatches = (long long)bad;
    if (checked) *checked = (long long)n;
    return WRFB200_OK;
}

extern "C" int wrfb200_last_kernel(wrfb200_handle *h, int *kernel)
{
    if (!h || !kernel) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    *kernel = h->last_kernel;
    return WRFB200_OK;
}

extern "C" int wrfb200_default_last_kernel(int *kernel)
{
    if (!kernel) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    const DeviceCallCache &dc = g_devcall[g_last_prec];
    const CompatCache &cc = g_cache[g_last_prec];
    *kernel = dc.valid ? dc.h.last_kernel : (cc.h ? cc.h->last_kernel : 0);
    return WRFB200_OK;
}
