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
#include <sched.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <tuple>
#include <type_traits>
#include <vector>

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

template <class P>
void wrfb200_fill_fields(const wrfb200_handle *h, P *p)
{
    using T = std::remove_pointer_t<decltype(P::ww)>;
    auto F = [h](int f) { return reinterpret_cast<T *>(h->d[f]); };
    p->ww = F(WRFB200_WW);       p->ww_1 = F(WRFB200_WW_1);
    p->u = F(WRFB200_U);         p->u_1 = F(WRFB200_U_1);
    p->v = F(WRFB200_V);         p->v_1 = F(WRFB200_V_1);
    p->t = F(WRFB200_T);         p->t_1 = F(WRFB200_T_1);
    p->t_ave = F(WRFB200_T_AVE); p->ft = F(WRFB200_FT);
    p->mu = F(WRFB200_MU);       p->mut = F(WRFB200_MUT);
    p->muave = F(WRFB200_MUAVE); p->muts = F(WRFB200_MUTS);
    p->muu = F(WRFB200_MUU);     p->muv = F(WRFB200_MUV);
    p->mudf = F(WRFB200_MUDF);   p->mu_tend = F(WRFB200_MU_TEND);
    p->msfuy = F(WRFB200_MSFUY); p->msfvx_inv = F(WRFB200_MSFVX_INV);
    p->msftx = F(WRFB200_MSFTX); p->msfty = F(WRFB200_MSFTY);
    p->dnw = F(WRFB200_DNW);     p->fnm = F(WRFB200_FNM);
    p->fnp = F(WRFB200_FNP);     p->rdnw = F(WRFB200_RDNW);
    p->pitch = h->pitch3;
    p->jstride = h->pitch3 * (long long)h->kdim;
    p->pitch2 = h->pitch2;
}
template void wrfb200_fill_fields(const wrfb200_handle *h, AmtParams *p);
template void wrfb200_fill_fields(const wrfb200_handle *h, AmtParamsR8 *p);

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

    P p{};
    wrfb200_fill_fields(h, &p);
    p.rdx = (T)h->rdx; p.rdy = (T)h->rdy; p.dts = (T)h->dts; p.epssm = (T)h->epssm;   // exact: stored from a T
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

int wrfb200_make_params(const wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                AmtParamsR8 *out, bool *empty)
{
    return make_params(h, its, ite, jts, jte, kts, kte, out, empty);
}

namespace {

// a kernel whose shared memory cannot hold the call's level count (amt_*_levels_fit)
int too_many_levels(const char *what, int nk, int max_levels)
{
    return fail(WRFB200_ERR_UNSUPPORTED, "the %s holds at most %d levels (nk=%d)", what, max_levels, nk);
}

int launch(wrfb200_handle *h, const AmtParams &p, cudaStream_t s, int kernel)
{
    cudaError_t e;
    int ran = kernel;
    int most = 0;
    if (kernel == WRFB200_KERNEL_COLUMN) {
        if (!amt_column_levels_fit(p, &most)) return too_many_levels("column kernel", p.nk, most);
        e = amt_launch_column(p, s);
    } else if (kernel == WRFB200_KERNEL_TILE) {
        if (!amt_tile_levels_fit(p, &most)) return too_many_levels("tile kernel", p.nk, most);
        if (!amt_tile_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "tile kernel needs 16-byte aligned fields and pitches that are multiples of 4");
        e = amt_launch_tile(p, s);
    } else if (kernel == WRFB200_KERNEL_PIPE) {
        if (!amt_pipe_levels_fit(p, &most)) return too_many_levels("pipe kernel", p.nk, most);
        if (!amt_pipe_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "pipe kernel needs 16-byte aligned fields and pitches that are multiples of 4");
        if (!amt_build_tma_maps(p, &h->maps)) return fail(WRFB200_ERR_CUDA, "cuTensorMapEncodeTiled failed");
        e = amt_launch_pipe(p, h->maps, s);
    } else {
        // AUTO: the TMA-pipelined tile kernel wherever the layout allows it; tiles narrower than a warp
        // of columns (e.g. the one-column strips behind an east halo) would stage 128-wide rows for
        // nothing, and unaligned caller layouts cannot be bulk-copied: those take the column kernel.
        const bool wide = (p.i1 - p.i0 + 1) >= 32;
        // Past the pipe kernel's level limit the column kernel runs, up to its own.
        if (wide && amt_pipe_supported(p) && amt_build_tma_maps(p, &h->maps)) {
            e = amt_launch_pipe(p, h->maps, s);
            ran = WRFB200_KERNEL_PIPE;
        } else {
            if (!amt_column_levels_fit(p, &most)) return too_many_levels("column kernel (AUTO's fallback)", p.nk, most);
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
    int most = 0;
    if (p.halo.enabled) {
        // a multi-GPU rank (comm.cu): the tile kernel with the halo exchange fused in; wrfb200_comm_init_r8 has
        // checked that the patch's layout and level count suit it
        if (!amt_tile_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "the fused real*8 exchange needs the tile kernel's layout and nk <= 220 (nk=%d)", p.nk);
        e = amt_launch_tile(p, s);
        ran = WRFB200_KERNEL_TILE;
    } else if (kernel == WRFB200_KERNEL_PIPE) {
        return fail(WRFB200_ERR_UNSUPPORTED, "the pipe kernel is binary32 only; a real*8 handle runs the tile or column kernel");
    } else if (kernel == WRFB200_KERNEL_COLUMN) {
        if (!amt_column_levels_fit(p, &most)) return too_many_levels("real*8 column kernel", p.nk, most);
        e = amt_launch_column(p, s);
    } else if (kernel == WRFB200_KERNEL_TILE) {
        if (!amt_tile_levels_fit(p, &most)) return too_many_levels("real*8 tile kernel", p.nk, most);
        if (!amt_tile_supported(p))
            return fail(WRFB200_ERR_UNSUPPORTED, "real*8 tile kernel needs 16-byte aligned fields and pitches of an even "
                                                 "number of doubles");
        e = amt_launch_tile(p, s);
    } else {
        // AUTO: tiles narrower than a warp of columns take the column kernel, as for binary32; so do level counts
        // past the tile kernel's limit, up to the column kernel's own
        const bool wide = (p.i1 - p.i0 + 1) >= 32;
        if (wide && amt_tile_supported(p)) {
            e = amt_launch_tile(p, s);
            ran = WRFB200_KERNEL_TILE;
        } else {
            if (!amt_column_levels_fit(p, &most)) return too_many_levels("real*8 column kernel (AUTO's fallback)", p.nk, most);
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

int wrfb200_launch_params(wrfb200_handle *h, const AmtParamsR8 &p, cudaStream_t s, int kernel)
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

// elements of the device mirror of field f: rows of `pitch` elements
size_t mirror_elems(int f, long pitch, long kdim, long jdim)
{
    return is3d(f) ? (size_t)pitch * kdim * jdim : is2d(f) ? (size_t)pitch * jdim : (size_t)kdim;
}

// bytes of the 26 mirrors create() allocates for the memory extents of d
size_t mirror_bytes(const wrfb200_domain &d, int esize)
{
    const long pitch = round_up(d.ime - d.ims + 1, 128 / esize), jdim = d.jme - d.jms + 1, kdim = d.kme - d.kms + 1;
    size_t n = 0;
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) n += mirror_elems(f, pitch, kdim, jdim);
    return n * esize;
}

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
            const size_t n = mirror_elems(f, is3d(f) ? h->pitch3 : h->pitch2, h->kdim, h->jdim);
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
// advance_mu_t_no_async.cu:245-306 (H2D) and :366-390 (D2H).  Each verb has a binary32 and an _r8 form (WRF built
// with -r8) that run one body with the verb's element size and name.
namespace {

const int kConstantFields[] = {WRFB200_WW_1, WRFB200_U_1, WRFB200_V_1, WRFB200_T_1, WRFB200_FT, WRFB200_MUT,
                               WRFB200_MUU, WRFB200_MUV, WRFB200_MU_TEND, WRFB200_MSFUY, WRFB200_MSFVX_INV,
                               WRFB200_MSFTX, WRFB200_MSFTY, WRFB200_DNW, WRFB200_FNM, WRFB200_FNP, WRFB200_RDNW};
const int kStateFields[] = {WRFB200_WW, WRFB200_T, WRFB200_MU};
const int kUVFields[] = {WRFB200_U, WRFB200_V};
const int kOutputFields[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE, WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS,
                             WRFB200_MUDF};

// a binary32 verb refuses a real*8 handle as binary32 only; an _r8 verb names the real*4 handle it was given
int resident_precision(const wrfb200_handle *h, int esize, const char *verb)
{
    if (!h) return fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (esize == 4) return wrfb200_require_r4(h, verb);
    return h->esize == 8 ? WRFB200_OK : wrong_precision(h, verb);
}

template <size_t N>
int upload_fields(wrfb200_handle *h, int esize, const char *verb, const int (&ids)[N], const void *const (&host)[N])
{
    if (int rc = resident_precision(h, esize, verb)) return rc;
    for (size_t x = 0; x < N; ++x)
        if (host[x]) if (int rc = copy_verb_all(h, esize, verb, ids[x], host[x], nullptr)) return rc;
    return WRFB200_OK;
}

// Downloads exactly the cells the routine writes for the tile its:ite x jts:jte (everything else in the
// caller's arrays keeps its bytes, as with the Fortran).
int download_outputs(wrfb200_handle *h, int esize, const char *verb, int its, int ite, int jts, int jte, int kts,
                     int kte, void *const (&host)[7])
{
    if (int rc = resident_precision(h, esize, verb)) return rc;
    const wrfb200_domain &d = h->dom;
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   its, ite, jts, jte, kts, kte, &is, &ie, &js, &je, &ks, &ke);
    if (is > ie || js > je || ks > ke) return WRFB200_OK;
    for (int x = 0; x < 7; ++x)
        if (host[x])
            if (int rc = copy_verb(h, esize, verb, kOutputFields[x], nullptr, host[x], is, ie, ks, ke, js, je)) return rc;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_upload_constants(
    wrfb200_handle *h, const float *ww_1, const float *u_1, const float *v_1, const float *t_1, const float *ft,
    const float *mut, const float *muu, const float *muv, const float *mu_tend,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw)
{
    return upload_fields(h, 4, "wrfb200_upload_constants", kConstantFields,
                         {ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend, msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw});
}

extern "C" int wrfb200_upload_state(wrfb200_handle *h, const float *ww, const float *t, const float *mu)
{
    return upload_fields(h, 4, "wrfb200_upload_state", kStateFields, {ww, t, mu});
}

extern "C" int wrfb200_set_uv(wrfb200_handle *h, const float *u, const float *v)
{
    return upload_fields(h, 4, "wrfb200_set_uv", kUVFields, {u, v});
}

extern "C" int wrfb200_download_outputs(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                                        float *ww, float *t, float *t_ave, float *mu, float *muave, float *muts, float *mudf)
{
    return download_outputs(h, 4, "wrfb200_download_outputs", its, ite, jts, jte, kts, kte,
                            {ww, t, t_ave, mu, muave, muts, mudf});
}

extern "C" int wrfb200_upload_constants_r8(
    wrfb200_handle *h, const double *ww_1, const double *u_1, const double *v_1, const double *t_1, const double *ft,
    const double *mut, const double *muu, const double *muv, const double *mu_tend,
    const double *msfuy, const double *msfvx_inv, const double *msftx, const double *msfty,
    const double *dnw, const double *fnm, const double *fnp, const double *rdnw)
{
    return upload_fields(h, 8, "wrfb200_upload_constants_r8", kConstantFields,
                         {ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend, msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw});
}

extern "C" int wrfb200_upload_state_r8(wrfb200_handle *h, const double *ww, const double *t, const double *mu)
{
    return upload_fields(h, 8, "wrfb200_upload_state_r8", kStateFields, {ww, t, mu});
}

extern "C" int wrfb200_set_uv_r8(wrfb200_handle *h, const double *u, const double *v)
{
    return upload_fields(h, 8, "wrfb200_set_uv_r8", kUVFields, {u, v});
}

extern "C" int wrfb200_download_outputs_r8(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                                           double *ww, double *t, double *t_ave, double *mu, double *muave,
                                           double *muts, double *mudf)
{
    return download_outputs(h, 8, "wrfb200_download_outputs_r8", its, ite, jts, jte, kts, kte,
                            {ww, t, t_ave, mu, muave, muts, mudf});
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
thread_local std::vector<int> g_default_devices;      // wrfb200_set_default_devices; empty: the current device only

constexpr int kMaxSlabs = 16;
// Bounce buffers of the staged route: 0, 1 take uploads in turn; 2..4 the downloads of ww, t, t_ave; 5..8 those of
// the four 2-D outputs.  0..4 hold one slab of one 3-D field, 5..8 the same rows of a 2-D one.
constexpr int kBounceUp = 2, kBounce3 = 5, kBounce = 9;

struct Args {
    void *f[WRFB200_NUM_FIELDS];       // float or double arrays (the entry point's precision)
    double rdx, rdy, dts, epssm;
    wrfb200_domain dom;
    int its, ite, jts, jte, kts, kte;
};

// Per-thread cache of device mirrors for host-pointer callers (the reference allocates and frees 29 buffers on every
// call; we allocate once per domain).  A nested WRF run calls the routine for the parent and for each nest in turn,
// with other memory extents, so a cache keeps the mirrors of up to kMaxDomains domains, most recently used first,
// and a switch back to one of them allocates nothing.  Each domain owns its mirrors, device staging buffers and
// residency; the lanes, their events and the pinned bounce buffers belong to the cache and serve all its domains
// one call at a time, so N domains do not mean N sets of page-locked memory.
constexpr size_t kMaxDomains = 8;

// One domain of a cache, keyed by its device and memory extents (not by the caller's array addresses: solve_em
// passes locals that may move between calls).
struct DomainEntry {
    wrfb200_handle *h = nullptr;                                    // owns the 26 mirrors
    void *stage[2] = {nullptr, nullptr};                            // dense landing buffers for H2D slabs
    size_t stage_bytes = 0;
    // acoustic-loop residency (wrfb200_acoustic_loop_begin/end): after the first call of a loop the device
    // mirrors hold everything; later calls with the SAME arrays and index sets move only u, v up
    bool primed = false;
    Args primed_args{};
    ~DomainEntry()
    {
        if (!h) return;
        DeviceGuard g(h->device);
        h->stream = nullptr;               // never synchronise on a lane (they outlive the entry or are gone)
        wrfb200_destroy(h);                // device-wide sync, frees the mirrors
        for (void *b : stage) if (b) cudaFree(b);
        (void)cudaGetLastError();
    }
};

struct CompatCache {
    std::vector<std::unique_ptr<DomainEntry>> doms;                 // most recently used first
    int lane_device = -1;                                           // the device of the lanes and events
    cudaStream_t up = nullptr, comp = nullptr, down = nullptr;      // upload / compute / download lanes
    cudaEvent_t ev_up[kMaxSlabs] = {}, ev_comp[kMaxSlabs] = {};
    // staged route (pageable caller arrays): pinned bounce buffers, allocated on first use and grown to the largest
    // slab seen, and per buffer the event of the device copy that last read or filled it
    void *bounce[kBounce] = {};
    cudaEvent_t ev_bounce[kBounce] = {};
    size_t bounce3_bytes = 0, bounce2_bytes = 0;
    int next_up = 0;                                                // the upload buffer filled next
    bool loop_active = false;                                       // between wrfb200_acoustic_loop_begin and _end
    void forget()
    {
        for (auto &e : doms) e->primed = false;
    }
    void release_lanes()
    {
        if (lane_device < 0) return;
        DeviceGuard g(lane_device);
        for (cudaStream_t st : {up, comp, down}) if (st) cudaStreamSynchronize(st);
        for (void *&b : bounce) if (b) { cudaFreeHost(b); b = nullptr; }
        for (cudaEvent_t &e : ev_bounce) if (e) { cudaEventDestroy(e); e = nullptr; }
        bounce3_bytes = bounce2_bytes = 0;
        for (cudaEvent_t &e : ev_up) if (e) { cudaEventDestroy(e); e = nullptr; }
        for (cudaEvent_t &e : ev_comp) if (e) { cudaEventDestroy(e); e = nullptr; }
        for (cudaStream_t *st : {&up, &comp, &down}) if (*st) { cudaStreamDestroy(*st); *st = nullptr; }
        lane_device = -1;
        (void)cudaGetLastError();
    }
    void release()
    {
        doms.clear();
        release_lanes();
    }
    ~CompatCache() { release(); }
};
thread_local CompatCache g_cache[2];        // [0]: binary32 calls, [1]: real*8 calls

// wrfb200_default_last_cache: what the thread's last call did with its cache (wrfb200_cache; -1: no call has
// reached its cache yet)
thread_local int g_last_cache = -1;

// the same arrays, index sets and scalars as the call that primed a resident tile
bool same_call(const Args &p, const Args &a)
{
    return std::memcmp(p.f, a.f, sizeof(a.f)) == 0 && std::memcmp(&p.dom, &a.dom, sizeof(a.dom)) == 0 &&
           p.its == a.its && p.ite == a.ite && p.jts == a.jts && p.jte == a.jte && p.kts == a.kts &&
           p.kte == a.kte && p.rdx == a.rdx && p.rdy == a.rdy && p.dts == a.dts && p.epssm == a.epssm;
}

// ---- shared-tiles mode (wrfb200_set_shared_tiles) ----------------------------------------------------
// The host-array calls of every thread that pass the same 26 arrays and memory extents are tiles of ONE patch:
// one set of mirrors on the patch device, and acoustic-loop residency kept per tile (its..ite x jts..jte) in the
// patch rather than per thread, since an OpenMP schedule may hand a tile to another thread each step.  Each thread
// keeps its own lanes, events, staging buffers and a handle (allocate=0) bound to the shared mirrors, so that no
// handle field is written by two threads.
std::atomic<int> g_shared_mode{-1};          // -1: read WRFB200_SHARED_TILES on first use; 0 off; 1 on
std::atomic<int> g_shared_device{-1};        // the patch device (-1: not yet recorded)
std::atomic<bool> g_shared_loop{false};      // between wrfb200_acoustic_loop_begin and _end
std::mutex g_shared_mutex;                   // guards g_shared, g_shared_next_id and g_tile_threads

struct SharedPatch {
    wrfb200_handle *h = nullptr;             // owns the 26 mirrors
    int prec = 0;
    long id = 0;                             // unique in the process: a thread's handle re-binds when it changes
    void *ptrs[WRFB200_NUM_FIELDS] = {};     // the caller's 26 host arrays
    std::mutex mutex;                       // guards `primed`
    std::map<std::tuple<int, int, int, int>, Args> primed;   // tiles whose state is device-resident

    static std::tuple<int, int, int, int> key(const Args &a) { return std::make_tuple(a.its, a.ite, a.jts, a.jte); }
    // true when this tile was primed by the same call in the current loop; the tile counts as not primed until
    // this call has completed
    bool take(const Args &a)
    {
        std::lock_guard<std::mutex> lock(mutex);
        auto it = primed.find(key(a));
        if (it == primed.end()) return false;
        const bool same = same_call(it->second, a);
        primed.erase(it);
        return same && g_shared_loop.load();
    }
    void put(const Args &a)
    {
        std::lock_guard<std::mutex> lock(mutex);
        primed[key(a)] = a;
    }
    void forget()
    {
        std::lock_guard<std::mutex> lock(mutex);
        primed.clear();
    }
};
std::vector<std::unique_ptr<SharedPatch>> g_shared;
long g_shared_next_id = 1;

// A thread's state for shared calls, listed process-wide so that wrfb200_set_shared_tiles(0) and
// wrfb200_release_cache can free it whichever thread calls them.
struct TileThread;
std::vector<TileThread *> g_tile_threads;
struct TileThread {
    CompatCache c[2];                        // indexed like g_cache
    long bound[2] = {0, 0};                  // SharedPatch::id the handle's fields are bound to (0: none)
    bool listed = false;
    void enlist()
    {
        if (listed) return;
        std::lock_guard<std::mutex> lock(g_shared_mutex);
        g_tile_threads.push_back(this);
        listed = true;
    }
    void release()
    {
        for (int p = 0; p < 2; ++p) { c[p].release(); bound[p] = 0; }
    }
    ~TileThread()
    {
        std::lock_guard<std::mutex> lock(g_shared_mutex);
        for (size_t x = 0; x < g_tile_threads.size(); ++x)
            if (g_tile_threads[x] == this) { g_tile_threads.erase(g_tile_threads.begin() + x); break; }
        release();
    }
};
thread_local TileThread g_tiles;

bool shared_enabled()
{
    int m = g_shared_mode.load();
    if (m < 0) {
        const char *e = getenv("WRFB200_SHARED_TILES");
        g_shared_mode.compare_exchange_strong(m, (e && atoi(e) > 0) ? 1 : 0);
        m = g_shared_mode.load();
    }
    return m == 1;
}

// The patch device.  wrfb200_set_shared_tiles(1) records it; when the environment turned the mode on, the first
// thread that asks (wrfb200_acoustic_loop_begin or a host-array call) records its current device.
int shared_device(int *dev)
{
    int d = g_shared_device.load();
    if (d < 0) {
        int cur = 0;
        CU(cudaGetDevice(&cur));
        g_shared_device.compare_exchange_strong(d, cur);
        d = g_shared_device.load();
    }
    *dev = d;
    return WRFB200_OK;
}

// frees every shared patch and every thread's state for shared calls; no call may be in flight
void release_shared()
{
    std::lock_guard<std::mutex> lock(g_shared_mutex);
    for (TileThread *t : g_tile_threads) t->release();
    for (auto &sp : g_shared) wrfb200_destroy(sp->h);
    g_shared.clear();
}

// Device-pointer callers: the handle that wraps the caller's arrays (and its six TMA tensor maps) is kept
// between calls and re-used while the pointers and extents stay the same -- a 25-830 us step must not pay
// six cuTensorMapEncodeTiled and 26 cudaPointerGetAttributes every time.  A thread keeps kDeviceCalls of them
// per precision, the least recently used one replaced first, so that a nested run alternating its domains keeps
// the wrapper of each.  A host-pointer call drops them all.
constexpr int kDeviceCalls = 4;
struct DeviceCallCache {
    wrfb200_handle h;
    void *ptrs[WRFB200_NUM_FIELDS] = {};
    wrfb200_domain dom{};
    bool valid = false;
    long used = 0;                           // g_devcall_clock at its last call
};
thread_local DeviceCallCache g_devcall[2][kDeviceCalls];   // indexed like g_cache
thread_local long g_devcall_clock = 0;
thread_local int g_last_prec = 0;              // which of the two the most recent call used

// the entry of the thread's most recent device-pointer call of precision prec, if none has been dropped since
const DeviceCallCache *last_devcall(int prec)
{
    const DeviceCallCache *last = nullptr;
    for (const DeviceCallCache &c : g_devcall[prec])
        if (c.valid && (!last || c.used > last->used)) last = &c;
    return last;
}

void drop_devcalls(int prec)
{
    for (DeviceCallCache &c : g_devcall[prec]) c.valid = false;
}

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
    // portable: every device treats the range as page-locked (a host call may be split over several GPUs)
    cudaError_t e = cudaHostRegister(const_cast<void *>(p), bytes, cudaHostRegisterPortable);
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

// bytes of the dense host array of `field` with the memory extents of `d`
size_t field_bytes(const wrfb200_domain &d, int f, size_t esize)
{
    const size_t idim = d.ime - d.ims + 1, jdim = d.jme - d.jms + 1, kdim = d.kme - d.kms + 1;
    return (is3d(f) ? idim * kdim * jdim : is2d(f) ? idim * jdim : kdim) * esize;
}

// ---- staged route for pageable caller arrays --------------------------------------------------------
// The driver stages a pageable cudaMemcpyAsync itself, from the calling thread, at a fraction of the link rate.
// The staged route copies pageable arrays itself: host workers move a box of rows between the caller's array and
// a pinned bounce buffer of the cache, and the device copy starts or ends in that buffer, so it runs at the pinned
// rate while the workers fill the other buffer.  The caller's memory is never registered, so it may be freed and
// re-allocated at any time between calls.

// Host threads for those copies: one pool per process, shared by concurrent calls, sized to the CPUs the process may
// run on (a WRF MPI rank bound to a few cores gets a few threads), at most 16.  The workers make no CUDA call.
class HostPool {
public:
    const pid_t owner = getpid();

    explicit HostPool(int n)
    {
        for (int t = 0; t < n; ++t) {
            try {
                threads_.emplace_back([this] { work(); });
            } catch (const std::exception &) {
                break;                                    // fewer workers: slower, still correct
            }
        }
    }
    ~HostPool()
    {
        {
            std::lock_guard<std::mutex> lock(m_);
            stop_ = true;
        }
        work_cv_.notify_all();
        for (std::thread &t : threads_) t.join();
    }
    // fn(lo, hi) over [0, n) cut into contiguous ranges, one per worker, each of at least `grain`; returns when all
    // have run.  A job of one range runs in the calling thread.
    void run(long n, long grain, const std::function<void(long, long)> &fn)
    {
        long parts = grain > 0 ? n / grain : n;
        if (parts > (long)threads_.size()) parts = (long)threads_.size();
        if (parts <= 1) {
            if (n > 0) fn(0, n);
            return;
        }
        int left = (int)parts;
        {
            std::lock_guard<std::mutex> lock(m_);
            for (long p = 0; p < parts; ++p) q_.push_back(Task{&fn, n * p / parts, n * (p + 1) / parts, &left});
        }
        work_cv_.notify_all();
        std::unique_lock<std::mutex> lock(m_);
        done_cv_.wait(lock, [&] { return left == 0; });
    }

private:
    struct Task {
        const std::function<void(long, long)> *fn;
        long lo, hi;
        int *left;                                        // ranges of the job still running, under m_
    };
    void work()
    {
        std::unique_lock<std::mutex> lock(m_);
        for (;;) {
            work_cv_.wait(lock, [this] { return stop_ || !q_.empty(); });
            if (q_.empty()) return;
            const Task t = q_.front();
            q_.pop_front();
            lock.unlock();
            (*t.fn)(t.lo, t.hi);
            lock.lock();
            if (--*t.left == 0) done_cv_.notify_all();
        }
    }
    std::mutex m_;
    std::condition_variable work_cv_, done_cv_;
    std::deque<Task> q_;
    bool stop_ = false;
    std::vector<std::thread> threads_;
};

std::mutex g_pool_mutex;
HostPool *g_pool = nullptr;

int pool_size()
{
    cpu_set_t set;
    int n = sched_getaffinity(0, sizeof(set), &set) == 0 ? CPU_COUNT(&set) : (int)std::thread::hardware_concurrency();
    return n < 1 ? 1 : n > 16 ? 16 : n;
}

// the pool, started on first use
HostPool *host_pool()
{
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool && g_pool->owner != getpid()) g_pool = nullptr;      // inherited across fork(): no threads here
    if (!g_pool) g_pool = new (std::nothrow) HostPool(pool_size());
    return g_pool;
}

// Stops and joins the pool.  A pool inherited across fork() has no threads in this process: it is forgotten.
void stop_pool()
{
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool && g_pool->owner == getpid()) delete g_pool;
    g_pool = nullptr;
}

struct PoolReaper {
    ~PoolReaper() { stop_pool(); }                        // library unload / process exit
} g_pool_reaper;

// A box of one field, Fortran-numbered: i0..i1 x k0..k1 x j0..j1 (k0 = k1 = 0 for a 2-D field).  In a bounce
// buffer it is dense in the caller's order: rows of i, k next, j slowest.
struct Box {
    int f, i0, i1, k0, k1, j0, j1;
};

// Moves box b between the caller's array `arr` and the dense buffer `buf` on the pool's workers.
void host_box(HostPool *pool, const wrfb200_handle *h, const Box &b, char *arr, char *buf, bool gather)
{
    const wrfb200_domain &d = h->dom;
    const size_t es = (size_t)h->esize;
    const long kh = is3d(b.f) ? h->kdim : 1, kb = is3d(b.f) ? d.kms : 0;
    const long nk = b.k1 - b.k0 + 1, nrows = nk * (b.j1 - b.j0 + 1);
    const size_t w = (size_t)(b.i1 - b.i0 + 1) * es;
    char *first = arr + (((size_t)(b.j0 - d.jms) * kh + (b.k0 - kb)) * h->idim + (b.i0 - d.ims)) * es;
    const bool dense = w == (size_t)h->idim * es && nk == kh;       // one contiguous range of the array
    const std::function<void(long, long)> fn = [&](long lo, long hi) {
        if (dense) {
            if (gather) std::memcpy(buf + lo * w, first + lo * w, (hi - lo) * w);
            else        std::memcpy(first + lo * w, buf + lo * w, (hi - lo) * w);
            return;
        }
        for (long r = lo; r < hi; ++r) {
            char *row = first + ((size_t)(r / nk) * kh + (size_t)(r % nk)) * h->idim * es;
            if (gather) std::memcpy(buf + r * w, row, w);
            else        std::memcpy(row, buf + r * w, w);
        }
    };
    // ranges of at least 1 MB: a smaller copy is not worth waking a worker
    const long grain = (long)(((size_t)1 << 20) / w) + 1;
    if (pool) pool->run(nrows, grain, fn);
    else      fn(0, nrows);
}

// The device half: box b between the dense buffer `buf` (pinned) and the mirror, on stream s.
int device_box(wrfb200_handle *h, const Box &b, char *buf, bool to_dev, cudaStream_t s)
{
    const wrfb200_domain &d = h->dom;
    const size_t es = (size_t)h->esize;
    const bool three = is3d(b.f);
    const size_t dpitch = (size_t)(three ? h->pitch3 : h->pitch2) * es;
    const size_t kd = three ? h->kdim : 1;
    const long kb = three ? d.kms : 0;
    const size_t nk = b.k1 - b.k0 + 1, nj = b.j1 - b.j0 + 1, w = (size_t)(b.i1 - b.i0 + 1) * es;
    char *dev = reinterpret_cast<char *>(h->d[b.f]) +
                ((size_t)(b.j0 - d.jms) * kd + (size_t)(b.k0 - kb)) * dpitch + (size_t)(b.i0 - d.ims) * es;
    const cudaMemcpyKind kind = to_dev ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    if (nk == kd) {
        // whole columns: rows equally spaced across k and j
        if (to_dev) CU(cudaMemcpy2DAsync(dev, dpitch, buf, w, w, nk * nj, kind, s));
        else        CU(cudaMemcpy2DAsync(buf, w, dev, dpitch, w, nk * nj, kind, s));
        return WRFB200_OK;
    }
    cudaMemcpy3DParms cp{};
    const cudaPitchedPtr bufp = make_cudaPitchedPtr(buf, w, w, nk);
    const cudaPitchedPtr devp = make_cudaPitchedPtr(dev, dpitch, dpitch, kd);
    cp.srcPtr = to_dev ? bufp : devp;
    cp.dstPtr = to_dev ? devp : bufp;
    cp.extent = make_cudaExtent(w, nk, nj);
    cp.kind = kind;
    CU(cudaMemcpy3DAsync(&cp, s));
    return WRFB200_OK;
}

// wrfb200_bounce_allocations: sets of bounce buffers allocated by every cache of the process
std::atomic<long> g_bounce_allocs{0};

// The cache's bounce buffers, at least b3 bytes (0..4) and b2 bytes (5..8), and their events.  They only grow, each
// size to the largest seen, so that calls of the cache's domains in turn find them large enough whichever of the two
// sizes each domain needs more of.
int ensure_bounce(CompatCache &cc, size_t b3, size_t b2)
{
    if (cc.bounce3_bytes >= b3 && cc.bounce2_bytes >= b2) return WRFB200_OK;
    b3 = std::max(b3, cc.bounce3_bytes);
    b2 = std::max(b2, cc.bounce2_bytes);
    g_bounce_allocs.fetch_add(1);
    for (void *&b : cc.bounce) if (b) { cudaFreeHost(b); b = nullptr; }
    cc.bounce3_bytes = cc.bounce2_bytes = 0;
    for (int x = 0; x < kBounce; ++x) {
        // portable: a part of a split call copies on its own device
        CU(cudaHostAlloc(&cc.bounce[x], x < kBounce3 ? b3 : b2, cudaHostAllocPortable));
        if (!cc.ev_bounce[x]) CU(cudaEventCreateWithFlags(&cc.ev_bounce[x], cudaEventDisableTiming));
    }
    cc.bounce3_bytes = b3;
    cc.bounce2_bytes = b2;
    return WRFB200_OK;
}

// Staged upload of box b of the caller's array `arr`, in runs of j-planes that fit one upload buffer.  A buffer is
// refilled only after the copy that last read it has finished.  `land` (a device staging buffer; 3-D boxes of
// whole rows and columns only): each run lands there densely and is re-pitched into the mirror.
int upload_box(CompatCache &cc, wrfb200_handle *h, HostPool *pool, const Box &b, const void *arr, void *land)
{
    const size_t es = (size_t)h->esize;
    const size_t plane = (size_t)(b.i1 - b.i0 + 1) * (b.k1 - b.k0 + 1) * es;
    const int per = cc.bounce3_bytes / plane > 0 ? (int)(cc.bounce3_bytes / plane) : 1;
    for (int j = b.j0; j <= b.j1; j += per) {
        Box c = b;
        c.j0 = j;
        c.j1 = j + per - 1 < b.j1 ? j + per - 1 : b.j1;
        const int x = cc.next_up;
        cc.next_up = (x + 1) % kBounceUp;
        char *buf = static_cast<char *>(cc.bounce[x]);
        CU(cudaEventSynchronize(cc.ev_bounce[x]));
        host_box(pool, h, c, const_cast<char *>(static_cast<const char *>(arr)), buf, true);
        if (land) {
            const long long nrows = (long long)(c.j1 - c.j0 + 1) * h->kdim;
            const int fpe = h->esize / (int)sizeof(float);
            CU(cudaMemcpyAsync(land, buf, (size_t)nrows * h->idim * es, cudaMemcpyHostToDevice, cc.up));
            CU(cudaEventRecord(cc.ev_bounce[x], cc.up));
            const size_t doff = (size_t)(c.j0 - h->dom.jms) * h->kdim * h->pitch3;
            CU(wrfb200_repitch_rows(h->d[b.f] + doff * fpe, static_cast<float *>(land), h->pitch3 * fpe,
                                    h->idim * fpe, nrows, cc.up));
            h->launches += 1;
            continue;
        }
        if (int rc = device_box(h, c, buf, true, cc.up)) return rc;
        CU(cudaEventRecord(cc.ev_bounce[x], cc.up));
    }
    return WRFB200_OK;
}

// A staged download whose host half has not run yet: box `b` waits in bounce buffer x for the scatter into `arr`.
struct PendingDown {
    bool live = false;
    Box b{};
    void *arr = nullptr;
};

// The host half of the download waiting in buffer x, if any: waits for its device copy, then the workers write the
// box's cells, and no others, into the caller's array.
int finish_down(CompatCache &cc, const wrfb200_handle *h, HostPool *pool, PendingDown *pend, int x)
{
    if (!pend[x].live) return WRFB200_OK;
    pend[x].live = false;
    CU(cudaEventSynchronize(cc.ev_bounce[x]));
    host_box(pool, h, pend[x].b, static_cast<char *>(pend[x].arr), static_cast<char *>(cc.bounce[x]), false);
    return WRFB200_OK;
}

// Staged download of box b into buffer x on the download lane; its host half runs when x is needed again or at the
// end of the call (finish_down).
int download_box(CompatCache &cc, wrfb200_handle *h, HostPool *pool, PendingDown *pend, int x, const Box &b, void *arr)
{
    if (int rc = finish_down(cc, h, pool, pend, x)) return rc;
    if (int rc = device_box(h, b, static_cast<char *>(cc.bounce[x]), false, cc.down)) return rc;
    CU(cudaEventRecord(cc.ev_bounce[x], cc.down));
    pend[x].live = true;
    pend[x].b = b;
    pend[x].arr = arr;
    return WRFB200_OK;
}

// an array that is neither page-locked nor device memory takes the staged route
bool pageable(const void *p)
{
    bool pinned = false;
    return classify(p, &pinned) == PTR_HOST && !pinned;
}

// wrfb200_default_last_transfer of a host-array call: how many of its 26 arrays are pageable
thread_local int g_last_route = -1;                       // -1: no host-array call on this thread yet

int transfer_route(const Args &a)
{
    int n = 0;
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) n += pageable(a.f[f]) ? 1 : 0;
    return n == 0 ? 0 : n < WRFB200_NUM_FIELDS ? 1 : 2;
}

int run_device_in_place(const Args &a, int prec)
{
    // Caller-owned device arrays in the dense Fortran layout, wrapped in a (cached) handle.
    if (int rc = check_domain(a.dom)) return rc;
    int dev = 0;
    CU(cudaGetDevice(&dev));
    DeviceCallCache *hit = nullptr, *oldest = &g_devcall[prec][0];
    for (DeviceCallCache &x : g_devcall[prec]) {
        if (x.valid && x.h.device == dev && same_domain(x.dom, a.dom) && std::memcmp(x.ptrs, a.f, sizeof(x.ptrs)) == 0) {
            hit = &x;
            break;
        }
        if (oldest->valid && (!x.valid || x.used < oldest->used)) oldest = &x;    // a free entry first
    }
    DeviceCallCache &c = hit ? *hit : *oldest;
    g_last_cache = hit ? WRFB200_CACHE_REUSED : c.valid ? WRFB200_CACHE_EVICTED : WRFB200_CACHE_CREATED;
    c.used = ++g_devcall_clock;
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
//
// Page-locked arrays are copied directly; pageable 2-D and 3-D arrays take the staged route (upload_box,
// download_box): every such copy goes through the cache's pinned bounce buffers.
//
// `part`: this is one device's share of a split call (run_host_split), or a shared-tiles call (run_host_shared),
// whose calling thread has already synchronised the caller's stream and page-locked the caller's whole arrays.
//
// `sp`: a tile of a shared patch (shared-tiles mode), whose mirrors other threads' tiles read and write
// concurrently.  A tile then writes to the device only what no other tile reads or writes in between:
//   - t, mu and ww at level kts (the fields the routine reads AND writes, each read at its own column only):
//     the tile's own columns i_start..i_end x j_start..j_end.  The full-field mu / ww copies and the ring rows
//     of t would overwrite a neighbouring tile's fresh outputs;
//   - the read-only inputs: the tile's rows plus the one-cell ring (all of i), 2-D ones over the same rows.  Two
//     tiles that both copy a ring row write the same bytes from the same host array, which the caller does not
//     change during the loop's steps (u, v only between them); that is why those copies may overlap;
//   - residency is kept per tile in `sp` (SharedPatch::take / put), whichever thread makes the call.
// The slab pipeline's cut of nj computed rows of a call on memory extents d: nslab slabs of at most `rows` rows each,
// ring rows included (the rows of a staging buffer and of a bounce buffer).
struct SlabPlan {
    int nslab;
    size_t rows;
};
SlabPlan slab_plan(const wrfb200_domain &d, int nj, size_t es)
{
    const size_t idim = d.ime - d.ims + 1, jdim = d.jme - d.jms + 1, kdim = d.kme - d.kms + 1;
    int nslab = 1;
    if (idim * kdim * jdim * es >= ((size_t)16 << 20) && nj >= 32) nslab = nj / 16 < kMaxSlabs ? nj / 16 : kMaxSlabs;
    return SlabPlan{nslab, (size_t)(nj / nslab + 3)};         // at most kMaxSlabs: one event pair per slab
}

int run_host_compat_body(const Args &a, int nsteps, DomainEntry &e, CompatCache &cc, bool part,
                         SharedPatch *sp = nullptr)
{
    wrfb200_handle *h = e.h;
    const wrfb200_domain &d = a.dom;
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   a.its, a.ite, a.jts, a.jte, a.kts, a.kte, &is, &ie, &js, &je, &ks, &ke);
    if (is > ie || js > je || ks > ke) return WRFB200_OK;
    if (is - 1 < d.ims || ie + 1 > d.ime || js - 1 < d.jms || je + 1 > d.jme)
        return fail(WRFB200_ERR_INVALID_ARG,
                    "computed range i=%d..%d j=%d..%d needs a one-cell ring inside memory i=%d..%d j=%d..%d",
                    is, ie, js, je, d.ims, d.ime, d.jms, d.jme);
    if (!part) CU(cudaStreamSynchronize(g_default_stream));   // the caller's earlier work on its stream is done

    static const int in3_all[] = {WRFB200_WW_1, WRFB200_U, WRFB200_U_1, WRFB200_V, WRFB200_V_1,
                                  WRFB200_T, WRFB200_T_1, WRFB200_FT};
    static const int in3_uv[] = {WRFB200_U, WRFB200_V};
    static const int in3_ring[] = {WRFB200_WW_1, WRFB200_U, WRFB200_U_1, WRFB200_V, WRFB200_V_1,
                                   WRFB200_T_1, WRFB200_FT};      // shared tiles: the read-only ones (t per slab)
    static const int in2[] = {WRFB200_MU, WRFB200_MUT, WRFB200_MUU, WRFB200_MUV, WRFB200_MU_TEND,
                              WRFB200_MSFUY, WRFB200_MSFVX_INV, WRFB200_MSFTX, WRFB200_MSFTY};
    static const int in1[] = {WRFB200_DNW, WRFB200_FNM, WRFB200_FNP, WRFB200_RDNW};
    static const int out3[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE};
    static const int out2[] = {WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF};

    // resident step: same arrays, same index sets, same scalars as the call that primed the mirrors
    const bool resident = sp ? sp->take(a) : cc.loop_active && e.primed && same_call(e.primed_args, a);
    e.primed = false;                                     // until this call has completed
    const int *in3 = resident ? in3_uv : sp ? in3_ring : in3_all;
    const int n_in3 = resident ? 2 : sp ? 7 : 8;

    if (pin_enabled() && !part)
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) pin_host(a.f[f], field_bytes(d, f, h->esize));

    const int nj = je - js + 1;
    const size_t es = (size_t)h->esize;
    const SlabPlan plan = slab_plan(d, nj, es);
    const int nslab = plan.nslab;
    const size_t slab_bytes = plan.rows * h->kdim * h->idim * es;

    // The route of each array: page-locked ones (by the caller or by opt-in pinning) are copied directly, pageable
    // 2-D and 3-D ones through the cache's bounce buffers (the 1-D ones, a few hundred bytes, directly as well).
    bool bounce[WRFB200_NUM_FIELDS];
    bool any_bounce = false;
    for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) {
        bounce[f] = !is1d(f) && pageable(a.f[f]);
        any_bounce = any_bounce || bounce[f];
    }
    HostPool *pool = nullptr;
    PendingDown pend[kBounce];
    if (any_bounce) {
        if (int rc = ensure_bounce(cc, slab_bytes, plan.rows * h->idim * es)) return rc;
        pool = host_pool();
    }

    // small operands first: 2-D and 1-D inputs, and ww at level 1 (the only level of ww the routine
    // reads, module_small_step_em.f90:159-161)
    h->stream = cc.up;
    if (!resident && !sp) {
        for (int f : in2) {
            if (bounce[f]) {
                if (int rc = upload_box(cc, h, pool, Box{f, d.ims, d.ime, 0, 0, d.jms, d.jme}, a.f[f], nullptr)) return rc;
            } else if (int rc = copy_field(h, f, a.f[f], nullptr)) return rc;
        }
        for (int f : in1) if (int rc = copy_field(h, f, a.f[f], nullptr)) return rc;
        if (bounce[WRFB200_WW]) {
            const Box b{WRFB200_WW, d.ims, d.ime, a.kts, a.kts, d.jms, d.jme};
            if (int rc = upload_box(cc, h, pool, b, a.f[WRFB200_WW], nullptr)) return rc;
        } else if (int rc = copy_range(h, WRFB200_WW, a.f[WRFB200_WW], nullptr, d.ims, d.ime, a.kts, a.kts, d.jms, d.jme)) return rc;
    } else if (!resident) {
        for (int f : in2) {
            if (f == WRFB200_MU) continue;
            if (bounce[f]) {
                if (int rc = upload_box(cc, h, pool, Box{f, d.ims, d.ime, 0, 0, js - 1, je + 1}, a.f[f], nullptr)) return rc;
            } else if (int rc = copy_range(h, f, a.f[f], nullptr, d.ims, d.ime, 0, 0, js - 1, je + 1)) return rc;
        }
        for (int f : in1) if (int rc = copy_field(h, f, a.f[f], nullptr)) return rc;
        if (bounce[WRFB200_MU]) {
            if (int rc = upload_box(cc, h, pool, Box{WRFB200_MU, is, ie, 0, 0, js, je}, a.f[WRFB200_MU], nullptr)) return rc;
        } else if (int rc = copy_range(h, WRFB200_MU, a.f[WRFB200_MU], nullptr, is, ie, 0, 0, js, je)) return rc;
        if (bounce[WRFB200_WW]) {
            const Box b{WRFB200_WW, is, ie, a.kts, a.kts, js, je};
            if (int rc = upload_box(cc, h, pool, b, a.f[WRFB200_WW], nullptr)) return rc;
        } else if (int rc = copy_range(h, WRFB200_WW, a.f[WRFB200_WW], nullptr, is, ie, a.kts, a.kts, js, je)) return rc;
    }

    int next_row = js - 1;                                // first row of the 3-D inputs not yet uploaded
    // A row-pitched (2-D) host->device copy runs ~18 % below a contiguous one on this link (40 vs 49 GB/s
    // measured, tools/pcie_probe.py).  When the mirror is padded, land each slab densely in a staging buffer
    // with ONE contiguous copy and re-pitch it on the device (HBM speed, negligible).
    const bool staged = (h->pitch3 != h->idim) && nslab > 1;
    if (staged && e.stage_bytes < slab_bytes) {
        for (void *&b : e.stage) { if (b) cudaFree(b); b = nullptr; }
        e.stage_bytes = 0;
        for (void *&b : e.stage) CU(cudaMalloc(&b, slab_bytes));
        e.stage_bytes = slab_bytes;
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
                if (bounce[f]) {
                    void *land = staged ? e.stage[flip] : nullptr;
                    if (staged) flip ^= 1;
                    const Box b{f, d.ims, d.ime, d.kms, d.kme, next_row, hi};
                    if (int rc = upload_box(cc, h, pool, b, a.f[f], land)) return rc;
                    continue;
                }
                if (!staged) {
                    if (int rc = copy_range(h, f, a.f[f], nullptr, d.ims, d.ime, d.kms, d.kme, next_row, hi)) return rc;
                    continue;
                }
                float *st = static_cast<float *>(e.stage[flip]);
                flip ^= 1;
                CU(cudaMemcpyAsync(st, static_cast<const char *>(a.f[f]) + hoff * es, (size_t)nrows * h->idim * es,
                                   cudaMemcpyHostToDevice, cc.up));
                CU(wrfb200_repitch_rows(h->d[f] + doff * fpe, st, h->pitch3 * fpe, h->idim * fpe, nrows, cc.up));
                h->launches += 1;
            }
            next_row = hi + 1;
        }
        // shared tiles: t over the slab's own columns (all levels: no tile reads or writes t outside its columns)
        if (sp && !resident && bounce[WRFB200_T]) {
            const Box b{WRFB200_T, is, ie, d.kms, d.kme, ja, jb};
            if (int rc = upload_box(cc, h, pool, b, a.f[WRFB200_T], nullptr)) return rc;
        } else if (sp && !resident)
            if (int rc = copy_range(h, WRFB200_T, a.f[WRFB200_T], nullptr, is, ie, d.kms, d.kme, ja, jb)) return rc;
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
        for (int x = 0; x < 3; ++x) {
            const int f = out3[x];
            if (bounce[f]) {
                if (int rc = download_box(cc, h, pool, pend, kBounceUp + x, Box{f, is, ie, ks, ke, ja, jb}, a.f[f])) return rc;
            } else if (int rc = copy_range(h, f, nullptr, a.f[f], is, ie, ks, ke, ja, jb)) return rc;
        }
        for (int x = 0; x < 4; ++x) {
            const int f = out2[x];
            if (bounce[f]) {
                if (int rc = download_box(cc, h, pool, pend, kBounce3 + x, Box{f, is, ie, 0, 0, ja, jb}, a.f[f])) return rc;
            } else if (int rc = copy_range(h, f, nullptr, a.f[f], is, ie, 0, 0, ja, jb)) return rc;
        }
    }
    for (int x = 0; x < kBounce; ++x)
        if (int rc = finish_down(cc, h, pool, pend, x)) return rc;
    CU(cudaStreamSynchronize(cc.up));
    CU(cudaStreamSynchronize(cc.comp));
    CU(cudaStreamSynchronize(cc.down));
    if (sp) {
        if (g_shared_loop.load()) sp->put(a);
    } else if (cc.loop_active) {
        e.primed = true;
        e.primed_args = a;
    }
    return WRFB200_OK;
}

// The cache's lanes and their events on `device`.  They move when a domain of the cache lives on another device
// than the last one (a single-device caller that changed its current device).
int open_lanes(CompatCache &cc, int device)
{
    if (cc.lane_device == device) return WRFB200_OK;
    cc.release_lanes();
    DeviceGuard g(device);
    if (!g.ok) return fail(WRFB200_ERR_CUDA, "cannot select CUDA device %d", device);
    cc.lane_device = device;
    const int rc = [&]() -> int {
        for (cudaStream_t *st : {&cc.up, &cc.comp, &cc.down})
            CU(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
        for (int i = 0; i < kMaxSlabs; ++i) {
            CU(cudaEventCreateWithFlags(&cc.ev_up[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&cc.ev_comp[i], cudaEventDisableTiming));
        }
        return WRFB200_OK;
    }();
    if (rc != WRFB200_OK) {
        const std::string msg = wrfb200_last_error();
        cc.release_lanes();
        wrfb200_fail(rc, "%s", msg.c_str());
    }
    return rc;
}

// A new domain at the front of the cache: its handle (mirrors allocated or, with allocate=0, to be bound).
int open_domain(CompatCache &cc, const wrfb200_domain &dom, int device, int allocate, int prec)
{
    std::unique_ptr<DomainEntry> e(new (std::nothrow) DomainEntry());
    if (!e) return fail(WRFB200_ERR_NOMEM, "out of host memory");
    if (int rc = create(&e->h, &dom, device, allocate, prec ? 8 : 4)) return rc;
    cc.doms.insert(cc.doms.begin(), std::move(e));
    return WRFB200_OK;
}

// The domain of the call's memory extents at the front of cache cc, found or created; *state tells which
// (wrfb200_cache).  device < 0 (the single-device call): an entry of the same extents is re-used wherever it
// lives, a new one goes on the current device; device >= 0 (a part of a split call): the entry must live there.
// Before creating, the cache gives up its least recently used domains: beyond kMaxDomains, and on the target
// device while its free memory cannot hold the new mirrors and the staging buffers the call will allocate.  If the allocation still runs out of memory, every
// other domain of the cache (and of the thread's other precision, unless this is a part of a split call running
// beside the thread's other parts) is freed and it is tried once more.
int find_domain(CompatCache &cc, const Args &a, int device, int prec, bool part, int *state)
{
    const wrfb200_domain &dom = a.dom;
    for (size_t x = 0; x < cc.doms.size(); ++x) {
        const wrfb200_handle *h = cc.doms[x]->h;
        if (same_shape(h->dom, dom) && (device < 0 || h->device == device)) {
            std::rotate(cc.doms.begin(), cc.doms.begin() + x, cc.doms.begin() + x + 1);
            *state = WRFB200_CACHE_REUSED;
            return WRFB200_OK;
        }
    }
    if (device < 0) CU(cudaGetDevice(&device));
    *state = WRFB200_CACHE_CREATED;
    if (cc.doms.size() >= kMaxDomains) {
        cc.doms.pop_back();
        *state = WRFB200_CACHE_EVICTED;
    }
    {
        DeviceGuard g(device);
        if (!g.ok) return fail(WRFB200_ERR_CUDA, "cannot select CUDA device %d", device);
        const int es = prec ? 8 : 4;
        size_t need = mirror_bytes(dom, es);
        int is, ie, js, je, ks, ke;
        wrfb200_bounds(dom.periodic_x, dom.specified, dom.nested, dom.ids, dom.ide, dom.jds, dom.jde,
                       a.its, a.ite, a.jts, a.jte, a.kts, a.kte, &is, &ie, &js, &je, &ks, &ke);
        const long idim = dom.ime - dom.ims + 1, kdim = dom.kme - dom.kms + 1;
        const SlabPlan plan = slab_plan(dom, js <= je ? je - js + 1 : 0, es);
        if (round_up(idim, 128 / es) != idim && plan.nslab > 1)      // run_host_compat_body's staging buffers
            need += 2 * plan.rows * kdim * idim * es;
        for (;;) {
            size_t free_bytes = 0, total = 0;
            if (cudaMemGetInfo(&free_bytes, &total) != cudaSuccess) { (void)cudaGetLastError(); break; }
            if (free_bytes >= need) break;
            size_t x = cc.doms.size();
            while (x > 0 && cc.doms[x - 1]->h->device != device) --x;
            if (x == 0) break;
            cc.doms.erase(cc.doms.begin() + (x - 1));
            *state = WRFB200_CACHE_EVICTED;
        }
    }
    int rc = open_domain(cc, dom, device, 1, prec);
    CompatCache *other = part ? nullptr : &g_cache[1 - prec];
    if (rc == WRFB200_ERR_NOMEM && (!cc.doms.empty() || (other && !other->doms.empty()))) {
        (void)cudaGetLastError();
        cc.doms.clear();
        if (other) other->doms.clear();
        *state = WRFB200_CACHE_EVICTED;
        rc = open_domain(cc, dom, device, 1, prec);
    }
    return rc;
}

// run_host_compat_body on domain e of cache cc, with the calling thread's kernel choice and the call's scalars
int run_on_cache(const Args &a, int nsteps, CompatCache &cc, DomainEntry &e, int kernel, bool part, SharedPatch *sp)
{
    wrfb200_handle *h = e.h;
    GUARD(h);
    h->dom = a.dom;                       // same extents; domain dims / flags may differ between calls
    h->kernel = kernel;
    set_scalars(h, a.rdx, a.rdy, a.dts, a.epssm);
    const int rc = run_host_compat_body(a, nsteps, e, cc, part, sp);
    if (rc != WRFB200_OK) {
        // an early return must not leave copies on the caller's arrays in flight, nor the cached handle
        // pointing at one of the internal lanes
        const std::string msg = wrfb200_last_error();
        for (cudaStream_t st : {cc.up, cc.comp, cc.down}) if (st) cudaStreamSynchronize(st);
        (void)cudaGetLastError();
        e.primed = false;
        wrfb200_fail(rc, "%s", msg.c_str());
    }
    h->stream = part ? nullptr : g_default_stream;
    return rc;
}

// One host-pointer call, or one device's share of a split call, on its domain of cache `cc` (find_domain).
// `kernel` is the calling thread's choice, passed in because a part may run in a worker thread; *state receives
// what the call did with the cache.
int run_host_part(const Args &a, int nsteps, int prec, CompatCache &cc, int device, int kernel, bool part, int *state)
{
    if (int rc = check_domain(a.dom)) return rc;
    if (int rc = find_domain(cc, a, device, prec, part, state)) return rc;
    DomainEntry &e = *cc.doms.front();
    if (int rc = open_lanes(cc, e.h->device)) return rc;
    return run_on_cache(a, nsteps, cc, e, kernel, part, nullptr);
}

// One host-pointer call in shared-tiles mode: a tile of the shared patch of these arrays on the patch device,
// created by whichever tile comes first, run from this thread's own lanes and handle.
int run_host_shared(const Args &a, int nsteps, int prec)
{
    if (int rc = check_domain(a.dom)) return rc;
    int dev = 0;
    if (int rc = shared_device(&dev)) return rc;
    if (!g_default_devices.empty() && (g_default_devices.size() > 1 || g_default_devices[0] != dev))
        return fail(WRFB200_ERR_UNSUPPORTED,
                    "shared-tiles mode runs every host-array call on the patch device %d; this thread's device list "
                    "(wrfb200_set_default_devices: %zu device(s), first %d) names another or several",
                    dev, g_default_devices.size(), g_default_devices[0]);
    CU(cudaStreamSynchronize(g_default_stream));          // the caller's earlier work on its stream is done
    const size_t es = prec ? 8 : 4;
    if (pin_enabled())
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) pin_host(a.f[f], field_bytes(a.dom, f, es));

    SharedPatch *sp = nullptr;
    g_last_cache = WRFB200_CACHE_REUSED;
    {
        std::lock_guard<std::mutex> lock(g_shared_mutex);
        for (auto &q : g_shared)
            if (q->prec == prec && q->h->device == dev && same_shape(q->h->dom, a.dom) &&
                std::memcmp(q->ptrs, a.f, sizeof(a.f)) == 0) { sp = q.get(); break; }
        if (!sp) {
            std::unique_ptr<SharedPatch> q(new (std::nothrow) SharedPatch());
            if (!q) return fail(WRFB200_ERR_NOMEM, "out of host memory");
            if (int rc = create(&q->h, &a.dom, dev, 1, (int)es)) return rc;
            q->prec = prec;
            q->id = g_shared_next_id++;
            std::memcpy(q->ptrs, a.f, sizeof(a.f));
            sp = q.get();
            g_shared.push_back(std::move(q));
            g_last_cache = WRFB200_CACHE_CREATED;
        }
    }

    // the thread's one handle for shared calls, bound to the patch's mirrors
    TileThread &tt = g_tiles;
    tt.enlist();
    CompatCache &cc = tt.c[prec];
    if (!cc.doms.empty() && (!same_shape(cc.doms[0]->h->dom, a.dom) || cc.doms[0]->h->device != dev)) {
        cc.release();
        tt.bound[prec] = 0;
    }
    if (cc.doms.empty()) {
        if (int rc = open_domain(cc, a.dom, dev, 0, prec)) return rc;
        g_last_cache = WRFB200_CACHE_CREATED;
    }
    if (int rc = open_lanes(cc, dev)) return rc;
    DomainEntry &e = *cc.doms.front();
    if (tt.bound[prec] != sp->id) {
        tt.bound[prec] = 0;
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f)
            if (int rc = bind_device(e.h, f, sp->h->d[f], is3d(f) ? sp->h->pitch3 : sp->h->pitch2)) return rc;
        tt.bound[prec] = sp->id;
    }
    return run_on_cache(a, nsteps, cc, e, g_default_kernel, true, sp);
}

// ---- one host-pointer call split over several devices (wrfb200_set_default_devices) --------------------
constexpr int kMaxParts = 64;

// parts 1.. of a split call (part 0 is g_cache), indexed like g_cache
thread_local std::vector<std::unique_ptr<CompatCache>> g_parts[2];

// The split rule, shared by wrfb200_host_split_plan and the call: the computed rows j_start..j_end are cut into n
// contiguous parts with the slab loop's formula; a part's memory is its rows plus the one-row ring on each side.
int host_split(const wrfb200_domain &d, int its, int ite, int jts, int jte, int kts, int kte, int n, int *rows4)
{
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   its, ite, jts, jte, kts, kte, &is, &ie, &js, &je, &ks, &ke);
    const bool empty = is > ie || js > je || ks > ke;
    if (!empty && (is - 1 < d.ims || ie + 1 > d.ime || js - 1 < d.jms || je + 1 > d.jme))
        return fail(WRFB200_ERR_INVALID_ARG,
                    "computed range i=%d..%d j=%d..%d needs a one-cell ring inside memory i=%d..%d j=%d..%d",
                    is, ie, js, je, d.ims, d.ime, d.jms, d.jme);
    const int nj = empty ? 0 : je - js + 1;
    for (int p = 0; p < n; ++p) {
        const int ja = js + (int)((long long)nj * p / n);
        const int jb = js + (int)((long long)nj * (p + 1) / n) - 1;
        int *r = rows4 + 4 * p;
        r[0] = ja; r[1] = jb;
        r[2] = ja <= jb ? ja - 1 : ja; r[3] = ja <= jb ? jb + 1 : jb;
    }
    return WRFB200_OK;
}

// The host-pointer call as one sub-call per used part.  A part is the single-device call on a sub-domain: field
// pointers offset to the part's first memory row (j is the slowest index, so that slice of a dense array is
// dense), jms..jme narrowed to the part's memory and jts..jte to its rows; ids..jde, the flags, its..ite and
// kts..kte unchanged.  Part 0 runs in the calling thread, every other part in a thread of its own, so that each
// device's copies and launches are issued concurrently (a pageable cudaMemcpyAsync blocks its thread); all are
// joined before the call returns.
int run_host_split(const Args &a, int nsteps, int prec)
{
    if (int rc = check_domain(a.dom)) return rc;
    const int n = (int)g_default_devices.size();
    int rows4[4 * kMaxParts];
    if (int rc = host_split(a.dom, a.its, a.ite, a.jts, a.jte, a.kts, a.kte, n, rows4)) return rc;
    CU(cudaStreamSynchronize(g_default_stream));          // the caller's earlier work on its stream is done
    const size_t es = prec ? 8 : 4;
    // the caller's WHOLE arrays, once: part slices overlap by the ring rows, and a second registration of an
    // overlapping range would fail
    if (pin_enabled())
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f) pin_host(a.f[f], field_bytes(a.dom, f, es));

    // the cache of part p, whether or not a call uses it: p's device list entry, so that each cache keeps serving one
    // device for every domain, also when a domain with fewer rows than devices leaves parts unused
    std::vector<std::unique_ptr<CompatCache>> &pool = g_parts[prec];
    while ((int)pool.size() + 1 < n) {
        pool.emplace_back(new (std::nothrow) CompatCache());
        if (!pool.back()) { pool.pop_back(); return fail(WRFB200_ERR_NOMEM, "out of host memory"); }
        pool.back()->loop_active = g_cache[prec].loop_active;
    }
    struct Part {
        Args a;
        CompatCache *cache;
        int device, rc = WRFB200_OK, state = -1;
        std::string err;
    };
    std::vector<Part> parts;
    for (int p = 0; p < n; ++p) {
        const int *r = rows4 + 4 * p;
        if (r[0] > r[1]) continue;                        // no rows: not used
        Part q;
        q.a = a;
        q.cache = p == 0 ? &g_cache[prec] : pool[p - 1].get();      // taken here: g_cache is the calling thread's
        q.device = g_default_devices[p];
        const size_t row3 = field_bytes(a.dom, WRFB200_U, es) / (a.dom.jme - a.dom.jms + 1);
        const size_t row2 = field_bytes(a.dom, WRFB200_MU, es) / (a.dom.jme - a.dom.jms + 1);
        for (int f = 0; f < WRFB200_NUM_FIELDS; ++f)
            if (!is1d(f)) q.a.f[f] = static_cast<char *>(a.f[f]) + (size_t)(r[2] - a.dom.jms) * (is3d(f) ? row3 : row2);
        q.a.dom.jms = r[2]; q.a.dom.jme = r[3];
        q.a.jts = r[0]; q.a.jte = r[1];
        parts.push_back(q);
    }
    if (parts.empty()) return WRFB200_OK;

    const int kernel = g_default_kernel;
    auto run = [&](size_t q) {
        Part &p = parts[q];
        p.rc = run_host_part(p.a, nsteps, prec, *p.cache, p.device, kernel, true, &p.state);
        if (p.rc != WRFB200_OK) p.err = wrfb200_last_error();
    };
    std::vector<std::thread> workers;
    workers.reserve(parts.size());
    for (size_t q = 1; q < parts.size(); ++q) {
        try {
            workers.emplace_back(run, q);
        } catch (const std::exception &) {
            parts[q].rc = WRFB200_ERR_NOMEM;
            parts[q].err = "cannot start a host thread";
        }
    }
    run(0);
    for (std::thread &t : workers) t.join();

    for (const Part &p : parts) g_last_cache = std::max(g_last_cache, p.state);     // the most any part did
    for (size_t q = 0; q < parts.size(); ++q) {
        if (parts[q].rc == WRFB200_OK) continue;
        for (const Part &r : parts) r.cache->forget();
        const Part &p = parts[q];
        return fail(p.rc, "device %d, rows j=%d..%d: %s", p.device, p.a.jts, p.a.jte, p.err.c_str());
    }
    return WRFB200_OK;
}

int run_host_compat(const Args &a, int nsteps, int prec)
{
    if (shared_enabled()) return run_host_shared(a, nsteps, prec);
    if (!g_default_devices.empty()) {
        int cur = 0;
        CU(cudaGetDevice(&cur));
        if (g_default_devices.size() > 1 || g_default_devices[0] != cur) return run_host_split(a, nsteps, prec);
    }
    return run_host_part(a, nsteps, prec, g_cache[prec], -1, g_default_kernel, false, &g_last_cache);
}

void release_parts()
{
    for (CompatCache &c : g_cache) c.release();
    for (auto &pool : g_parts)
        for (auto &c : pool) c->release();
}

// prec: 0 = binary32 entry points, 1 = real*8 entry points
int dispatch(Args &a, int nsteps, bool allow_device, int prec)
{
    g_last_prec = prec;
    g_last_cache = -1;
    // device-pointer fast path: the very same arrays as a recent call need no re-classification
    if (allow_device && nsteps == 1)
        for (const DeviceCallCache &dc : g_devcall[prec])
            if (dc.valid && std::memcmp(dc.ptrs, a.f, sizeof(a.f)) == 0) return run_device_in_place(a, prec);
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
    drop_devcalls(prec);
    const int rc = run_host_compat(a, nsteps, prec);
    g_last_route = transfer_route(a);                     // after the call: opt-in pinning may have locked the arrays
    return rc;
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

extern "C" int wrfb200_set_default_devices(const int *devices, int n)
{
    if (n < 0 || n > kMaxParts) return fail(WRFB200_ERR_INVALID_ARG, "n=%d: 0..%d devices", n, kMaxParts);
    if (n > 0 && !devices) return fail(WRFB200_ERR_INVALID_ARG, "null device list with n=%d", n);
    if (n > 0) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            return fail(WRFB200_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
        }
        for (int p = 0; p < n; ++p)
            if (devices[p] < 0 || devices[p] >= ndev)
                return fail(WRFB200_ERR_INVALID_ARG, "device %d out of range (%d devices)", devices[p], ndev);
    }
    std::vector<int> list(devices, devices + n);
    if (list != g_default_devices) {
        release_parts();
        g_default_devices.swap(list);
    }
    return WRFB200_OK;
}

extern "C" int wrfb200_host_split_plan(const wrfb200_domain *dom, int its, int ite, int jts, int jte, int kts, int kte,
                                       int n, int *rows4)
{
    if (!dom || !rows4) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (n < 1 || n > kMaxParts) return fail(WRFB200_ERR_INVALID_ARG, "n=%d: 1..%d parts", n, kMaxParts);
    if (int rc = check_domain(*dom)) return rc;
    return host_split(*dom, its, ite, jts, jte, kts, kte, n, rows4);
}

extern "C" int wrfb200_release_cache(void)
{
    release_parts();
    release_shared();
    for (int prec = 0; prec < 2; ++prec) drop_devcalls(prec);
    unpin_all();
    stop_pool();
    return WRFB200_OK;
}

namespace {

// the shared patches' residency follows the loop whichever thread begins or ends it
void shared_loop(bool active)
{
    if (!shared_enabled()) return;
    int dev = 0;
    if (active && shared_device(&dev) != WRFB200_OK) (void)cudaGetLastError();   // records the patch device
    g_shared_loop.store(active);
    std::lock_guard<std::mutex> lock(g_shared_mutex);
    for (auto &sp : g_shared) sp->forget();
}

}  // namespace

extern "C" int wrfb200_acoustic_loop_begin(void)
{
    for (CompatCache &c : g_cache) { c.loop_active = true; c.forget(); }
    for (auto &pool : g_parts)
        for (auto &c : pool) { c->loop_active = true; c->forget(); }
    shared_loop(true);
    return WRFB200_OK;
}

extern "C" int wrfb200_acoustic_loop_end(void)
{
    for (CompatCache &c : g_cache) { c.loop_active = false; c.forget(); }
    for (auto &pool : g_parts)
        for (auto &c : pool) { c->loop_active = false; c->forget(); }
    shared_loop(false);
    return WRFB200_OK;
}

extern "C" int wrfb200_set_shared_tiles(int enable)
{
    if (!enable) {
        g_shared_mode.store(0);
        g_shared_device.store(-1);
        release_shared();
        return WRFB200_OK;
    }
    int ndev = 0, dev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return fail(WRFB200_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    if (g_shared_mode.load() == 1 && g_shared_device.load() == dev) return WRFB200_OK;
    release_shared();                                      // patches of another device, if any
    g_shared_device.store(dev);
    g_shared_mode.store(1);
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
    int most = 0;
    if (!amt_pipe_levels_fit(p, &most)) return too_many_levels("pipe kernel", p.nk, most);
    if (!amt_pipe_plan(p, resident_blocks > 0 ? resident_blocks : 2 * 148, plan10))
        return fail(WRFB200_ERR_INVALID_ARG, "empty index sets");
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
    const DeviceCallCache *dc = last_devcall(g_last_prec);
    const CompatCache &cc = shared_enabled() ? g_tiles.c[g_last_prec] : g_cache[g_last_prec];
    *kernel = dc ? dc->h.last_kernel : (cc.doms.empty() ? 0 : cc.doms.front()->h->last_kernel);
    return WRFB200_OK;
}

extern "C" int wrfb200_default_last_transfer(int *route)
{
    if (!route) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (g_last_route < 0) return fail(WRFB200_ERR_STATE, "no host-array call on this thread yet");
    *route = g_last_route;
    return WRFB200_OK;
}

extern "C" int wrfb200_default_last_cache(int *state)
{
    if (!state) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (g_last_cache < 0) return fail(WRFB200_ERR_STATE, "no advance_mu_t call on this thread has reached its cache yet");
    *state = g_last_cache;
    return WRFB200_OK;
}

extern "C" int wrfb200_bounce_allocations(long *count)
{
    if (!count) return fail(WRFB200_ERR_INVALID_ARG, "null argument");
    *count = g_bounce_allocs.load();
    return WRFB200_OK;
}
