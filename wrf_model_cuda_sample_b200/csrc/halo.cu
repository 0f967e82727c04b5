// halo.cu -- device-side halo packing for the 2-D (i,j) patch decomposition, plus the deterministic
// stand-in for advance_uv used by the multi-step tests.
//
// The reference has no device-to-device exchange at all: every call re-uploads j-slabs that overlap by
// three rows from pinned host memory (/root/reference/advance_mu_t_no_async.cu:87-162, :276-298).
// advance_mu_t only reads a ONE-cell ring (u,u_1,muu,msfuy at i+1; v,v_1,muv,msfvx_inv at j+1; t_1 at
// i+-1, j+-1 -- module_small_step_em.f90:143-146, :241-245), so a one-wide halo is packed into a dense
// buffer here, moved between ranks by the host layer (NCCL send/recv), and unpacked on the other side.
#include "capi_internal.h"

namespace {

// Copy the box [i0,i0+ni) x [0,nk) x [j0,j0+nj) (memory indices) between a field and a dense
// [j][k][i] buffer.
template <bool PACK>
__global__ void box_copy_kernel(float *field, float *buf, long long pitch, long long jstride,
                                int i0, int j0, int ni, int nk, int nj)
{
    const long long n = (long long)ni * nk * nj;
    for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < n;
         x += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(x % ni);
        const long long r = x / ni;
        const int k = (int)(r % nk);
        const int j = (int)(r / nk);
        const long long o = (long long)(j0 + j) * jstride + (long long)k * pitch + (i0 + i);
        if (PACK) buf[x] = field[o];
        else field[o] = buf[x];
    }
}

// u(i,k,j) += c*(mudf(i,j)-mudf(i-1,j))   or   v(i,k,j) += c*(mudf(i,j)-mudf(i,j-1)); one block per (k,j) row
__global__ void standin_uv_kernel(float *f, const float *mudf, long long pitch, long long jstride,
                                  long long pitch2, long long dshift, float c,
                                  int i0, int j0, int ni, int nk, int nj)
{
    for (long long r = blockIdx.x; r < (long long)nk * nj; r += gridDim.x) {
        const int k = (int)(r % nk);
        const int j = (int)(r / nk);
        float *row = f + (long long)(j0 + j) * jstride + (long long)k * pitch + i0;
        const float *m = mudf + (long long)(j0 + j) * pitch2 + i0;
        for (int i = threadIdx.x; i < ni; i += blockDim.x)
            row[i] = __fadd_rn(row[i], __fmul_rn(c, __fsub_rn(m[i], m[i - dshift])));
    }
}

// rows of `ni` floats, dense in `src`, to rows `pitch` floats apart in `dst`
__global__ void repitch_rows_kernel(float *dst, const float *src, long long pitch, int ni, long long nrows)
{
    const long long n = nrows * ni;
    for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < n;
         x += (long long)gridDim.x * blockDim.x) {
        const long long r = x / ni;
        const int i = (int)(x - r * ni);
        dst[r * pitch + i] = src[x];
    }
}

int halo_box(const wrfb200_handle *h, int side, int width, bool inside,
             int ips, int ipe, int jps, int jpe, int *i0, int *i1, int *j0, int *j1)
{
    if (width < 1) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "halo width %d", width);
    switch (side) {
    case WRFB200_WEST:  *j0 = jps; *j1 = jpe; *i0 = inside ? ips : ips - width; *i1 = *i0 + width - 1; break;
    case WRFB200_EAST:  *j0 = jps; *j1 = jpe; *i0 = inside ? ipe - width + 1 : ipe + 1; *i1 = *i0 + width - 1; break;
    case WRFB200_SOUTH: *i0 = ips; *i1 = ipe; *j0 = inside ? jps : jps - width; *j1 = *j0 + width - 1; break;
    case WRFB200_NORTH: *i0 = ips; *i1 = ipe; *j0 = inside ? jpe - width + 1 : jpe + 1; *j1 = *j0 + width - 1; break;
    default: return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "bad side %d", side);
    }
    const wrfb200_domain &d = h->dom;
    if (*i0 < d.ims || *i1 > d.ime || *j0 < d.jms || *j1 > d.jme || *i0 > *i1 || *j0 > *j1)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "halo box i=%d..%d j=%d..%d outside memory", *i0, *i1, *j0, *j1);
    return WRFB200_OK;
}

int halo_copy(wrfb200_handle *h, int field, int side, int width, int ips, int ipe, int jps, int jpe,
              float *buf, bool pack)
{
    if (!h || !buf) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (int rc = wrfb200_require_r4(h, pack ? "wrfb200_pack_halo" : "wrfb200_unpack_halo")) return rc;
    const bool f3 = field >= WRFB200_WW && field <= WRFB200_FT;
    const bool f2 = field >= WRFB200_MU && field <= WRFB200_MSFTY;
    if (!f3 && !f2) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "field %d has no horizontal halo", field);
    if (!h->d[field]) return wrfb200_fail(WRFB200_ERR_STATE, "field %d has no device buffer", field);
    int i0, i1, j0, j1;
    if (int rc = halo_box(h, side, width, pack, ips, ipe, jps, jpe, &i0, &i1, &j0, &j1)) return rc;
    const int ni = i1 - i0 + 1, nj = j1 - j0 + 1, nk = f3 ? h->kdim : 1;
    const long long pitch = f3 ? h->pitch3 : h->pitch2;
    const long long jstride = f3 ? pitch * h->kdim : pitch;
    const long long n = (long long)ni * nk * nj;
    int prev = -1;
    cudaGetDevice(&prev);
    if (prev != h->device) cudaSetDevice(h->device);
    const int threads = 256;
    const unsigned blocks = (unsigned)((n + threads - 1) / threads < 1184 ? (n + threads - 1) / threads : 1184);
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    if (pack)
        box_copy_kernel<true><<<blocks, threads, 0, h->stream>>>(h->d[field], buf, pitch, jstride,
                                                                 i0 - h->dom.ims, j0 - h->dom.jms, ni, nk, nj);
    else
        box_copy_kernel<false><<<blocks, threads, 0, h->stream>>>(h->d[field], buf, pitch, jstride,
                                                                  i0 - h->dom.ims, j0 - h->dom.jms, ni, nk, nj);
    cudaError_t e = cudaGetLastError();
    if (prev != h->device && prev >= 0) cudaSetDevice(prev);
    if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "halo kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    return WRFB200_OK;
}

}  // namespace

// Dense rows (as they lie in a host array that was copied to the device in one contiguous transfer) into the
// pitched mirror.  Stream-ordered on `stream`.
cudaError_t wrfb200_repitch_rows(float *dst, const float *src, long long pitch, int ni, long long nrows,
                                 cudaStream_t stream)
{
    if (nrows <= 0 || ni <= 0) return cudaSuccess;
    const long long n = nrows * ni;
    const long long want = (n + 255) / 256;
    const unsigned blocks = (unsigned)(want < 148 * 16 ? want : 148 * 16);
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    repitch_rows_kernel<<<blocks, 256, 0, stream>>>(dst, src, pitch, ni, nrows);
    return cudaGetLastError();
}

// load the kernels of this translation unit (see amt_pipe_preload)
cudaError_t wrfb200_halo_preload()
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, (const void *)standin_uv_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, (const void *)box_copy_kernel<true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, (const void *)box_copy_kernel<false>);
    return e;
}

extern "C" int wrfb200_pack_halo(wrfb200_handle *h, int field, int side, int width,
                                 int ips, int ipe, int jps, int jpe, float *device_buf)
{
    return halo_copy(h, field, side, width, ips, ipe, jps, jpe, device_buf, true);
}

extern "C" int wrfb200_unpack_halo(wrfb200_handle *h, int field, int side, int width,
                                   int ips, int ipe, int jps, int jpe, const float *device_buf)
{
    return halo_copy(h, field, side, width, ips, ipe, jps, jpe, const_cast<float *>(device_buf), false);
}

extern "C" int wrfb200_standin_advance_uv(wrfb200_handle *h, int field, float c, int i0, int i1, int j0, int j1)
{
    if (!h) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (int rc = wrfb200_require_r4(h, "wrfb200_standin_advance_uv")) return rc;
    if (field != WRFB200_U && field != WRFB200_V)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "stand-in update applies to u or v only");
    if (i0 > i1 || j0 > j1) return WRFB200_OK;
    const wrfb200_domain &d = h->dom;
    const int di = field == WRFB200_U ? 1 : 0, dj = field == WRFB200_V ? 1 : 0;
    if (i0 - di < d.ims || i1 > d.ime || j0 - dj < d.jms || j1 > d.jme)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "stand-in box outside memory");
    if (!h->d[field] || !h->d[WRFB200_MUDF]) return wrfb200_fail(WRFB200_ERR_STATE, "fields not allocated");
    const int ni = i1 - i0 + 1, nj = j1 - j0 + 1, nk = h->kdim;
    const long long n = (long long)ni * nk * nj;
    int prev = -1;
    cudaGetDevice(&prev);
    if (prev != h->device) cudaSetDevice(h->device);
    const int threads = ni >= 256 ? 256 : (ni >= 64 ? 64 : 32);
    const long long rows = (long long)nk * nj;
    const unsigned blocks = (unsigned)(rows < 148 * 64 ? rows : 148 * 64);
    (void)n;
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    standin_uv_kernel<<<blocks, threads, 0, h->stream>>>(
        h->d[field], h->d[WRFB200_MUDF], h->pitch3, h->pitch3 * (long long)h->kdim, h->pitch2,
        field == WRFB200_U ? 1 : h->pitch2, c, i0 - d.ims, j0 - d.jms, ni, nk, nj);
    cudaError_t e = cudaGetLastError();
    if (prev != h->device && prev >= 0) cudaSetDevice(prev);
    if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "stand-in kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    return WRFB200_OK;
}
