// amt_column.cu -- advance_mu_t, one thread per (i,j) column.  Works on ANY layout (no alignment
// or pitch requirement), so it serves caller-owned device arrays in the dense Fortran layout and is
// the simple cross-check for the tile kernel.  sm_100a.  amt_column_kernel_r8 is the same body in binary64
// (the any-layout fallback of real*8 handles).
//
// Per column (SURVEY.md section 8, "Exact semantics"; module_small_step_em.f90 lines cited inline):
//   sweep 1 (k ascending): dvdxi(k) -> shared memory, dmdt += dnw(k)*dvdxi(k)
//   2-D update of mu, mudf, muts, muave
//   sweep 2 (k ascending): ww prefix, ww -= ww_1, t_ave, t update with the vertical flux wdtn
// The reference kernel keeps dvdxi/wdtn as full 3-D global arrays and dmdt as a 2-D global array
// (advance_mu_t_kernel.cu:86,112,117,164-171) and sweeps k six times; here dvdxi lives in shared
// memory ([k][thread], conflict-free), wdtn and dmdt in registers, and k is swept twice.
#include "amt_column_body.h"

namespace {

constexpr int kColThreads = 128;

__global__ void __launch_bounds__(kColThreads)
amt_column_kernel(const AmtParams p, const int nbx)
{
    extern __shared__ float s_dvdxi[];                  // [nk][kColThreads]
    const int tid = threadIdx.x;
    const int bx = blockIdx.x % nbx;
    const int by = blockIdx.x / nbx;
    const int i = p.i0 + bx * kColThreads + tid;
    const int j = p.j0 + by;
    if (i > p.i1) return;                               // no block-wide barrier is used below

    amt_column_thread(p, i, j, s_dvdxi + tid, kColThreads);
}

}  // namespace

// Outside the anonymous namespace, like amt_tile_kernel_r8: the symbol then carries no hash of the source path, so
// the library's kernel and this file compiled elsewhere (tests/test_r8.py compares their SASS) have the same name.
__global__ void __launch_bounds__(kColThreads)
amt_column_kernel_r8(const AmtParamsR8 p, const int nbx)
{
    extern __shared__ double s_dvdxi_r8[];              // [nk][kColThreads]
    const int tid = threadIdx.x;
    const int bx = blockIdx.x % nbx;
    const int by = blockIdx.x / nbx;
    const int i = p.i0 + bx * kColThreads + tid;
    const int j = p.j0 + by;
    if (i > p.i1) return;

    amt_column_thread(p, i, j, s_dvdxi_r8 + tid, kColThreads);
}

namespace {

// One launcher for both element types (the two kernels differ in their argument block only).
template <class P, class T, class K>
cudaError_t launch_column(const P &p, K kernel, bool (&raised)[64], cudaStream_t stream)
{
    const int ni = p.i1 - p.i0 + 1, nj = p.j1 - p.j0 + 1;
    if (ni <= 0 || nj <= 0 || p.nk <= 0) return cudaSuccess;
    const int nbx = (ni + kColThreads - 1) / kColThreads;
    const size_t smem = (size_t)p.nk * kColThreads * sizeof(T);
    if (smem > (size_t)kMaxDynSmemOptIn) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {                   // opt in once per device; the limit is only ever raised
        cudaError_t e = amt_raise_smem_limit(kernel, raised);
        if (e != cudaSuccess) return e;
    }
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    kernel<<<(unsigned)((long long)nbx * nj), kColThreads, smem, stream>>>(p, nbx);
    return cudaGetLastError();
}

template <class P, class T>
bool column_levels_fit(const P &p, int *max_levels)
{
    const int most = kMaxDynSmemOptIn / (int)(kColThreads * sizeof(T));
    if (max_levels) *max_levels = most;
    return p.nk <= most;
}

}  // namespace

// the [nk][128] dvdxi slab in dynamic shared memory: 512 B per level in binary32, 1 KB in binary64
bool amt_column_levels_fit(const AmtParams &p, int *max_levels) { return column_levels_fit<AmtParams, float>(p, max_levels); }
bool amt_column_levels_fit(const AmtParamsR8 &p, int *max_levels) { return column_levels_fit<AmtParamsR8, double>(p, max_levels); }

cudaError_t amt_launch_column(const AmtParams &p, cudaStream_t stream)
{
    static bool raised[64] = {};
    return launch_column<AmtParams, float>(p, amt_column_kernel, raised, stream);
}

cudaError_t amt_launch_column(const AmtParamsR8 &p, cudaStream_t stream)
{
    static bool raised[64] = {};
    return launch_column<AmtParamsR8, double>(p, amt_column_kernel_r8, raised, stream);
}
