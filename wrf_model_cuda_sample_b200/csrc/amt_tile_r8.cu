// amt_tile_r8.cu -- advance_mu_t in binary64 (WRF built with -r8): the k-parallel double2 tile kernel, sm_100a.
//
// The structure of amt_tile.cu (read that header first) with 64-column tiles: a lane owns 2 adjacent
// columns and moves them with one 16-byte double2 access, so a warp covers the 64 columns of a tile row.
//
//   phase 1  (warp = one (row, level-chunk); lane = 2 adjacent columns)
//            dvdxi(i,k)  -> shared memory D[row][k][i]          (:142-146)
//            ww_1(i,k,j) -> shared memory W[row][k][i]
//   phase 2  (thread = one column)
//            dmdt sum, mu / mudf / muts / muave, ww prefix; final ww -> W   (:147-172)
//   phase 3  (same mapping as phase 1)
//            t_ave, t with the horizontal and vertical fluxes; ww, t, t_ave stored (:208-248)
//
// Why 64 columns and not 128: D and W hold every level of the tile, 2 x 8 B x TI per level and row.  At
// TI = 128 that is 2 KB x nk, over the 227 KB a block may have at nk = 120; at TI = 64 a one-row tile needs
// 1056 B x nk (with the four 1-D coefficient arrays), so every nk <= 220 fits (amt_tile_supported).  Two
// rows per tile and two resident blocks per SM while nk <= 55, one row otherwise.
//
// Arithmetic: every operation is one __d*_rn intrinsic in the Fortran's order (amt_params.h), so the result is
// the Fortran's evaluated in real*8 bit for bit.  Division is the IEEE __ddiv_rn; the float pipe
// kernel's hoisted reciprocal is proven for the 2^23 binary32 mantissas only and is not used here.
//
// Layout requirement: 16-byte aligned base pointers and row pitches that are even numbers of doubles.
// WRF's default halo-5 patch (ims = ids-5 .. ime = ide+5, e.g. 1810 points on a 1800-point domain) is such
// a layout, so caller-owned dense device arrays take this kernel directly.
#include <cstdint>
#include "amt_params.h"

namespace {

constexpr int TI = 64;              // columns per tile = 32 lanes x 2
constexpr int kTileThreads = 256;   // 8 warps
constexpr int kWarps = kTileThreads / 32;
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double2 ld2(const double *p) { return __ldg(reinterpret_cast<const double2 *>(p)); }
__device__ __forceinline__ double ld1(const double *p) { return __ldg(p); }
// fields this kernel also writes (t) are read through the coherent path
__device__ __forceinline__ double2 ld2_rw(const double *p) { return *reinterpret_cast<const double2 *>(p); }

__device__ __forceinline__ void st2_masked(double *p, const double2 v, const unsigned m)
{
    if (m == 0x3u) {
        *reinterpret_cast<double2 *>(p) = v;
    } else {
        if (m & 1u) p[0] = v.x;
        if (m & 2u) p[1] = v.y;
    }
}

}  // namespace

template <int TJ>
__global__ void __launch_bounds__(kTileThreads, 2)
amt_tile_kernel_r8(const AmtParamsR8 p, const int nbx, const int ti_origin)
{
    extern __shared__ __align__(16) double smem_r8[];
    const int nk = p.nk;
    double *sD = smem_r8;                   // [TJ][nk][TI]   dvdxi
    double *sW = sD + TJ * nk * TI;         // [TJ][nk][TI]   ww_1, then final ww
    double *s_dnw = sW + TJ * nk * TI;      // [nk] each
    double *s_fnm = s_dnw + nk;
    double *s_fnp = s_fnm + nk;
    double *s_rdnw = s_fnp + nk;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int bx = blockIdx.x % nbx;
    const int by = blockIdx.x / nbx;
    const int ti0 = ti_origin + bx * TI;    // first column of the tile (memory index, even)
    const int tj0 = p.j0 + by * TJ;         // first row of the tile

    for (int x = tid; x < nk; x += kTileThreads) {
        s_dnw[x] = p.dnw[p.k0 + x];
        s_fnm[x] = p.fnm[p.k0 + x];
        s_fnp[x] = p.fnp[p.k0 + x];
        s_rdnw[x] = p.rdnw[p.k0 + x];
    }

    // ---- phase-2 operands of this thread's column, fetched early so their latency hides behind phase 1 ----
    const int sc_jj = tid / TI, sc_ci = tid % TI;
    const int sc_i = ti0 + sc_ci, sc_j = tj0 + sc_jj;
    const bool sc_valid = (tid < TI * TJ) && sc_i >= p.i0 && sc_i <= p.i1 && sc_j <= p.j1;
    double sc_mu = 0., sc_mu_tend = 0., sc_mut = 0., sc_msfty = 1., sc_ww0 = 0.;
    if (sc_valid) {
        const long long c2 = (long long)sc_j * p.pitch2 + sc_i;
        sc_mu = p.mu[c2];
        sc_mu_tend = ld1(p.mu_tend + c2);
        sc_mut = ld1(p.mut + c2);
        sc_msfty = ld1(p.msfty + c2);
        sc_ww0 = p.ww[(long long)sc_j * p.jstride + (long long)p.k0 * p.pitch + sc_i];
    }

    // ---- elementwise mapping: warp -> (row jj, level chunk [ka,kb)), lane -> columns c, c+1 ----
    constexpr int NCH = kWarps / TJ;                    // level chunks per row
    const int jj = warp / NCH;
    const int ch = warp % NCH;
    const int L = (nk + NCH - 1) / NCH;
    const int ka = ch * L;
    const int kb = min(nk, ka + L);
    const int j = tj0 + jj;
    const bool row_on = (j <= p.j1) && (ka < kb);       // warp-uniform
    const int c = ti0 + 2 * lane;
    // columns this lane must LOAD: anything inside the computed range widened by the one-cell ring
    const bool act = row_on && (c <= p.i1 + 1) && (c + 1 >= p.i0 - 1);
    unsigned m = 0;                                     // columns this lane OWNS (stores / valid results)
    if (c >= p.i0 && c <= p.i1) m |= 1u;
    if (c + 1 >= p.i0 && c + 1 <= p.i1) m |= 2u;
    if (!row_on) m = 0;
    const bool need_e = (lane == 31) && (m & 2u);       // east neighbour lives in the next tile
    const bool need_w = (lane == 0) && (m & 1u);        // west neighbour lives in the previous tile

    const long long c2 = (long long)j * p.pitch2 + c;
    const long long rowbase = (long long)j * p.jstride + (long long)p.k0 * p.pitch + c;
    double *dD = sD + (jj * nk) * TI + 2 * lane;
    double *dW = sW + (jj * nk) * TI + 2 * lane;

    // =========================== phase 1 ===========================
    if (row_on) {
        double2 muu = {0, 0}, mfu = {1, 1}, muv_s = muu, muv_n = muu, mvi_s = muu, mvi_n = muu, cof = muu;
        double muu_e = 0., mfu_e = 1.;
        if (act) {
            muu = ld2(p.muu + c2);
            mfu = ld2(p.msfuy + c2);
            muv_s = ld2(p.muv + c2);
            muv_n = ld2(p.muv + c2 + p.pitch2);
            mvi_s = ld2(p.msfvx_inv + c2);
            mvi_n = ld2(p.msfvx_inv + c2 + p.pitch2);
            const double2 mx = ld2(p.msftx + c2), my = ld2(p.msfty + c2);
            cof.x = f_mul(mx.x, my.x); cof.y = f_mul(mx.y, my.y);          // :142 msftx*msfty
        }
        if (need_e) { muu_e = ld1(p.muu + c2 + 2); mfu_e = ld1(p.msfuy + c2 + 2); }

#pragma unroll 2
        for (int k = ka; k < kb; ++k) {
            const long long o = rowbase + (long long)k * p.pitch;
            double2 U = {0, 0}, U1 = U, VS = U, VN = U, V1S = U, V1N = U, W1 = U;
            double u_e = 0., u1_e = 0.;
            if (act) {
                U = ld2(p.u + o);
                U1 = ld2(p.u_1 + o);
                VS = ld2(p.v + o);
                VN = ld2(p.v + o + p.jstride);
                V1S = ld2(p.v_1 + o);
                V1N = ld2(p.v_1 + o + p.jstride);
                W1 = ld2(p.ww_1 + o);
            }
            if (need_e) { u_e = ld1(p.u + o + 2); u1_e = ld1(p.u_1 + o + 2); }
            // u-face flux u + muu*u_1/msfuy (:145-146), one division per face
            const double f0 = f_add(U.x, f_div(f_mul(muu.x, U1.x), mfu.x));
            const double f1 = f_add(U.y, f_div(f_mul(muu.y, U1.y), mfu.y));
            double f2 = __shfl_down_sync(FULL, f0, 1);
            if (need_e) f2 = f_add(u_e, f_div(f_mul(muu_e, u1_e), mfu_e));
            // v-face fluxes v + muv*v_1*msfvx_inv (:143-144)
            double2 dv;
            {
                const double n = f_add(VN.x, f_mul(f_mul(muv_n.x, V1N.x), mvi_n.x));
                const double s = f_add(VS.x, f_mul(f_mul(muv_s.x, V1S.x), mvi_s.x));
                dv.x = f_mul(cof.x, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f1, f0))));
            }
            {
                const double n = f_add(VN.y, f_mul(f_mul(muv_n.y, V1N.y), mvi_n.y));
                const double s = f_add(VS.y, f_mul(f_mul(muv_s.y, V1S.y), mvi_s.y));
                dv.y = f_mul(cof.y, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f2, f1))));
            }
            *reinterpret_cast<double2 *>(dD + k * TI) = dv;
            *reinterpret_cast<double2 *>(dW + k * TI) = W1;
        }
    }
    __syncthreads();

    // =========================== phase 2 ===========================
    if (sc_valid) {
        const double *D = sD + (sc_jj * nk) * TI + sc_ci;
        double *W = sW + (sc_jj * nk) * TI + sc_ci;
        double dmdt = 0.;                                                   // :115
#pragma unroll 4
        for (int k = 0; k < nk; ++k) dmdt = f_add(dmdt, f_mul(s_dnw[k], D[k * TI]));   // :147
        const long long c2s = (long long)sc_j * p.pitch2 + sc_i;
        const double tend = f_add(dmdt, sc_mu_tend);
        const double mu_new = f_add(sc_mu, f_mul(p.dts, tend));             // :153
        p.mu[c2s] = mu_new;
        p.mudf[c2s] = tend;                                                 // :154
        p.muts[c2s] = f_add(sc_mut, mu_new);                                // :155
        p.muave[c2s] = f_mul(0.5, f_add(f_mul(f_add(1.0, p.epssm), mu_new),
                                        f_mul(f_sub(1.0, p.epssm), sc_mu)));            // :156
        double w = sc_ww0;                                                  // ww(i,1,j) is an input (:159 starts at k=2)
        W[0] = f_sub(w, W[0]);                                              // :170 at k=1
#pragma unroll 4
        for (int k = 1; k < nk; ++k) {
            const double inner = f_add(f_add(dmdt, D[(k - 1) * TI]), sc_mu_tend);
            w = f_sub(w, f_div(f_mul(s_dnw[k - 1], inner), sc_msfty));      // :161
            W[k * TI] = f_sub(w, W[k * TI]);                                // :170
        }
    }
    __syncthreads();

    // =========================== phase 3 ===========================
    if (row_on) {
        double2 mx = {0, 0}, dtm = mx;
        if (act) {
            mx = ld2(p.msftx + c2);
            const double2 my = ld2(p.msfty + c2);
            dtm.x = f_mul(p.dts, my.x); dtm.y = f_mul(p.dts, my.y);         // :237 dts*msfty (== msfty*dts, :212)
        }
        const double hrdy = f_mul(0.5, p.rdy);                              // :240
        const double hrdx = f_mul(0.5, p.rdx);                              // :243

        // rolling state: t_1 at level k (C) and the flux through the bottom face of level k
        double2 T1C = {0, 0}, wd_k = {0, 0};                                // :220 wdtn(i,1)=0
        if (act) T1C = ld2(p.t_1 + rowbase + (long long)ka * p.pitch);
        if (ka > 0) {
            double2 T1P = {0, 0};
            if (act) T1P = ld2(p.t_1 + rowbase + (long long)(ka - 1) * p.pitch);
            const double2 wk = *reinterpret_cast<const double2 *>(dW + ka * TI);
            const double a = s_fnm[ka], b = s_fnp[ka];
            wd_k.x = f_mul(wk.x, f_add(f_mul(a, T1C.x), f_mul(b, T1P.x)));  // :227
            wd_k.y = f_mul(wk.y, f_add(f_mul(a, T1C.y), f_mul(b, T1P.y)));
        }

        for (int k = ka; k < kb; ++k) {
            const long long o = rowbase + (long long)k * p.pitch;
            const bool has_n = (k + 1 < nk);
            double2 T1S = {0, 0}, T1N = T1S, T1U = T1S, U = T1S, VS = T1S, VN = T1S, FT = T1S, T = T1S;
            double u_e = 0., t1_e = 0., t1_w = 0.;
            if (act) {
                T1S = ld2(p.t_1 + o - p.jstride);
                T1N = ld2(p.t_1 + o + p.jstride);
                if (has_n) T1U = ld2(p.t_1 + o + p.pitch);
                U = ld2(p.u + o);
                VS = ld2(p.v + o);
                VN = ld2(p.v + o + p.jstride);
                FT = ld2(p.ft + o);
                T = ld2_rw(p.t + o);
            }
            if (need_e) { u_e = ld1(p.u + o + 2); t1_e = ld1(p.t_1 + o + 2); }
            if (need_w) { t1_w = ld1(p.t_1 + o - 1); }
            const double2 wk = *reinterpret_cast<const double2 *>(dW + k * TI);
            double2 wd_n = {0, 0};                                          // :221 wdtn(i,kde)=0
            if (has_n) {
                const double2 wn = *reinterpret_cast<const double2 *>(dW + (k + 1) * TI);
                const double a = s_fnm[k + 1], b = s_fnp[k + 1];
                wd_n.x = f_mul(wn.x, f_add(f_mul(a, T1U.x), f_mul(b, T1C.x)));          // :227
                wd_n.y = f_mul(wn.y, f_add(f_mul(a, T1U.y), f_mul(b, T1C.y)));
            }
            // i+1 / i-1 neighbours of the lane's 2 columns
            double t1_ee = __shfl_down_sync(FULL, T1C.x, 1);
            double t1_ww = __shfl_up_sync(FULL, T1C.y, 1);
            double u_ee = __shfl_down_sync(FULL, U.x, 1);
            if (lane == 31) { t1_ee = t1_e; u_ee = u_e; }
            if (lane == 0) t1_ww = t1_w;

            const double rd = s_rdnw[k];
            double2 TO;
#define AMT_THETA(X, UW, UE, TW, TE)                                                                              \
            {                                                                                                     \
                const double t_mid = f_add(T.X, f_mul(dtm.X, FT.X));                                   /* :212 */ \
                const double fy = f_mul(hrdy, f_sub(f_mul(VN.X, f_add(T1N.X, T1C.X)),                            \
                                                    f_mul(VS.X, f_add(T1C.X, T1S.X))));            /* :240-242 */ \
                const double fx = f_mul(hrdx, f_sub(f_mul(UE, f_add(TE, T1C.X)),                                 \
                                                    f_mul(UW, f_add(T1C.X, TW))));                 /* :243-245 */ \
                const double fz = f_mul(rd, f_sub(wd_n.X, wd_k.X));                                    /* :246 */ \
                TO.X = f_sub(t_mid, f_mul(dtm.X, f_add(f_mul(mx.X, f_add(fy, fx)), fz)));              /* :237 */ \
            }
            AMT_THETA(x, U.x, U.y, t1_ww, T1C.y)
            AMT_THETA(y, U.y, u_ee, T1C.x, t1_ee)
#undef AMT_THETA
            if (m) {
                st2_masked(p.ww + o, wk, m);
                st2_masked(p.t_ave + o, T, m);                              // :211
                st2_masked(p.t + o, TO, m);
            }
            T1C = T1U;
            wd_k = wd_n;
        }
    }
}

namespace {

size_t tile_smem_r8(int tj, int nk) { return ((size_t)2 * tj * nk * TI + 4 * (size_t)nk) * sizeof(double); }

template <int TJ>
cudaError_t launch_tj(const AmtParamsR8 &p, cudaStream_t stream)
{
    const int ti_origin = p.i0 & ~15;                       // tiles start on a 128-byte boundary of the row
    const int ni = p.i1 - ti_origin + 1;
    const int nj = p.j1 - p.j0 + 1;
    const int nbx = (ni + TI - 1) / TI;
    const int nby = (nj + TJ - 1) / TJ;
    const size_t smem = tile_smem_r8(TJ, p.nk);
    if (smem > (size_t)kMaxDynSmemOptIn) return cudaErrorInvalidValue;
    static bool raised[64] = {};            // per template instance
    cudaError_t e = amt_raise_smem_limit(amt_tile_kernel_r8<TJ>, raised);
    if (e != cudaSuccess) return e;
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    amt_tile_kernel_r8<TJ><<<(unsigned)((long long)nbx * nby), kTileThreads, smem, stream>>>(p, nbx, ti_origin);
    return cudaGetLastError();
}

}  // namespace

bool amt_tile_supported(const AmtParamsR8 &p)
{
    const void *ptrs3[] = {p.ww, p.ww_1, p.u, p.u_1, p.v, p.v_1, p.t, p.t_1, p.t_ave, p.ft};
    const void *ptrs2[] = {p.mu, p.mut, p.muave, p.muts, p.muu, p.muv, p.mudf, p.mu_tend,
                           p.msfuy, p.msfvx_inv, p.msftx, p.msfty};
    for (const void *q : ptrs3) if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) return false;
    for (const void *q : ptrs2) if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) return false;
    if (p.pitch % 2 != 0 || p.pitch2 % 2 != 0 || p.jstride % 2 != 0) return false;
    if (tile_smem_r8(1, p.nk) > (size_t)kMaxDynSmemOptIn) return false;        // nk <= 220
    return true;
}

cudaError_t amt_launch_tile(const AmtParamsR8 &p, cudaStream_t stream)
{
    if (p.i1 < p.i0 || p.j1 < p.j0 || p.nk <= 0) return cudaSuccess;
    // two-row tiles while two blocks still fit an SM (nk <= 55), one-row tiles otherwise
    const int nj = p.j1 - p.j0 + 1;
    if (nj >= 2 && 2 * tile_smem_r8(2, p.nk) <= (size_t)kMaxDynSmemOptIn) return launch_tj<2>(p, stream);
    return launch_tj<1>(p, stream);
}
