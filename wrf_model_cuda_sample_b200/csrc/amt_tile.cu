// amt_tile.cu -- advance_mu_t, k-parallel float4 tile kernel for sm_100a (the register-staged tile kernel).
//
// A block owns a tile of TI=128 columns (i) x TJ rows (j) and ALL levels of those columns.
// The two strictly ordered recurrences of the routine -- the column sum dmdt
// (module_small_step_em.f90:147) and the ww prefix (:161) -- are the only work done one thread per
// column; everything else is elementwise in (i,k,j) and is spread over all 8 warps with the level
// range of a row cut into contiguous chunks, one chunk per warp:
//
//   phase 1  (warp = one (row, level-chunk); lane = 4 adjacent columns, 128-bit loads)
//            dvdxi(i,k)  -> shared memory D[row][k][i]          (:142-146)
//            ww_1(i,k,j) -> shared memory W[row][k][i]          (staged for phase 2)
//   phase 2  (thread = one column)
//            dmdt = sum_k dnw(k)*D[k] in ascending k            (:147)
//            mu, mudf, muts, muave                              (:151-157)
//            ww prefix and ww -= ww_1, final ww -> W[row][k][i] (:159-172)
//   phase 3  (same mapping as phase 1)
//            t_ave, t update with horizontal fluxes and the vertical flux wdtn built from the final
//            ww in W (:208-248); ww, t, t_ave stored with 128-bit stores
//
// HBM traffic is the algorithmic minimum (44 B per 3-D point, SURVEY.md section 8d): the reference
// kernel's global scratch arrays dvdxi/wdtn/dmdt (advance_mu_t_kernel.cu:26,86,112,164-171) live in
// shared memory / registers, ww and t are touched once.  The i+1 / i-1 neighbours come from the
// adjacent lane by warp shuffle (one extra scalar load per 128 columns), the flux u + muu*u_1/msfuy is
// computed once per face and shuffled, so a point costs two IEEE divisions, not three.
// Arithmetic uses explicit round-to-nearest intrinsics in the Fortran's order: results are bit-identical
// to the reference for any -fmad setting.
//
// Layout requirement: 16-byte aligned base pointers and row pitches that are multiples of 4 floats
// (amt_tile_supported); the handle allocates rows padded to 32 floats so a warp's 512-byte row
// segment is four whole 128-byte lines.
#include <cstdint>
#include "amt_params.h"

namespace {

constexpr int TI = 128;             // columns per tile = 32 lanes x 4
constexpr int kTileThreads = 256;   // 8 warps
constexpr int kWarps = kTileThreads / 32;
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float4 ld4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float ld1(const float *p) { return __ldg(p); }
// fields this kernel also writes (t) are read through the coherent path
__device__ __forceinline__ float4 ld4_rw(const float *p) { return *reinterpret_cast<const float4 *>(p); }

__device__ __forceinline__ void st4_masked(float *p, const float4 v, const unsigned m)
{
    if (m == 0xfu) {
        *reinterpret_cast<float4 *>(p) = v;
    } else {
        if (m & 1u) p[0] = v.x;
        if (m & 2u) p[1] = v.y;
        if (m & 4u) p[2] = v.z;
        if (m & 8u) p[3] = v.w;
    }
}

template <int TJ>
__global__ void __launch_bounds__(kTileThreads, 2)
amt_tile_kernel(const AmtParams p, const int nbx, const int ti_origin)
{
    extern __shared__ __align__(16) float smem[];
    const int nk = p.nk;
    float *sD = smem;                       // [TJ][nk][TI]   dvdxi
    float *sW = sD + TJ * nk * TI;          // [TJ][nk][TI]   ww_1, then final ww
    float *s_dnw = sW + TJ * nk * TI;       // [nk] each
    float *s_fnm = s_dnw + nk;
    float *s_fnp = s_fnm + nk;
    float *s_rdnw = s_fnp + nk;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int bx = blockIdx.x % nbx;
    const int by = blockIdx.x / nbx;
    const int ti0 = ti_origin + bx * TI;    // first column of the tile (memory index, multiple of 4)
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
    float sc_mu = 0.f, sc_mu_tend = 0.f, sc_mut = 0.f, sc_msfty = 1.f, sc_ww0 = 0.f;
    if (sc_valid) {
        const long long c2 = (long long)sc_j * p.pitch2 + sc_i;
        sc_mu = p.mu[c2];
        sc_mu_tend = ld1(p.mu_tend + c2);
        sc_mut = ld1(p.mut + c2);
        sc_msfty = ld1(p.msfty + c2);
        sc_ww0 = p.ww[(long long)sc_j * p.jstride + (long long)p.k0 * p.pitch + sc_i];
    }

    // ---- elementwise mapping: warp -> (row jj, level chunk [ka,kb)), lane -> columns c..c+3 ----
    constexpr int NCH = kWarps / TJ;                    // level chunks per row
    const int jj = warp / NCH;
    const int ch = warp % NCH;
    const int L = (nk + NCH - 1) / NCH;
    const int ka = ch * L;
    const int kb = min(nk, ka + L);
    const int j = tj0 + jj;
    const bool row_on = (j <= p.j1) && (ka < kb);       // warp-uniform
    const int c = ti0 + 4 * lane;
    // columns this lane must LOAD: anything inside the computed range widened by the one-cell ring
    const bool act = row_on && (c <= p.i1 + 1) && (c + 3 >= p.i0 - 1);
    unsigned m = 0;                                     // columns this lane OWNS (stores / valid results)
#pragma unroll
    for (int q = 0; q < 4; ++q) m |= (c + q >= p.i0 && c + q <= p.i1) ? (1u << q) : 0u;
    if (!row_on) m = 0;
    const bool need_e = (lane == 31) && (m & 8u);       // east neighbour lives in the next tile
    const bool need_w = (lane == 0) && (m & 1u);        // west neighbour lives in the previous tile

    const long long c2 = (long long)j * p.pitch2 + c;
    const long long rowbase = (long long)j * p.jstride + (long long)p.k0 * p.pitch + c;
    float *dD = sD + (jj * nk) * TI + 4 * lane;
    float *dW = sW + (jj * nk) * TI + 4 * lane;

    // =========================== phase 1 ===========================
    if (row_on) {
        float4 muu = {0, 0, 0, 0}, mfu = {1, 1, 1, 1}, muv_s = muu, muv_n = muu, mvi_s = muu, mvi_n = muu, cof = muu;
        float muu_e = 0.f, mfu_e = 1.f;
        if (act) {
            muu = ld4(p.muu + c2);
            mfu = ld4(p.msfuy + c2);
            muv_s = ld4(p.muv + c2);
            muv_n = ld4(p.muv + c2 + p.pitch2);
            mvi_s = ld4(p.msfvx_inv + c2);
            mvi_n = ld4(p.msfvx_inv + c2 + p.pitch2);
            const float4 mx = ld4(p.msftx + c2), my = ld4(p.msfty + c2);
            cof.x = f_mul(mx.x, my.x); cof.y = f_mul(mx.y, my.y);          // :142 msftx*msfty
            cof.z = f_mul(mx.z, my.z); cof.w = f_mul(mx.w, my.w);
        }
        if (need_e) { muu_e = ld1(p.muu + c2 + 4); mfu_e = ld1(p.msfuy + c2 + 4); }

#pragma unroll 2
        for (int k = ka; k < kb; ++k) {
            const long long o = rowbase + (long long)k * p.pitch;
            float4 U = {0, 0, 0, 0}, U1 = U, VS = U, VN = U, V1S = U, V1N = U, W1 = U;
            float u_e = 0.f, u1_e = 0.f;
            if (act) {
                U = ld4(p.u + o);
                U1 = ld4(p.u_1 + o);
                VS = ld4(p.v + o);
                VN = ld4(p.v + o + p.jstride);
                V1S = ld4(p.v_1 + o);
                V1N = ld4(p.v_1 + o + p.jstride);
                W1 = ld4(p.ww_1 + o);
            }
            if (need_e) { u_e = ld1(p.u + o + 4); u1_e = ld1(p.u_1 + o + 4); }
            // u-face flux u + muu*u_1/msfuy (:145-146), one division per face
            const float f0 = f_add(U.x, f_div(f_mul(muu.x, U1.x), mfu.x));
            const float f1 = f_add(U.y, f_div(f_mul(muu.y, U1.y), mfu.y));
            const float f2 = f_add(U.z, f_div(f_mul(muu.z, U1.z), mfu.z));
            const float f3 = f_add(U.w, f_div(f_mul(muu.w, U1.w), mfu.w));
            float f4 = __shfl_down_sync(FULL, f0, 1);
            if (need_e) f4 = f_add(u_e, f_div(f_mul(muu_e, u1_e), mfu_e));
            // v-face fluxes v + muv*v_1*msfvx_inv (:143-144)
            float4 dv;
            {
                const float n = f_add(VN.x, f_mul(f_mul(muv_n.x, V1N.x), mvi_n.x));
                const float s = f_add(VS.x, f_mul(f_mul(muv_s.x, V1S.x), mvi_s.x));
                dv.x = f_mul(cof.x, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f1, f0))));
            }
            {
                const float n = f_add(VN.y, f_mul(f_mul(muv_n.y, V1N.y), mvi_n.y));
                const float s = f_add(VS.y, f_mul(f_mul(muv_s.y, V1S.y), mvi_s.y));
                dv.y = f_mul(cof.y, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f2, f1))));
            }
            {
                const float n = f_add(VN.z, f_mul(f_mul(muv_n.z, V1N.z), mvi_n.z));
                const float s = f_add(VS.z, f_mul(f_mul(muv_s.z, V1S.z), mvi_s.z));
                dv.z = f_mul(cof.z, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f3, f2))));
            }
            {
                const float n = f_add(VN.w, f_mul(f_mul(muv_n.w, V1N.w), mvi_n.w));
                const float s = f_add(VS.w, f_mul(f_mul(muv_s.w, V1S.w), mvi_s.w));
                dv.w = f_mul(cof.w, f_add(f_mul(p.rdy, f_sub(n, s)), f_mul(p.rdx, f_sub(f4, f3))));
            }
            *reinterpret_cast<float4 *>(dD + k * TI) = dv;
            *reinterpret_cast<float4 *>(dW + k * TI) = W1;
        }
    }
    __syncthreads();

    // =========================== phase 2 ===========================
    if (sc_valid) {
        const float *D = sD + (sc_jj * nk) * TI + sc_ci;
        float *W = sW + (sc_jj * nk) * TI + sc_ci;
        float dmdt = 0.0f;                                                  // :115
#pragma unroll 4
        for (int k = 0; k < nk; ++k) dmdt = f_add(dmdt, f_mul(s_dnw[k], D[k * TI]));   // :147
        const long long c2s = (long long)sc_j * p.pitch2 + sc_i;
        const float tend = f_add(dmdt, sc_mu_tend);
        const float mu_new = f_add(sc_mu, f_mul(p.dts, tend));              // :153
        p.mu[c2s] = mu_new;
        p.mudf[c2s] = tend;                                                 // :154
        p.muts[c2s] = f_add(sc_mut, mu_new);                                // :155
        p.muave[c2s] = f_mul(0.5f, f_add(f_mul(f_add(1.0f, p.epssm), mu_new),
                                         f_mul(f_sub(1.0f, p.epssm), sc_mu)));          // :156
        float w = sc_ww0;                                                   // ww(i,1,j) is an input (:159 starts at k=2)
        W[0] = f_sub(w, W[0]);                                              // :170 at k=1
#pragma unroll 4
        for (int k = 1; k < nk; ++k) {
            const float inner = f_add(f_add(dmdt, D[(k - 1) * TI]), sc_mu_tend);
            w = f_sub(w, f_div(f_mul(s_dnw[k - 1], inner), sc_msfty));      // :161
            W[k * TI] = f_sub(w, W[k * TI]);                                // :170
        }
    }
    __syncthreads();

    // =========================== phase 3 ===========================
    if (row_on) {
        float4 mx = {0, 0, 0, 0}, dtm = mx;
        if (act) {
            mx = ld4(p.msftx + c2);
            const float4 my = ld4(p.msfty + c2);
            dtm.x = f_mul(p.dts, my.x); dtm.y = f_mul(p.dts, my.y);         // :237 dts*msfty (== msfty*dts, :212)
            dtm.z = f_mul(p.dts, my.z); dtm.w = f_mul(p.dts, my.w);
        }
        const float hrdy = f_mul(0.5f, p.rdy);                              // :240
        const float hrdx = f_mul(0.5f, p.rdx);                              // :243

        // rolling state: t_1 at level k (C) and the flux through the bottom face of level k
        float4 T1C = {0, 0, 0, 0}, wd_k = {0, 0, 0, 0};                     // :220 wdtn(i,1)=0
        if (act) T1C = ld4(p.t_1 + rowbase + (long long)ka * p.pitch);
        if (ka > 0) {
            float4 T1P = {0, 0, 0, 0};
            if (act) T1P = ld4(p.t_1 + rowbase + (long long)(ka - 1) * p.pitch);
            const float4 wk = *reinterpret_cast<const float4 *>(dW + ka * TI);
            const float a = s_fnm[ka], b = s_fnp[ka];
            wd_k.x = f_mul(wk.x, f_add(f_mul(a, T1C.x), f_mul(b, T1P.x)));  // :227
            wd_k.y = f_mul(wk.y, f_add(f_mul(a, T1C.y), f_mul(b, T1P.y)));
            wd_k.z = f_mul(wk.z, f_add(f_mul(a, T1C.z), f_mul(b, T1P.z)));
            wd_k.w = f_mul(wk.w, f_add(f_mul(a, T1C.w), f_mul(b, T1P.w)));
        }

        for (int k = ka; k < kb; ++k) {
            const long long o = rowbase + (long long)k * p.pitch;
            const bool has_n = (k + 1 < nk);
            float4 T1S = {0, 0, 0, 0}, T1N = T1S, T1U = T1S, U = T1S, VS = T1S, VN = T1S, FT = T1S, T = T1S;
            float u_e = 0.f, t1_e = 0.f, t1_w = 0.f;
            if (act) {
                T1S = ld4(p.t_1 + o - p.jstride);
                T1N = ld4(p.t_1 + o + p.jstride);
                if (has_n) T1U = ld4(p.t_1 + o + p.pitch);
                U = ld4(p.u + o);
                VS = ld4(p.v + o);
                VN = ld4(p.v + o + p.jstride);
                FT = ld4(p.ft + o);
                T = ld4_rw(p.t + o);
            }
            if (need_e) { u_e = ld1(p.u + o + 4); t1_e = ld1(p.t_1 + o + 4); }
            if (need_w) { t1_w = ld1(p.t_1 + o - 1); }
            const float4 wk = *reinterpret_cast<const float4 *>(dW + k * TI);
            float4 wd_n = {0, 0, 0, 0};                                     // :221 wdtn(i,kde)=0
            if (has_n) {
                const float4 wn = *reinterpret_cast<const float4 *>(dW + (k + 1) * TI);
                const float a = s_fnm[k + 1], b = s_fnp[k + 1];
                wd_n.x = f_mul(wn.x, f_add(f_mul(a, T1U.x), f_mul(b, T1C.x)));          // :227
                wd_n.y = f_mul(wn.y, f_add(f_mul(a, T1U.y), f_mul(b, T1C.y)));
                wd_n.z = f_mul(wn.z, f_add(f_mul(a, T1U.z), f_mul(b, T1C.z)));
                wd_n.w = f_mul(wn.w, f_add(f_mul(a, T1U.w), f_mul(b, T1C.w)));
            }
            // i+1 / i-1 neighbours of the lane's 4 columns
            float t1_ee = __shfl_down_sync(FULL, T1C.x, 1);
            float t1_ww = __shfl_up_sync(FULL, T1C.w, 1);
            float u_ee = __shfl_down_sync(FULL, U.x, 1);
            if (lane == 31) { t1_ee = t1_e; u_ee = u_e; }
            if (lane == 0) t1_ww = t1_w;

            const float rd = s_rdnw[k];
            float4 TO;
#define AMT_THETA(X, UW, UE, TW, TE)                                                                              \
            {                                                                                                     \
                const float t_mid = f_add(T.X, f_mul(dtm.X, FT.X));                                    /* :212 */ \
                const float fy = f_mul(hrdy, f_sub(f_mul(VN.X, f_add(T1N.X, T1C.X)),                             \
                                                   f_mul(VS.X, f_add(T1C.X, T1S.X))));             /* :240-242 */ \
                const float fx = f_mul(hrdx, f_sub(f_mul(UE, f_add(TE, T1C.X)),                                  \
                                                   f_mul(UW, f_add(T1C.X, TW))));                  /* :243-245 */ \
                const float fz = f_mul(rd, f_sub(wd_n.X, wd_k.X));                                     /* :246 */ \
                TO.X = f_sub(t_mid, f_mul(dtm.X, f_add(f_mul(mx.X, f_add(fy, fx)), fz)));              /* :237 */ \
            }
            AMT_THETA(x, U.x, U.y, t1_ww, T1C.y)
            AMT_THETA(y, U.y, U.z, T1C.x, T1C.z)
            AMT_THETA(z, U.z, U.w, T1C.y, T1C.w)
            AMT_THETA(w, U.w, u_ee, T1C.z, t1_ee)
#undef AMT_THETA
            if (m) {
                st4_masked(p.ww + o, wk, m);
                st4_masked(p.t_ave + o, T, m);                              // :211
                st4_masked(p.t + o, TO, m);
            }
            T1C = T1U;
            wd_k = wd_n;
        }
    }
}

template <int TJ>
cudaError_t launch_tj(const AmtParams &p, cudaStream_t stream)
{
    const int ti_origin = p.i0 & ~31;                       // tiles start on a 128-byte boundary
    const int ni = p.i1 - ti_origin + 1;
    const int nj = p.j1 - p.j0 + 1;
    const int nbx = (ni + TI - 1) / TI;
    const int nby = (nj + TJ - 1) / TJ;
    const size_t smem = ((size_t)2 * TJ * p.nk * TI + 4 * (size_t)p.nk) * sizeof(float);
    if (smem > (size_t)kMaxDynSmemOptIn) return cudaErrorInvalidValue;
    static bool raised[64] = {};            // per template instance
    cudaError_t e = amt_raise_smem_limit(amt_tile_kernel<TJ>, raised);
    if (e != cudaSuccess) return e;
    (void)cudaGetLastError();   // a launch status must not inherit a stale error of some earlier, unrelated call
    amt_tile_kernel<TJ><<<(unsigned)((long long)nbx * nby), kTileThreads, smem, stream>>>(p, nbx, ti_origin);
    return cudaGetLastError();
}

constexpr size_t kSmemMax = 227 * 1024;
size_t tile_smem(int tj, int nk) { return ((size_t)2 * tj * nk * TI + 4 * (size_t)nk) * sizeof(float); }

}  // namespace

// a one-row tile: 1040 B per level
bool amt_tile_levels_fit(const AmtParams &p, int *max_levels)
{
    const int most = (int)(kSmemMax / tile_smem(1, 1));
    if (max_levels) *max_levels = most;
    return p.nk <= most;
}

bool amt_tile_supported(const AmtParams &p)
{
    const void *ptrs3[] = {p.ww, p.ww_1, p.u, p.u_1, p.v, p.v_1, p.t, p.t_1, p.t_ave, p.ft};
    const void *ptrs2[] = {p.mu, p.mut, p.muave, p.muts, p.muu, p.muv, p.mudf, p.mu_tend,
                           p.msfuy, p.msfvx_inv, p.msftx, p.msfty};
    for (const void *q : ptrs3) if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) return false;
    for (const void *q : ptrs2) if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) return false;
    if (p.pitch % 4 != 0 || p.pitch2 % 4 != 0 || p.jstride % 4 != 0) return false;
    return amt_tile_levels_fit(p);
}

cudaError_t amt_launch_tile(const AmtParams &p, cudaStream_t stream)
{
    if (p.i1 < p.i0 || p.j1 < p.j0 || p.nk <= 0) return cudaSuccess;
    // Two resident blocks per SM need 2*smem <= 227 KB; prefer the taller tile (more v / t_1 row reuse
    // inside a block) while that still holds.
    const int nj = p.j1 - p.j0 + 1;
    if (nj >= 2 && 2 * tile_smem(2, p.nk) <= kSmemMax) return launch_tj<2>(p, stream);
    return launch_tj<1>(p, stream);
}
