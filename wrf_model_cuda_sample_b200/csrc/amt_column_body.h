// amt_column_body.h -- advance_mu_t for ONE (i,j) column, executed by one thread (any layout, scalar accesses).
// Shared by amt_column.cu (the any-layout kernels, float and double) and amt_pipe.cu (the narrow remainder strip
// of a row of 128-column tiles, folded into the same launch).  module_small_step_em.f90 lines cited inline.
//   sweep 1 (k ascending): dvdxi(k) -> stash, dmdt += dnw(k)*dvdxi(k)
//   2-D update of mu, mudf, muts, muave (+ the fused multi-GPU push of the patch's east column / north row)
//   sweep 2 (k ascending): ww prefix, ww -= ww_1, t_ave, t update with the vertical flux wdtn
#pragma once
#include <type_traits>

#include "amt_params.h"

// `stash`: this thread's first dvdxi slot in shared memory; level k lives at stash[k * stride].
// P is AmtParams (T = float) or AmtParamsR8 (T = double); the fused halo exchange exists for float only.
template <class P, class T>
__device__ __forceinline__ void amt_column_thread(const P &p, const int i, const int j,
                                                  T *stash, const int stride)
{
    const long long c2 = (long long)j * p.pitch2 + i;
    const T msftx = p.msftx[c2];
    const T msfty = p.msfty[c2];
    const T cof = f_mul(msftx, msfty);              // :142 msftx*msfty*( ... )
    const T muv_s = p.muv[c2],           muv_n = p.muv[c2 + p.pitch2];
    const T mvi_s = p.msfvx_inv[c2],     mvi_n = p.msfvx_inv[c2 + p.pitch2];
    const T muu_w = p.muu[c2],           muu_e = p.muu[c2 + 1];
    const T mfu_w = p.msfuy[c2],         mfu_e = p.msfuy[c2 + 1];
    const T mu_tend = p.mu_tend[c2];

    const long long base = (long long)j * p.jstride + (long long)p.k0 * p.pitch + i;
    const T *dnw = p.dnw + p.k0;

    // ---- sweep 1: :140-149 ----
    T dmdt = T(0);                                  // :115
#pragma unroll 4
    for (int k = 0; k < p.nk; ++k) {
        const long long o = base + (long long)k * p.pitch;
        const T vn = f_add(p.v[o + p.jstride], f_mul(f_mul(muv_n, p.v_1[o + p.jstride]), mvi_n));   // :143
        const T vs = f_add(p.v[o],             f_mul(f_mul(muv_s, p.v_1[o]), mvi_s));               // :144
        const T ue = f_add(p.u[o + 1],         f_div(f_mul(muu_e, p.u_1[o + 1]), mfu_e));           // :145
        const T uw = f_add(p.u[o],             f_div(f_mul(muu_w, p.u_1[o]), mfu_w));               // :146
        const T dv = f_mul(cof, f_add(f_mul(p.rdy, f_sub(vn, vs)), f_mul(p.rdx, f_sub(ue, uw))));
        stash[k * stride] = dv;
        dmdt = f_add(dmdt, f_mul(dnw[k], dv));          // :147
    }

    // ---- 2-D update: :151-157 ----
    const T mu_old = p.mu[c2];
    const T tend = f_add(dmdt, mu_tend);
    const T mu_new = f_add(mu_old, f_mul(p.dts, tend));                     // :153
    p.mu[c2] = mu_new;
    p.mudf[c2] = tend;                                                          // :154
    p.muts[c2] = f_add(p.mut[c2], mu_new);                                      // :155
    p.muave[c2] = f_mul(T(0.5), f_add(f_mul(f_add(T(1), p.epssm), mu_new),
                                    f_mul(f_sub(T(1), p.epssm), mu_old)));      // :156
    if constexpr (std::is_same<T, float>::value) if (p.halo.enabled) {   // fused halo exchange, as the tile kernel's scan thread
        const AmtHalo &hx = p.halo;
        if (hx.e_mudf && i == hx.ipe_mem) {
            const long long o = (long long)j * hx.e_pitch2;
            hx.e_mu[o] = mu_new; hx.e_muts[o] = f_add(p.mut[c2], mu_new); hx.e_mudf[o] = tend;
        }
        if (hx.n_mudf && j == hx.jpe_mem) {
            hx.n_mu[i] = mu_new; hx.n_muts[i] = f_add(p.mut[c2], mu_new); hx.n_mudf[i] = tend;
        }
    }

    // ---- sweep 2: ww prefix :159-172, theta :208-248, fused with a one-level look-ahead ----
    // Levels are processed in batches of kColBatch: ALL operand loads of a batch are issued first, then the
    // batch is computed and stored.  (The stores to ww / t / t_ave may alias the loads as far as the compiler
    // can tell, so a plain level loop waits out a full memory latency per level; batching keeps 12 x kColBatch
    // loads in flight per thread.)
    const T *fnm = p.fnm + p.k0, *fnp = p.fnp + p.k0, *rdnw = p.rdnw + p.k0;
    const T dts_msfty = f_mul(p.dts, msfty);        // :237 dts*msfty  (== msfty*dts of :212)
    const T hrdy = f_mul(T(0.5), p.rdy);              // :240 .5*rdy
    const T hrdx = f_mul(T(0.5), p.rdx);              // :243 .5*rdx

    T w_raw = p.ww[base];                           // ww(i,1,j): input value, never re-integrated (:159 starts at k=2)
    T w_fin = f_sub(w_raw, p.ww_1[base]);           // :170 at k=1
    T wdtn_k = T(0);                                // :220 wdtn(i,1)=0
    T t1_c = p.t_1[base];                           // t_1(i,k,j)
    constexpr int kColBatch = 4;
    for (int kb = 0; kb < p.nk; kb += kColBatch) {
        T a_t[kColBatch], a_ft[kColBatch], a_vn[kColBatch], a_t1n[kColBatch], a_vs[kColBatch], a_t1s[kColBatch];
        T a_ue[kColBatch], a_t1e[kColBatch], a_uw[kColBatch], a_t1w[kColBatch], a_ww1u[kColBatch], a_t1u[kColBatch];
#pragma unroll
        for (int q = 0; q < kColBatch; ++q) {
            const int k = kb + q;
            const long long o = base + (long long)k * p.pitch;
            const bool on = k < p.nk, up = k + 1 < p.nk;
            a_t[q] = on ? p.t[o] : T(0);                 a_ft[q] = on ? p.ft[o] : T(0);
            a_vn[q] = on ? p.v[o + p.jstride] : T(0);    a_t1n[q] = on ? p.t_1[o + p.jstride] : T(0);
            a_vs[q] = on ? p.v[o] : T(0);                a_t1s[q] = on ? p.t_1[o - p.jstride] : T(0);
            a_ue[q] = on ? p.u[o + 1] : T(0);            a_t1e[q] = on ? p.t_1[o + 1] : T(0);
            a_uw[q] = on ? p.u[o] : T(0);                a_t1w[q] = on ? p.t_1[o - 1] : T(0);
            a_ww1u[q] = up ? p.ww_1[o + p.pitch] : T(0); a_t1u[q] = up ? p.t_1[o + p.pitch] : T(0);
        }
#pragma unroll
        for (int q = 0; q < kColBatch; ++q) {
            const int k = kb + q;
            if (k < p.nk) {
                const long long o = base + (long long)k * p.pitch;
                // level k+1 of the prefix, its final value and the flux through the top face of level k
                T w_raw_n = T(0), w_fin_n = T(0), wdtn_n = T(0), t1_n = T(0);   // :221 wdtn(i,kde)=0
                if (k + 1 < p.nk) {
                    const T inner = f_add(f_add(dmdt, stash[k * stride]), mu_tend);
                    w_raw_n = f_sub(w_raw, f_div(f_mul(dnw[k], inner), msfty));     // :161
                    w_fin_n = f_sub(w_raw_n, a_ww1u[q]);                            // :170
                    t1_n = a_t1u[q];
                    wdtn_n = f_mul(w_fin_n, f_add(f_mul(fnm[k + 1], t1_n), f_mul(fnp[k + 1], t1_c)));   // :227
                }
                const T t_old = a_t[q];
                const T t_mid = f_add(t_old, f_mul(dts_msfty, a_ft[q]));        // :212
                const T fy = f_mul(hrdy, f_sub(f_mul(a_vn[q], f_add(a_t1n[q], t1_c)),
                                                   f_mul(a_vs[q], f_add(t1_c, a_t1s[q]))));             // :240-242
                const T fx = f_mul(hrdx, f_sub(f_mul(a_ue[q], f_add(a_t1e[q], t1_c)),
                                                   f_mul(a_uw[q], f_add(t1_c, a_t1w[q]))));             // :243-245
                const T fz = f_mul(rdnw[k], f_sub(wdtn_n, wdtn_k));                                  // :246
                p.ww[o] = w_fin;
                p.t_ave[o] = t_old;                                                                      // :211
                p.t[o] = f_sub(t_mid, f_mul(dts_msfty, f_add(f_mul(msftx, f_add(fy, fx)), fz)));         // :237
                w_raw = w_raw_n; w_fin = w_fin_n; wdtn_k = wdtn_n; t1_c = t1_n;
            }
        }
    }
}
