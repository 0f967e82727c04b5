// host_utils.cu -- host-side harness utilities of the C ABI (no device code):
//   * wrfb200_synth_field : deterministic atmosphere-like input fields (SURVEY.md section 8d).  The reference
//     reads its inputs from /data2/WRFV3_Input_Output/V3.4.1/dyn_em/advance_mu_t/*.bin
//     (advance_mu_t_driver.f90:36-167), which are not shipped; these fields have the same roles and magnitudes.
//   * wrfb200_compare     : the reference's error report, /root/reference/common.cu:68-164 (metric set only;
//     the reference prints and has no pass/fail threshold); wrfb200_compare_r8 is the same over doubles.
#include <cmath>
#include <cstdint>
#include <climits>
#include <cstring>
#include <thread>
#include <vector>

#include "capi_internal.h"

namespace {

inline uint64_t mix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// Counter-based uniform in [0,1): a pure function of (seed, field, global i, k, j).
inline float unit(uint64_t seed, int field, int gi, int gk, int gj)
{
    uint64_t key = mix64(seed ^ mix64((uint64_t)field + 0x51ED27ull));
    key = mix64(key ^ ((uint64_t)(uint32_t)gi | ((uint64_t)(uint32_t)gj << 32)));
    key = mix64(key ^ (uint64_t)(uint32_t)gk);
    return (float)(key >> 40) * (1.0f / 16777216.0f);
}
inline float sym(uint64_t seed, int field, int gi, int gk, int gj) { return 2.0f * unit(seed, field, gi, gk, gj) - 1.0f; }

constexpr double kTwoPi = 6.283185307179586;

struct Norm {
    double x, y;
};
inline Norm norm_xy(const wrfb200_domain &d, int gi, int gj)
{
    const double nx = d.ide > d.ids ? (double)(d.ide - d.ids) : 1.0;
    const double ny = d.jde > d.jds ? (double)(d.jde - d.jds) : 1.0;
    return {(double)(gi - d.ids) / nx, (double)(gj - d.jds) / ny};
}

inline float mut_at(const wrfb200_domain &d, int gi, int gj)
{
    const Norm n = norm_xy(d, gi, gj);
    return (float)(94000.0 + 3000.0 * std::sin(kTwoPi * 2.0 * n.x) * std::cos(kTwoPi * 1.5 * n.y)
                   + 800.0 * std::sin(kTwoPi * 7.0 * n.x + 1.0) * std::sin(kTwoPi * 5.0 * n.y));
}

float value2d(int field, uint64_t seed, const wrfb200_domain &d, int gi, int gj)
{
    const Norm n = norm_xy(d, gi, gj);
    switch (field) {
    case WRFB200_MUT: return mut_at(d, gi, gj);
    case WRFB200_MUU: return 0.5f * (mut_at(d, gi, gj) + mut_at(d, gi - 1, gj));
    case WRFB200_MUV: return 0.5f * (mut_at(d, gi, gj) + mut_at(d, gi, gj - 1));
    case WRFB200_MU: return 300.0f * sym(seed, field, gi, 0, gj);
    case WRFB200_MU_TEND: return 0.5f * sym(seed, field, gi, 0, gj);
    case WRFB200_MSFTX: return (float)(1.0 + 0.1 * std::sin(kTwoPi * n.y) * std::cos(0.5 * kTwoPi * n.x));
    case WRFB200_MSFTY: return (float)(1.0 + 0.1 * std::cos(kTwoPi * 0.7 * n.y + 0.3));
    case WRFB200_MSFUY: return (float)(1.0 + 0.1 * std::cos(kTwoPi * 0.7 * n.y + 0.3) + 0.01 * std::sin(kTwoPi * 3.0 * n.x));
    case WRFB200_MSFVX_INV: return (float)(1.0 / (1.0 + 0.1 * std::sin(kTwoPi * n.y - 0.2) * std::cos(0.5 * kTwoPi * n.x)));
    // INTENT(OUT) fields: recognisable garbage, so tests can prove cells outside the computed range stay untouched
    case WRFB200_MUAVE: return 1000.0f + 100.0f * sym(seed, field, gi, 0, gj);
    case WRFB200_MUTS: return 2000.0f + 100.0f * sym(seed, field, gi, 0, gj);
    case WRFB200_MUDF: return 3000.0f + 100.0f * sym(seed, field, gi, 0, gj);
    default: return 0.0f;
    }
}

float value3d(int field, uint64_t seed, const wrfb200_domain &d, int gi, int gk, int gj)
{
    const Norm n = norm_xy(d, gi, gj);
    const double z = d.kde > 1 ? (double)(gk - 1) / (double)(d.kde - 1) : 0.0;
    const float r = sym(seed, field, gi, gk, gj);
    switch (field) {
    case WRFB200_U_1: return (float)(10.0 + 20.0 * z * std::sin(kTwoPi * (n.x + n.y))) + 2.0f * r;
    case WRFB200_V_1: return (float)(-5.0 + 20.0 * z * std::cos(kTwoPi * (n.x - n.y))) + 2.0f * r;
    case WRFB200_U: return (float)(500.0 * std::sin(kTwoPi * 3.0 * n.x) * std::cos(kTwoPi * 2.0 * n.y)) + 1500.0f * r;
    case WRFB200_V: return (float)(500.0 * std::cos(kTwoPi * 2.0 * n.x) * std::sin(kTwoPi * 3.0 * n.y)) + 1500.0f * r;
    case WRFB200_T_1: return (float)(150.0 * z) + 2.0f * r;
    case WRFB200_T: return 50.0f * r;
    case WRFB200_FT: return 5.0f * r;
    case WRFB200_WW_1: return gk <= 1 ? 0.0f : 0.5f * r;
    case WRFB200_WW: return (gk <= 1 || gk >= d.kde) ? 0.0f : 0.5f * r;
    case WRFB200_T_AVE: return 4000.0f + 100.0f * r;      // INTENT(INOUT) but write-only: recognisable garbage
    default: return 0.0f;
    }
}

// Stretched eta levels: znw(1)=1 ... znw(kde)=0, finer near the surface.
inline double znw_at(const wrfb200_domain &d, int k)
{
    const double s = d.kde > 1 ? (double)(k - 1) / (double)(d.kde - 1) : 0.0;
    const double a = 2.5;
    return (std::exp(-a * s) - std::exp(-a)) / (1.0 - std::exp(-a));
}
inline float dnw_at(const wrfb200_domain &d, int k)
{
    int kk = k < 1 ? 1 : (k > d.kde - 1 ? d.kde - 1 : k);
    if (kk < 1) kk = 1;
    return (float)(znw_at(d, kk + 1) - znw_at(d, kk));
}

float value1d(int field, const wrfb200_domain &d, int k)
{
    if (k < 1 || k > d.kde) return 0.0f;
    const float dnw = dnw_at(d, k);
    switch (field) {
    case WRFB200_DNW: return dnw;
    case WRFB200_RDNW: return 1.0f / dnw;
    case WRFB200_FNM:
    case WRFB200_FNP: {
        if (k < 2) return 0.0f;
        const float dnwm = dnw_at(d, k - 1);
        const float dn = 0.5f * (dnw + dnwm);
        return field == WRFB200_FNP ? 0.5f * dnwm / dn : 0.5f * dnw / dn;
    }
    default: return 0.0f;
    }
}

template <class F>
void parallel_rows(int n, F fn)
{
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (nt > 64) nt = 64;
    if ((int)nt > n) nt = (unsigned)(n > 0 ? n : 1);
    if (nt <= 1) { for (int r = 0; r < n; ++r) fn(r); return; }
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; ++t)
        th.emplace_back([=]() { for (int r = (int)t; r < n; r += (int)nt) fn(r); });
    for (auto &x : th) x.join();
}

inline long ulp_distance(float a, float b)
{
    // sign-magnitude -> lexicographically ordered two's-complement integer, as common.cu:51-66
    // (there `0x80000000 - aint` in 32-bit arithmetic is minus the magnitude); 64-bit here so the
    // difference cannot overflow.
    uint32_t ai, bi;
    std::memcpy(&ai, &a, 4);
    std::memcpy(&bi, &b, 4);
    const int64_t al = (ai & 0x80000000u) ? -(int64_t)(ai & 0x7fffffffu) : (int64_t)ai;
    const int64_t bl = (bi & 0x80000000u) ? -(int64_t)(bi & 0x7fffffffu) : (int64_t)bi;
    const int64_t dlt = al - bl;
    return (long)(dlt < 0 ? -dlt : dlt);
}

inline long ulp_distance(double a, double b)
{
    // the same over the 64-bit patterns: distance of the magnitudes on one side of zero, their sum across it;
    // only opposite-signed values near the infinities exceed LONG_MAX, and saturate there
    uint64_t ai, bi;
    std::memcpy(&ai, &a, 8);
    std::memcpy(&bi, &b, 8);
    const uint64_t sign = 0x8000000000000000ull, am = ai & ~sign, bm = bi & ~sign;
    const uint64_t d = ((ai ^ bi) & sign) ? am + bm : (am > bm ? am - bm : bm - am);
    return d > (uint64_t)LONG_MAX ? LONG_MAX : (long)d;
}

// wrfb200_compare / _compare_r8: T is the element type, R the result struct of that precision
template <class T, class R>
int compare_values(const T *a, const T *b, long n, R *out)
{
    if (!a || !b || !out || n < 0) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "bad argument");
    R r{};
    r.n = n;
    double sq = 0.0;
    for (long x = 0; x < n; ++x) {
        const T va = a[x], vb = b[x];
        if (std::isnan(va) || std::isnan(vb))
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "NaN at element %ld (a=%g b=%g)", x, (double)va, (double)vb);
        const T abs_err = std::fabs(va - vb);
        T rel;
        if (std::fabs(va) != (T)0 && std::fabs(vb) != (T)0)
            rel = abs_err / std::fmax(std::fabs(va), std::fabs(vb));
        else
            rel = std::fmax(std::fabs(va), std::fabs(vb));
        if (rel > r.max_rel) r.max_rel = rel;
        if (abs_err > r.max_abs) r.max_abs = abs_err;
        const long ulp = ulp_distance(va, vb);
        if (ulp > r.max_ulp) r.max_ulp = ulp;
        sq += (double)abs_err * (double)abs_err;
        if (va == vb) r.n_equal++; else r.n_different++;
    }
    r.rmse = n > 0 ? (T)std::sqrt(sq / (double)n) : (T)0;
    *out = r;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_synth_field(int field, uint64_t seed, const wrfb200_domain *dom, float dx_m, float *out)
{
    (void)dx_m;   // magnitudes are grid-spacing independent; rdx/rdy/dts are set by the caller
    if (!dom || !out) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (field < 0 || field >= WRFB200_NUM_FIELDS) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "bad field id %d", field);
    const wrfb200_domain d = *dom;
    const int ni = d.ime - d.ims + 1, nj = d.jme - d.jms + 1, nk = d.kme - d.kms + 1;
    if (ni <= 0 || nj <= 0 || nk <= 0) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "empty memory extents");
    if (field >= WRFB200_DNW) {
        for (int k = 0; k < nk; ++k) out[k] = value1d(field, d, d.kms + k);
        return WRFB200_OK;
    }
    if (field >= WRFB200_MU) {
        parallel_rows(nj, [&](int j) {
            float *row = out + (size_t)j * ni;
            for (int i = 0; i < ni; ++i) row[i] = value2d(field, seed, d, d.ims + i, d.jms + j);
        });
        return WRFB200_OK;
    }
    parallel_rows(nj, [&](int j) {
        for (int k = 0; k < nk; ++k) {
            float *row = out + ((size_t)j * nk + k) * ni;
            for (int i = 0; i < ni; ++i) row[i] = value3d(field, seed, d, d.ims + i, d.kms + k, d.jms + j);
        }
    });
    return WRFB200_OK;
}

extern "C" int wrfb200_compare(const float *a, const float *b, long n, wrfb200_compare_result *out)
{
    return compare_values(a, b, n, out);
}

extern "C" int wrfb200_compare_r8(const double *a, const double *b, long n, wrfb200_compare_result_r8 *out)
{
    return compare_values(a, b, n, out);
}
