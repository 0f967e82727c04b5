/* tests/c_abi_harness_r8.c -- calls wrfb200_advance_mu_t_r8 the way the Fortran shim does when WRF is built
 * with -r8 (module_small_step_em.F90 resolves its generic interface to the REAL(c_double) body): double
 * arrays by reference in the Fortran order, double scalars by value, Fortran-numbered indices.
 *
 *   gcc tests/c_abi_harness_r8.c -Iinclude -Lwrf_model_cuda_sample_b200 -lwrfb200 -o /tmp/c_abi_harness_r8
 *   /tmp/c_abi_harness_r8         -> prints a checksum of every output field (needs a GPU), or, without a
 *                                    GPU, the library's "no CPU fallback" error and exit code 3.
 */
#include <stdio.h>
#include <stdlib.h>
#include "wrfb200.h"

int main(void)
{
    const int ids = 1, ide = 40, jds = 1, jde = 30, kde = 12;
    const int ims = -2, ime = 43, jms = -2, jme = 33, kms = 1, kme = 12;
    wrfb200_domain dom = {ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme, 0, 1, 0};
    const size_t n3 = (size_t)(ime - ims + 1) * (kme - kms + 1) * (jme - jms + 1);
    const size_t n2 = (size_t)(ime - ims + 1) * (jme - jms + 1);
    const size_t n1 = (size_t)(kme - kms + 1);
    double *f[WRFB200_NUM_FIELDS];
    for (int i = 0; i < WRFB200_NUM_FIELDS; ++i) {
        size_t n = i < WRFB200_NUM_3D ? n3 : i < WRFB200_NUM_3D + WRFB200_NUM_2D ? n2 : n1;
        float *tmp = (float *)malloc(n * sizeof(float));
        f[i] = (double *)malloc(n * sizeof(double));
        if (wrfb200_synth_field(i, 20240617ull, &dom, 12000.0f, tmp) != WRFB200_OK) {
            fprintf(stderr, "synth: %s\n", wrfb200_last_error());
            return 2;
        }
        /* widen, and fill low mantissa bits a float cannot hold */
        for (size_t x = 0; x < n; ++x) f[i][x] = (double)tmp[x] * (1.0 + 0x1p-40);
        free(tmp);
    }
    int rc = wrfb200_advance_mu_t_r8(
        f[WRFB200_WW], f[WRFB200_WW_1], f[WRFB200_U], f[WRFB200_U_1], f[WRFB200_V], f[WRFB200_V_1],
        f[WRFB200_MU], f[WRFB200_MUT], f[WRFB200_MUAVE], f[WRFB200_MUTS], f[WRFB200_MUU], f[WRFB200_MUV],
        f[WRFB200_MUDF], f[WRFB200_T], f[WRFB200_T_1], f[WRFB200_T_AVE], f[WRFB200_FT], f[WRFB200_MU_TEND],
        1.0 / 12000.0, 1.0 / 12000.0, 12.0, 0.1,
        f[WRFB200_DNW], f[WRFB200_FNM], f[WRFB200_FNP], f[WRFB200_RDNW],
        f[WRFB200_MSFUY], f[WRFB200_MSFVX_INV], f[WRFB200_MSFTX], f[WRFB200_MSFTY],
        0, 1, 0, ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme,
        ids, ide, jds, jde, 1, kde);
    if (rc != WRFB200_OK) {
        fprintf(stderr, "wrfb200_advance_mu_t_r8: status %d: %s\n", rc, wrfb200_last_error());
        return rc;
    }
    const int outs[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE, WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF};
    for (unsigned q = 0; q < sizeof(outs) / sizeof(outs[0]); ++q) {
        const size_t n = outs[q] < WRFB200_NUM_3D ? n3 : n2;
        unsigned long long h = 1469598103934665603ull;           /* FNV-1a over the raw bytes */
        const unsigned char *b = (const unsigned char *)f[outs[q]];
        for (size_t x = 0; x < n * 8; ++x) { h ^= b[x]; h *= 1099511628211ull; }
        printf("field %d fnv1a %016llx\n", outs[q], h);
    }
    return 0;
}
