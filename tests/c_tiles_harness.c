/* tests/c_tiles_harness.c -- the host-array call as a WRF OpenMP build makes it: the patch cut into 2 x 2 tiles
 * (ragged), one 48-argument wrfb200_advance_mu_t call per tile from four threads whose current device is the default
 * one, a 6-step acoustic loop bracketed by wrfb200_acoustic_loop_begin / _end on the main thread, and the stand-in
 * advance_uv (include/wrfb200.h section 3) applied to the host u, v by the main thread between steps, while the
 * workers wait.  Tiles rotate between the threads every step, as schedule(dynamic) may do.  Shared-tiles mode is
 * enabled once on the main thread.
 *
 *   gcc -ffp-contract=off tests/c_tiles_harness.c -Iinclude -Lwrf_model_cuda_sample_b200 -lwrfb200 -lpthread
 *   ./a.out OUTDIR      -> OUTDIR/field<id>.bin for the seven outputs and u, v (needs a GPU); without a GPU the
 *                          library's "no CPU fallback" error and exit code 3.
 */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "wrfb200.h"

#define NX 150
#define NY 110
#define NZ 16
#define HALO 5
#define NTHREADS 4
#define NSTEPS 6

static const int ids = 1, ide = NX, jds = 1, jde = NY, kde = NZ;
static const int ims = 1 - HALO, ime = NX + HALO, jms = 1 - HALO, jme = NY + HALO, kms = 1, kme = NZ;
static const int tiles[NTHREADS][4] = {{1, 61, 1, 47}, {62, NX, 1, 47}, {1, 61, 48, NY}, {62, NX, 48, NY}};
static const float rdx = 1.0f / 3000.0f, rdy = 1.0f / 3000.0f, dts = 3.0f, epssm = 0.1f, c_uv = 0.25f;

static float *f[WRFB200_NUM_FIELDS];
static pthread_barrier_t barrier;
static int status[NTHREADS];
static char message[NTHREADS][512];

static int call_tile(const int *t)
{
    return wrfb200_advance_mu_t(
        f[WRFB200_WW], f[WRFB200_WW_1], f[WRFB200_U], f[WRFB200_U_1], f[WRFB200_V], f[WRFB200_V_1],
        f[WRFB200_MU], f[WRFB200_MUT], f[WRFB200_MUAVE], f[WRFB200_MUTS], f[WRFB200_MUU], f[WRFB200_MUV],
        f[WRFB200_MUDF], f[WRFB200_T], f[WRFB200_T_1], f[WRFB200_T_AVE], f[WRFB200_FT], f[WRFB200_MU_TEND],
        rdx, rdy, dts, epssm,
        f[WRFB200_DNW], f[WRFB200_FNM], f[WRFB200_FNP], f[WRFB200_RDNW],
        f[WRFB200_MSFUY], f[WRFB200_MSFVX_INV], f[WRFB200_MSFTX], f[WRFB200_MSFTY],
        0, 1, 0, ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme,
        t[0], t[1], t[2], t[3], 1, kde);
}

static void *worker(void *arg)
{
    const int me = (int)(size_t)arg;
    for (int step = 0; step < NSTEPS; ++step) {
        pthread_barrier_wait(&barrier);                               /* the main thread's stand-in is done */
        const int rc = call_tile(tiles[(me + step) % NTHREADS]);
        if (rc != WRFB200_OK && status[me] == WRFB200_OK) {
            status[me] = rc;
            snprintf(message[me], sizeof(message[me]), "%s", wrfb200_last_error());
        }
        pthread_barrier_wait(&barrier);                               /* every tile of this step is done */
    }
    return NULL;
}

#define AT3(i, k, j) ((size_t)((j) - jms) * (kme - kms + 1) * (ime - ims + 1) + (size_t)((k) - kms) * (ime - ims + 1) + (size_t)((i) - ims))
#define AT2(i, j) ((size_t)((j) - jms) * (ime - ims + 1) + (size_t)((i) - ims))

/* u += c*(mudf(i)-mudf(i-1)) and v += c*(mudf(j)-mudf(j-1)) over the global update boxes, every memory level */
static void standin_advance_uv(void)
{
    int is, ie, js, je, ks, ke;
    wrfb200_bounds(0, 1, 0, ids, ide, jds, jde, ids, ide, jds, jde, 1, kde, &is, &ie, &js, &je, &ks, &ke);
    float *u = f[WRFB200_U], *v = f[WRFB200_V];
    const float *mudf = f[WRFB200_MUDF];
    for (int j = js; j <= je; ++j)
        for (int i = is + 1; i <= ie; ++i) {
            const float du = c_uv * (mudf[AT2(i, j)] - mudf[AT2(i - 1, j)]);
            for (int k = kms; k <= kme; ++k) u[AT3(i, k, j)] = u[AT3(i, k, j)] + du;
        }
    for (int j = js + 1; j <= je; ++j)
        for (int i = is; i <= ie; ++i) {
            const float dv = c_uv * (mudf[AT2(i, j)] - mudf[AT2(i, j - 1)]);
            for (int k = kms; k <= kme; ++k) v[AT3(i, k, j)] = v[AT3(i, k, j)] + dv;
        }
}

int main(int argc, char **argv)
{
    if (argc != 2) {
        fprintf(stderr, "usage: %s OUTDIR\n", argv[0]);
        return 2;
    }
    wrfb200_domain dom = {ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme, 0, 1, 0};
    const size_t n3 = (size_t)(ime - ims + 1) * (kme - kms + 1) * (jme - jms + 1);
    const size_t n2 = (size_t)(ime - ims + 1) * (jme - jms + 1);
    const size_t n1 = (size_t)(kme - kms + 1);
    for (int i = 0; i < WRFB200_NUM_FIELDS; ++i) {
        const size_t n = i < WRFB200_NUM_3D ? n3 : i < WRFB200_NUM_3D + WRFB200_NUM_2D ? n2 : n1;
        f[i] = (float *)malloc(n * sizeof(float));
        if (wrfb200_synth_field(i, 99ull, &dom, 3000.0f, f[i]) != WRFB200_OK) {
            fprintf(stderr, "synth: %s\n", wrfb200_last_error());
            return 2;
        }
    }
    int rc = wrfb200_set_shared_tiles(1);
    if (rc != WRFB200_OK) {
        fprintf(stderr, "wrfb200_set_shared_tiles: status %d: %s\n", rc, wrfb200_last_error());
        return rc;
    }
    pthread_barrier_init(&barrier, NULL, NTHREADS + 1);
    pthread_t th[NTHREADS];
    for (int t = 0; t < NTHREADS; ++t) pthread_create(&th[t], NULL, worker, (void *)(size_t)t);
    wrfb200_acoustic_loop_begin();
    for (int step = 0; step < NSTEPS; ++step) {
        pthread_barrier_wait(&barrier);
        pthread_barrier_wait(&barrier);
        if (step + 1 < NSTEPS) standin_advance_uv();
    }
    wrfb200_acoustic_loop_end();
    for (int t = 0; t < NTHREADS; ++t) pthread_join(th[t], NULL);
    pthread_barrier_destroy(&barrier);
    for (int t = 0; t < NTHREADS; ++t)
        if (status[t] != WRFB200_OK) {
            fprintf(stderr, "thread %d: status %d: %s\n", t, status[t], message[t]);
            return status[t];
        }
    wrfb200_set_shared_tiles(0);

    const int outs[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE, WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF,
                        WRFB200_U, WRFB200_V};
    for (unsigned q = 0; q < sizeof(outs) / sizeof(outs[0]); ++q) {
        char path[4096];
        snprintf(path, sizeof(path), "%s/field%d.bin", argv[1], outs[q]);
        FILE *fp = fopen(path, "wb");
        if (!fp) { perror(path); return 2; }
        const size_t n = outs[q] < WRFB200_NUM_3D ? n3 : n2;
        if (fwrite(f[outs[q]], sizeof(float), n, fp) != n) { perror(path); fclose(fp); return 2; }
        fclose(fp);
    }
    return 0;
}
