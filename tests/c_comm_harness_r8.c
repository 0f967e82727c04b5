/* tests/c_comm_harness_r8.c -- tests/c_comm_harness.c in binary64: the real*8 multi-GPU path of libwrfb200.so
 * (wrfb200_create_r8, wrfb200_comm_init_r8, wrfb200_comm_loop_r8) driven from plain C, one PROCESS per rank, as a
 * Fortran/MPI host of a WRF build configured with -r8 would.  The synthetic fields are widened to double and given
 * low mantissa bits a float cannot hold (x * (1 + 2^-40), as tests/c_abi_harness_r8.c); outputs are raw float64.
 *
 * What follows is the binary32 harness's description, with every call in its _r8 form.
 *
 * The multi-GPU path of libwrfb200.so driven from plain C, one PROCESS per rank,
 * no Python and no collective library in the loop (what a Fortran/MPI host would do with MPI_Allgather is a
 * pair of pipes here).  The parent forks PX*PY rank processes before anything touches CUDA; every rank
 *   creates its patch (global domain extents, memory = patch + halo), fills it with the counter-based
 *   synthetic fields (identical global fields under every decomposition), poisons the halos its neighbours
 *   must fill, uploads, wrfb200_comm_init -> blob to the parent -> all blobs back -> wrfb200_comm_connect
 *   (CUDA IPC), wrfb200_comm_push_constants, wrfb200_comm_loop(nsteps, stand-in advance_uv, CUDA graph),
 *   wrfb200_comm_status, downloads, and writes OUTDIR/rank<r>_<field>.bin (raw float64, memory extents).
 * tests/test_fused_comm_r8.py compares every rank's patch with the binary64 checker loop, bit for bit.
 *
 *   gcc tests/c_comm_harness_r8.c -Iinclude -Lwrf_model_cuda_sample_b200 -lwrfb200 -o /tmp/c_comm_harness_r8
 *   /tmp/c_comm_harness_r8 PX PY NX NY NZ NSTEPS NDEVICES OUTDIR
 * Replaces (as a harness) the reference's multi-GPU driver loop, advance_mu_t_no_async.cu:329-357.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/types.h>
#include <sys/wait.h>
#include <unistd.h>
#include "wrfb200.h"

#define HALO 3
#define POISON 12345.0
#define SEED 99ull

static int read_all(int fd, void *buf, size_t n)
{
    char *p = (char *)buf;
    while (n) { ssize_t r = read(fd, p, n); if (r <= 0) return -1; p += r; n -= (size_t)r; }
    return 0;
}
static int write_all(int fd, const void *buf, size_t n)
{
    const char *p = (const char *)buf;
    while (n) { ssize_t r = write(fd, p, n); if (r <= 0) return -1; p += r; n -= (size_t)r; }
    return 0;
}
/* WRF-style even split of lo..hi into `parts` chunks (parallel.split_range) */
static void split(int lo, int hi, int parts, int idx, int *a, int *b)
{
    const int n = hi - lo + 1;
    *a = lo + (int)((long long)n * idx / parts);
    *b = lo + (int)((long long)n * (idx + 1) / parts) - 1;
}

#define CHECK(call)                                                                           \
    do { int rc_ = (call); if (rc_ != WRFB200_OK) {                                           \
        fprintf(stderr, "rank %d: %s -> status %d: %s\n", rank, #call, rc_, wrfb200_last_error()); \
        return 10 + rc_; } } while (0)

static int run_rank(int rank, int px, int py, int nx, int ny, int nz, int nsteps, int ndev, const char *outdir,
                    int to_parent, int from_parent)
{
    const int pi = rank % px, pj = rank / px;
    int ips, ipe, jps, jpe;
    split(1, nx, px, pi, &ips, &ipe);
    split(1, ny, py, pj, &jps, &jpe);
    wrfb200_domain dom = {1, nx, 1, ny, nz, ips - HALO, ipe + HALO, jps - HALO, jpe + HALO, 1, nz, 0, 1, 0};
    const int idim = dom.ime - dom.ims + 1, jdim = dom.jme - dom.jms + 1, kdim = nz;
    const size_t n3 = (size_t)idim * kdim * jdim, n2 = (size_t)idim * jdim, n1 = (size_t)kdim;
    double *f[WRFB200_NUM_FIELDS];
    for (int i = 0; i < WRFB200_NUM_FIELDS; ++i) {
        const size_t n = i < WRFB200_NUM_3D ? n3 : i < WRFB200_NUM_3D + WRFB200_NUM_2D ? n2 : n1;
        float *tmp = (float *)malloc(n * sizeof(float));
        f[i] = (double *)malloc(n * sizeof(double));
        CHECK(wrfb200_synth_field(i, SEED, &dom, 3000.0f, tmp));
        for (size_t x = 0; x < n; ++x) f[i][x] = (double)tmp[x] * (1.0 + 0x1p-40);
        free(tmp);
    }
    /* poison every horizontal halo cell of the exchanged fields that has a neighbour behind it */
    const int exch[] = {WRFB200_U, WRFB200_V, WRFB200_U_1, WRFB200_V_1, WRFB200_T_1, WRFB200_MUU, WRFB200_MUV,
                        WRFB200_MSFUY, WRFB200_MSFVX_INV, WRFB200_MU, WRFB200_MUTS, WRFB200_MUDF};
    for (unsigned q = 0; q < sizeof(exch) / sizeof(exch[0]); ++q) {
        const int id = exch[q];
        const int nk = id < WRFB200_NUM_3D ? kdim : 1;
        for (int j = 0; j < jdim; ++j)
            for (int k = 0; k < nk; ++k)
                for (int i = 0; i < idim; ++i) {
                    const int gi = dom.ims + i, gj = dom.jms + j;
                    const int west = gi < ips && pi > 0, east = gi > ipe && pi + 1 < px;
                    const int south = gj < jps && pj > 0, north = gj > jpe && pj + 1 < py;
                    if (west || east || south || north) f[id][((size_t)j * nk + k) * idim + i] = POISON;
                }
    }

    wrfb200_handle *h = NULL;
    CHECK(wrfb200_create_r8(&h, &dom, rank % ndev, 1));
    CHECK(wrfb200_set_scalars_r8(h, 1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1));
    for (int i = 0; i < WRFB200_NUM_FIELDS; ++i) CHECK(wrfb200_upload_r8(h, i, f[i]));

    const int world = px * py;
    char *mine = (char *)calloc(1, WRFB200_COMM_INFO_BYTES);
    char *all = (char *)calloc((size_t)world, WRFB200_COMM_INFO_BYTES);
    CHECK(wrfb200_comm_init_r8(h, px, py, rank, ips, ipe, jps, jpe, mine));
    if (write_all(to_parent, mine, WRFB200_COMM_INFO_BYTES) || read_all(from_parent, all, (size_t)world * WRFB200_COMM_INFO_BYTES)) {
        fprintf(stderr, "rank %d: blob exchange failed\n", rank);
        return 3;
    }
    CHECK(wrfb200_comm_connect(h, all, world));
    CHECK(wrfb200_comm_push_constants(h));
    CHECK(wrfb200_comm_loop_r8(h, nsteps, 1, 0.25, 1));
    int timeouts = 0;
    long steps = 0;
    CHECK(wrfb200_comm_status(h, &timeouts, &steps));
    if (timeouts != 0 || steps != nsteps) {
        fprintf(stderr, "rank %d: %d halo waits timed out, %ld of %d steps\n", rank, timeouts, steps, nsteps);
        return 4;
    }
    const int outs[] = {WRFB200_WW, WRFB200_T, WRFB200_T_AVE, WRFB200_MU, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUDF,
                        WRFB200_U, WRFB200_V};
    for (unsigned q = 0; q < sizeof(outs) / sizeof(outs[0]); ++q) CHECK(wrfb200_download_r8(h, outs[q], f[outs[q]]));
    CHECK(wrfb200_sync(h));
    for (unsigned q = 0; q < sizeof(outs) / sizeof(outs[0]); ++q) {
        char path[1024];
        snprintf(path, sizeof(path), "%s/rank%d_field%d.bin", outdir, rank, outs[q]);
        FILE *fp = fopen(path, "wb");
        const size_t n = outs[q] < WRFB200_NUM_3D ? n3 : n2;
        if (!fp || fwrite(f[outs[q]], sizeof(double), n, fp) != n) { fprintf(stderr, "rank %d: cannot write %s\n", rank, path); return 5; }
        fclose(fp);
    }
    /* nobody unmaps a neighbour that may still be storing into it: second rendezvous through the parent */
    char token = 1;
    if (write_all(to_parent, &token, 1) || read_all(from_parent, &token, 1)) return 6;
    CHECK(wrfb200_destroy(h));
    printf("rank %d ok: patch i=%d..%d j=%d..%d, %ld steps\n", rank, ips, ipe, jps, jpe, steps);
    return 0;
}

int main(int argc, char **argv)
{
    if (argc != 9) {
        fprintf(stderr, "usage: %s PX PY NX NY NZ NSTEPS NDEVICES OUTDIR\n", argv[0]);
        return 2;
    }
    const int px = atoi(argv[1]), py = atoi(argv[2]), nx = atoi(argv[3]), ny = atoi(argv[4]), nz = atoi(argv[5]);
    const int nsteps = atoi(argv[6]), ndev = atoi(argv[7]) > 0 ? atoi(argv[7]) : 1;
    const int world = px * py;
    if (world < 1 || world > 64) return 2;
    int up[64][2], down[64][2];
    pid_t pid[64];
    for (int r = 0; r < world; ++r) {
        if (pipe(up[r]) || pipe(down[r])) { perror("pipe"); return 2; }
        pid[r] = fork();
        if (pid[r] < 0) { perror("fork"); return 2; }
        if (pid[r] == 0) {                                   /* rank process: CUDA is first touched here */
            close(up[r][0]); close(down[r][1]);
            const int rc = run_rank(r, px, py, nx, ny, nz, nsteps, ndev, argv[8], up[r][1], down[r][0]);
            fflush(stdout); fflush(stderr);
            _exit(rc);
        }
        close(up[r][1]); close(down[r][0]);
    }
    /* the parent is the all-gather and the final barrier; it never touches CUDA */
    char *all = (char *)calloc((size_t)world, WRFB200_COMM_INFO_BYTES);
    int ok = 1;
    for (int r = 0; r < world && ok; ++r) ok = read_all(up[r][0], all + (size_t)r * WRFB200_COMM_INFO_BYTES, WRFB200_COMM_INFO_BYTES) == 0;
    for (int r = 0; r < world && ok; ++r) ok = write_all(down[r][1], all, (size_t)world * WRFB200_COMM_INFO_BYTES) == 0;
    char token;
    for (int r = 0; r < world && ok; ++r) ok = read_all(up[r][0], &token, 1) == 0;
    for (int r = 0; r < world; ++r) { token = 1; (void)write_all(down[r][1], &token, 1); close(down[r][1]); }
    int worst = ok ? 0 : 1;
    for (int r = 0; r < world; ++r) {
        int st = 0;
        waitpid(pid[r], &st, 0);
        const int rc = WIFEXITED(st) ? WEXITSTATUS(st) : 99;
        if (rc != 0) { fprintf(stderr, "rank %d exited with %d\n", r, rc); worst = rc; }
    }
    return worst;
}
