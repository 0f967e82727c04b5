/*
 * wrfb200.h -- C ABI of the B200-native `advance_mu_t` (WRF acoustic small step).
 *
 * This is the drop-in boundary: plain pointers, ints and floats, no C++ or torch
 * types.  Everything is exported from libwrfb200.so (built from
 * wrf_model_cuda_sample_b200/csrc/ by __graft_entry__.build()).
 *
 * What each entry point replaces in the reference (lydia-schiff/wrf-model-cuda-sample):
 *
 *   wrfb200_advance_mu_t            the operator itself:
 *                                     Fortran  module_small_step_em.f90:7-18   (48 dummy arguments)
 *                                     C        advance_mu_t.h:10-23
 *                                     CUDA     advance_mu_t_cu.h:3-17 / advance_mu_t_no_async.cu:35-48
 *   wrfb200_create/destroy/upload/
 *   download/step/...               the CUDA host layer advance_mu_t_no_async.cu:35-424
 *                                   (per-call cudaMalloc :178-244, H2D :245-306, launch :329-353,
 *                                   sync :354-357, D2H :366-390, free :392-423), split so that state
 *                                   stays device-resident across the acoustic sub-steps
 *   wrfb200_pack_halo/unpack_halo   the host re-upload of overlapping j-slabs that stands in for a halo
 *                                   exchange, advance_mu_t_no_async.cu:87-162, :276-298
 *   wrfb200_compare                 the error report of common.cu:68-164 (`compare`), same metric set
 *   wrfb200_last_error              HANDLE_ERROR's print+exit, advance_mu_t_no_async.cu:22-32
 *                                   (a library never calls exit(); it returns a status)
 *
 * Conventions
 *   - All grid indices are Fortran-numbered and inclusive, exactly as the Fortran subroutine receives
 *     them (ids..kte).  There is no `kds` argument (the Fortran has none; in the C translation it cancels,
 *     advance_mu_t.c:38,45,52).
 *   - 3-D fields are (ims:ime, kms:kme, jms:jme) with i fastest, then k, then j
 *     (module_small_step_em.f90:30-44); 2-D fields are (ims:ime, jms:jme) (:46-59); 1-D are (kms:kme) (:61-64).
 *   - Preconditions taken from the reference code itself: kts == 1 and kms <= 1 (literal k=1 / k=2 loops,
 *     module_small_step_em.f90:159,168,209,220,224,234), kde == kte (scratch indexed at kde, :221),
 *     and a one-cell ring of memory around the computed range (ims <= i_start-1, ime >= i_end+1, same in j).
 *   - Every function returns a wrfb200_status (0 = ok).  After a non-zero status,
 *     wrfb200_last_error() gives a human-readable message (thread-local).
 *   - No CPU fallback exists: without a CUDA device every compute entry point fails with WRFB200_ERR_CUDA.
 *   - Precision: the unsuffixed entry points take binary32 (`float`, WRF's default REAL = 4 bytes).  WRF built
 *     with -r8 (REAL = 8 bytes) calls the `_r8` entry points, which take `double` and compute every operation
 *     in binary64, in the same order.  A handle holds one precision, fixed by wrfb200_create / _create_r8;
 *     a verb typed for the other precision fails with WRFB200_ERR_STATE.  The multi-GPU, halo pack / unpack,
 *     stand-in and resident-bundle verbs have `_r8` twins (wrfb200_pack_halo_r8, ..., section 3;
 *     wrfb200_comm_init_r8, ..., section 3b); their binary32 forms return WRFB200_ERR_UNSUPPORTED on an r8 handle.
 *     wrfb200_compare_r8 is the error report over doubles.
 */
#ifndef WRFB200_H
#define WRFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WRFB200_VERSION 100

typedef enum wrfb200_status {
    WRFB200_OK = 0,
    WRFB200_ERR_INVALID_ARG = 1,   /* bad pointer / index set / field id */
    WRFB200_ERR_UNSUPPORTED = 2,   /* violates a precondition listed above */
    WRFB200_ERR_CUDA = 3,          /* CUDA runtime error (message has the detail) */
    WRFB200_ERR_NOMEM = 4,
    WRFB200_ERR_STATE = 5          /* e.g. step before upload, field not bound */
} wrfb200_status;

/* Field ids, in the order of the Fortran argument list within each rank. */
typedef enum wrfb200_field {
    /* 3-D (i,k,j) */
    WRFB200_WW = 0, WRFB200_WW_1, WRFB200_U, WRFB200_U_1, WRFB200_V, WRFB200_V_1,
    WRFB200_T, WRFB200_T_1, WRFB200_T_AVE, WRFB200_FT,
    /* 2-D (i,j) */
    WRFB200_MU, WRFB200_MUT, WRFB200_MUAVE, WRFB200_MUTS, WRFB200_MUU, WRFB200_MUV,
    WRFB200_MUDF, WRFB200_MU_TEND, WRFB200_MSFUY, WRFB200_MSFVX_INV, WRFB200_MSFTX, WRFB200_MSFTY,
    /* 1-D (k) */
    WRFB200_DNW, WRFB200_FNM, WRFB200_FNP, WRFB200_RDNW,
    WRFB200_NUM_FIELDS
} wrfb200_field;
#define WRFB200_NUM_3D 10
#define WRFB200_NUM_2D 12
#define WRFB200_NUM_1D 4

/* Domain / memory description of one patch (one rank).  d = domain (global), m = memory (patch + halo). */
typedef struct wrfb200_domain {
    int ids, ide, jds, jde, kde;
    int ims, ime, jms, jme, kms, kme;
    int periodic_x, specified, nested;   /* the three grid_config_rec_type members the routine reads,
                                            module_configure.f90:434,436,447 */
} wrfb200_domain;

/* Kernel selection (testing / benchmarking; AUTO is the product default).
 *
 * Level limits.  Each kernel holds all nk = kte-kts computed levels of its columns in shared memory, so nk bounds
 * which kernels can run:
 *                 binary32        real*8
 *   PIPE          nk <= 337       --
 *   TILE          nk <= 223       nk <= 220
 *   COLUMN        nk <= 454       nk <= 227
 * AUTO runs the pipe kernel (binary32) / tile kernel (real*8) where the layout and nk allow it, otherwise the column
 * kernel: binary32 nk 338 .. 454 and real*8 nk 221 .. 227 always run the column kernel.  A request past a kernel's
 * limit -- explicit, or AUTO past the column kernel's -- fails with WRFB200_ERR_UNSUPPORTED before anything is
 * launched, and the message quotes nk and the limit.  The multi-GPU path (section 3b) runs the pipe kernel for
 * binary32 and the tile kernel for real*8: wrfb200_comm_init / _init_r8 refuse a larger nk. */
typedef enum wrfb200_kernel {
    WRFB200_KERNEL_AUTO = 0,
    WRFB200_KERNEL_COLUMN = 1,   /* one thread per (i,j) column, any layout */
    WRFB200_KERNEL_TILE = 2,     /* k-parallel float4 tile kernel (register staged), needs 16-byte aligned rows;
                                    on an r8 handle the double2 tile kernel (the AUTO choice there), which needs
                                    16-byte aligned fields, pitches of an even number of doubles and nk <= 220 */
    WRFB200_KERNEL_PIPE = 3      /* tile kernel with per-warp TMA bulk-copy pipelines (the AUTO choice when the
                                    layout allows it); binary32 only */
} wrfb200_kernel;

/* Halo sides of a patch. */
typedef enum wrfb200_side { WRFB200_WEST = 0, WRFB200_EAST = 1, WRFB200_SOUTH = 2, WRFB200_NORTH = 3 } wrfb200_side;

/* What a wrfb200_advance_mu_t call did with the calling thread's cache (wrfb200_default_last_cache). */
typedef enum wrfb200_cache {
    WRFB200_CACHE_REUSED = 0,   /* the device state of its domain (or its device-pointer wrapper) was already there */
    WRFB200_CACHE_CREATED = 1,  /* it was created */
    WRFB200_CACHE_EVICTED = 2   /* it was created after the least recently used domain(s) had been freed */
} wrfb200_cache;

typedef struct wrfb200_handle wrfb200_handle;

/* ------------------------------------------------------------------------------------------------
 * 1. The operator, with the reference Fortran subroutine's argument list
 *    (module_small_step_em.f90:7-18; config_flags expanded to its three used members).
 *
 *    Pointers may be HOST pointers (compat mode: upload -> step -> download of the written ranges ->
 *    sync; device mirrors are cached per thread and precision, one set per domain -- device and memory
 *    extents -- for up to 8 domains, and re-used by later calls of that domain) or DEVICE pointers
 *    (launched in place on the current wrfb200 stream, returns without host sync).
 *    All array pointers of one call must be of the same kind.  Writes exactly the cells the Fortran
 *    writes: ww,t,t_ave for k<=kte-1 and mu,muave,muts,mudf, inside i_start..i_end x j_start..j_end only.
 * ---------------------------------------------------------------------------------------------- */
int wrfb200_advance_mu_t(
    float *ww, const float *ww_1, const float *u, const float *u_1, const float *v, const float *v_1,
    float *mu, const float *mut, float *muave, float *muts, const float *muu, const float *muv,
    float *mudf, float *t, const float *t_1, float *t_ave, const float *ft, const float *mu_tend,
    float rdx, float rdy, float dts, float epssm,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte);

/* Same call applied `nsteps` times back to back on device-resident state (the acoustic loop of one
 * RK3 sub-step with u,v held fixed): one upload, nsteps launches, one download.  Host pointers only. */
int wrfb200_advance_mu_t_loop(
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
    int nsteps);

/* The same two entry points in double precision, for WRF built with -r8.  Same semantics (host pointers in
 * compat mode with cached per-thread mirrors, residency and pinning as below; device pointers launched in place),
 * every operation rounded once in binary64. */
int wrfb200_advance_mu_t_r8(
    double *ww, const double *ww_1, const double *u, const double *u_1, const double *v, const double *v_1,
    double *mu, const double *mut, double *muave, double *muts, const double *muu, const double *muv,
    double *mudf, double *t, const double *t_1, double *t_ave, const double *ft, const double *mu_tend,
    double rdx, double rdy, double dts, double epssm,
    const double *dnw, const double *fnm, const double *fnp, const double *rdnw,
    const double *msfuy, const double *msfvx_inv, const double *msftx, const double *msfty,
    int periodic_x, int specified, int nested,
    int ids, int ide, int jds, int jde, int kde,
    int ims, int ime, int jms, int jme, int kms, int kme,
    int its, int ite, int jts, int jte, int kts, int kte);
int wrfb200_advance_mu_t_loop_r8(
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
    int nsteps);

/* Stream used by the device-pointer form of wrfb200_advance_mu_t (a cudaStream_t; NULL = default stream)
 * and kernel selection for it. Thread-local. */
int wrfb200_set_default_stream(void *cuda_stream);
int wrfb200_set_default_kernel(int kernel /* wrfb200_kernel */);

/* Domain caches.  A nested run calls the host-pointer form for the parent and each nest in turn, with other memory
 * extents (and often another kde).  The calling thread keeps, per precision, the device state of up to 8 domains,
 * keyed by device and memory extents ims..ime, jms..jme, kms..kme (not by array addresses), most recently used
 * first: its mirrors, device staging buffers and acoustic-loop residency.  A call for a domain seen before
 * allocates nothing.  The thread's lanes and pinned bounce buffers serve all its domains; the buffers only grow,
 * to the largest slab any of them needs.  Before a new domain is created, the least recently used ones are freed:
 * beyond 8, and on the domain's device while the free memory there cannot hold the new mirrors and staging buffers;
 * if the allocation still runs out of memory, every other domain of the thread is freed and it is tried once more,
 * then the call fails with WRFB200_ERR_NOMEM.  Each entry of a split call's device list (wrfb200_set_default_devices)
 * keeps its domains the same way, in a cache of its own.  Device-pointer calls keep the wrapping handle and
 * tensor maps of the thread's 4 most recent sets of (26 pointers, domain) per precision.
 *
 * wrfb200_release_cache frees all of it: every domain of the calling thread's caches, its device-pointer wrappers,
 * every host registration, and the shared patches of shared-tiles mode (wrfb200_set_shared_tiles) with every
 * thread's state for them.  Call it to hand the device memory back to the model, e.g. before a phase that needs it
 * or at the end of a run.  It also stops and joins the host threads of the staged route (wrfb200_set_host_pinning);
 * no call may be in flight then. */
int wrfb200_release_cache(void);

/* Acoustic-loop residency for HOST-pointer callers of wrfb200_advance_mu_t (thread-local).  Between begin and
 * end, the first call uploads everything; every later call with the SAME arrays, index sets and scalars
 * uploads only u and v -- what advance_uv changed -- runs the step on the device-resident state and
 * downloads the seven outputs.  Contract: between those calls the caller changes nothing but u and v (ww, t,
 * mu on the device are this routine's own previous outputs; the rest are constants of the RK sub-step).
 * This is the reference's per-call H2D of all 26 arrays (advance_mu_t_no_async.cu:245-306) reduced to the
 * two that change.  Residency is kept per domain, and begin / end act on every domain of the thread: the first
 * call of each domain in a loop uploads everything, whatever another domain did in between. */
int wrfb200_acoustic_loop_begin(void);
int wrfb200_acoustic_loop_end(void);

/* Page-locking of the caller's host arrays (process-wide; default off, or WRFB200_PIN_HOST=1).  When on,
 * every host array of a compat call is cudaHostRegister'ed the first time it is seen and stays registered
 * until wrfb200_release_cache / wrfb200_host_unregister_all, and is then copied directly at the pinned link
 * rate.  The caller must keep registered arrays allocated until then.  wrfb200_host_register pins one array
 * explicitly (the role of cudaHostAlloc in advance_mu_t_driver.cu:97-167).
 * Without it, pageable arrays take the staged route: host threads of the library copy them through pinned bounce
 * buffers it owns, overlapped with the transfers, so nothing of the caller's is registered.  What pinning still
 * buys over that route is the host-side copy that cannot overlap (DESIGN.md section 5 has the measured numbers).
 * The route is chosen per array from whether it is page-locked; wrfb200_default_last_transfer reports it.  The
 * staged route's pool of host threads (one per process, one thread per CPU of the process's affinity mask, at
 * most 16) starts with the first staged call and is stopped by wrfb200_release_cache and at unload; a process
 * forked after a staged call has no pool until its own first staged call. */
int wrfb200_set_host_pinning(int enable);
int wrfb200_host_register(const float *host, size_t bytes);
int wrfb200_host_unregister_all(void);

/* Kernel the most recent wrfb200_advance_mu_t call of this thread ran (a wrfb200_kernel id; AUTO resolved; for a
 * call split over several devices, the first part's). */
int wrfb200_default_last_kernel(int *kernel);

/* How the most recent host-pointer call of wrfb200_advance_mu_t / _loop (or the _r8 pair) of this thread moved its
 * arrays (thread-local): *route = 0 every array direct (page-locked: by the caller, e.g. cudaHostAlloc or torch
 * pin_memory, or by wrfb200_set_host_pinning), 1 some arrays staged through the library's pinned bounce buffers
 * (pageable ones), 2 every array staged.  The four 1-D arrays, a few hundred bytes, are copied directly even when
 * pageable but count by what they are.  No host-pointer call on this thread yet: WRFB200_ERR_STATE. */
int wrfb200_default_last_transfer(int *route);

/* What the most recent wrfb200_advance_mu_t / _loop call of this thread (either precision, host or device pointers)
 * did with its cache (thread-local): *state is a wrfb200_cache -- 0 re-used its domain's device state (or
 * device-pointer wrapper), 1 created it, 2 created it after freeing the least recently used domain(s).  A call split
 * over several devices reports the most any part did; a shared-tiles call, 1 when it created the shared patch or
 * the thread's handle for it.  No call on this thread has reached its cache yet (or the last one was refused
 * before): WRFB200_ERR_STATE. */
int wrfb200_default_last_cache(int *state);

/* How many times the host-pointer caches of this process have allocated their pinned bounce buffers (the staged
 * route's nine cudaHostAlloc buffers), first allocations and growth alike.  A diagnostic: the buffers only grow, to
 * the largest slab each cache has seen, so calls that alternate between domains a cache already holds allocate none. */
int wrfb200_bounce_allocations(long *count);

/* Devices the HOST-pointer form of wrfb200_advance_mu_t / _loop (and the _r8 pair) spreads its j-rows over.
 * Thread-local, like wrfb200_set_default_stream / _kernel.  n = 0 (devices may be NULL): back to the current
 * device only (the default).  Ids may repeat (several parts on one device).  Device-pointer calls ignore it and
 * run in place on the current device; the multi-GPU comm path (3b) is unaffected.
 * Each part is the single-device call applied to its rows: its own cached mirrors on its device, its rows plus
 * the one-row ring copied straight from the caller's arrays (no GPU-to-GPU traffic), issued from a host thread
 * of its own; every thread is joined before the call returns.  Results are bit-identical to the single-device
 * call.  Acoustic-loop residency, pinning (registered portable, so every device copies at the pinned rate) and
 * wrfb200_release_cache cover every part.  A failing part makes the call return its status, with the device and
 * rows in the message, after every part has finished.
 * n < 0, n > 64, devices == NULL with n > 0, or an id outside [0, device count): WRFB200_ERR_INVALID_ARG; no
 * device at all: WRFB200_ERR_CUDA.  Changing the list releases this thread's cached mirrors. */
int wrfb200_set_default_devices(const int *devices, int n);

/* Shared-tiles mode, for WRF's OpenMP builds (smpar, dm+sm), which cut a patch into tiles and make the HOST-pointer
 * call once per tile from the threads of a `!$OMP PARALLEL DO`.  Process-wide and opt-in (default off, or
 * WRFB200_SHARED_TILES=1); while it is off nothing behaves differently from the per-thread caches described above.
 * While it is on, host-pointer calls of wrfb200_advance_mu_t / _loop (and the _r8 pair) from ANY thread that pass
 * the same 26 arrays and the same memory extents are tiles of one patch:
 *   - One set of device mirrors per (precision, patch device, memory extents, 26 arrays), created by whichever tile
 *     arrives first.  Each thread keeps its own streams, staging buffers and handle bound to those mirrors, so its
 *     default stream (synchronised before the call) and kernel choice still apply.
 *   - The patch device is the calling thread's current device when the mode is enabled (with the environment
 *     variable: that of the first thread to call wrfb200_acoustic_loop_begin or a host-pointer entry point).
 *     Every shared call runs there whatever the calling thread's current device is, which is unchanged on return.
 *   - A tile's call uploads only what no concurrent tile reads or writes: t, mu and ww at level kts (read and
 *     written by the routine) over the tile's own columns, the read-only inputs over the tile's rows plus the
 *     one-cell ring.  It downloads the cells it writes, as always.
 *   - wrfb200_acoustic_loop_begin / _end (from any one thread, e.g. the master in the serial part of solve_em) act
 *     on every thread: the first call of a tile (its..ite x jts..jte) in the loop uploads that tile's set, later
 *     calls of the same tile with the same arrays and scalars upload only its rows of u and v plus the ring,
 *     whichever thread makes them.  The residency contract above applies per tile.
 *   - Contract: tiles of one patch must not overlap in computed cells (as in the Fortran); the caller changes no
 *     array while a tile's call runs.  Disabling the mode and wrfb200_release_cache free the shared mirrors and
 *     every thread's shared-call state: no call may be in flight then.
 *   - A shared call from a thread whose device list (wrfb200_set_default_devices) names several devices or another
 *     device than the patch device fails with WRFB200_ERR_UNSUPPORTED.  Device-pointer calls, handles (section 2)
 *     and the multi-GPU comm path (3b) are not affected.
 * Enabling without a CUDA device returns WRFB200_ERR_CUDA; enabling again on another device frees the patches of
 * the previous one. */
int wrfb200_set_shared_tiles(int enable);

/* Host-only: how a host-pointer call of this tile is split over n parts (1 <= n <= 64).  rows4[4p..4p+3] =
 * {first computed row, last computed row, first memory row, last memory row} of part p (Fortran j; a part
 * without rows has first > last).  The computed rows j_start..j_end are cut with j_start + nj*p/n; a part's
 * memory is its rows plus one ring row on each side (in i it keeps ims..ime).  Needs no GPU. */
int wrfb200_host_split_plan(const wrfb200_domain *dom, int its, int ite, int jts, int jte, int kts, int kte,
                            int n, int *rows4);

/* ------------------------------------------------------------------------------------------------
 * 2. Device-resident state (replaces the per-call malloc/H2D/D2H/free of advance_mu_t_no_async.cu).
 * ---------------------------------------------------------------------------------------------- */

/* Create a patch on CUDA device `device` (-1 = current).  If `allocate` is non-zero all 26 fields get
 * device mirrors with rows padded to a multiple of 32 floats; otherwise fields must be bound with
 * wrfb200_bind_device before use. */
int wrfb200_create(wrfb200_handle **out, const wrfb200_domain *dom, int device, int allocate);
int wrfb200_destroy(wrfb200_handle *h);

int wrfb200_set_stream(wrfb200_handle *h, void *cuda_stream);
int wrfb200_set_scalars(wrfb200_handle *h, float rdx, float rdy, float dts, float epssm);
int wrfb200_set_kernel(wrfb200_handle *h, int kernel /* wrfb200_kernel */);

/* Adopt a caller-owned device buffer for `field`.  pitch = row stride in floats (>= ime-ims+1);
 * for 1-D fields pitch is ignored. */
int wrfb200_bind_device(wrfb200_handle *h, int field, float *device_ptr, long pitch);
/* Query the device buffer of `field` (owned or bound). */
int wrfb200_device_ptr(wrfb200_handle *h, int field, float **device_ptr, long *pitch);

/* Async copies on the handle's stream between DENSE host arrays (Fortran extents ims:ime etc.) and the
 * device mirrors.  Host memory should be pinned for the copies to be truly asynchronous. */
int wrfb200_upload(wrfb200_handle *h, int field, const float *host);
int wrfb200_download(wrfb200_handle *h, int field, float *host);
/* Only the sub-range [i0..i1] x [k0..k1] x [j0..j1] (Fortran-numbered, inclusive; k ignored for 2-D). */
int wrfb200_upload_range(wrfb200_handle *h, int field, const float *host, int i0, int i1, int k0, int k1, int j0, int j1);
int wrfb200_download_range(wrfb200_handle *h, int field, float *host, int i0, int i1, int k0, int k1, int j0, int j1);

/* Resident-state verbs: the arrays a host-resident caller moves at the three cadences of the acoustic loop
 * (once per RK sub-step: constants and the state the loop starts from; every small step: u, v up and the
 * outputs down).  Dense host arrays, async on the handle's stream, NULL skips an array.
 * wrfb200_download_outputs copies exactly the cells the routine writes for the given tile. */
int wrfb200_upload_constants(
    wrfb200_handle *h, const float *ww_1, const float *u_1, const float *v_1, const float *t_1, const float *ft,
    const float *mut, const float *muu, const float *muv, const float *mu_tend,
    const float *msfuy, const float *msfvx_inv, const float *msftx, const float *msfty,
    const float *dnw, const float *fnm, const float *fnp, const float *rdnw);
int wrfb200_upload_state(wrfb200_handle *h, const float *ww, const float *t, const float *mu);
int wrfb200_set_uv(wrfb200_handle *h, const float *u, const float *v);
int wrfb200_download_outputs(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                             float *ww, float *t, float *t_ave, float *mu, float *muave, float *muts, float *mudf);
/* The same four verbs for a real*8 handle (double arrays). */
int wrfb200_upload_constants_r8(
    wrfb200_handle *h, const double *ww_1, const double *u_1, const double *v_1, const double *t_1, const double *ft,
    const double *mut, const double *muu, const double *muv, const double *mu_tend,
    const double *msfuy, const double *msfvx_inv, const double *msftx, const double *msfty,
    const double *dnw, const double *fnm, const double *fnp, const double *rdnw);
int wrfb200_upload_state_r8(wrfb200_handle *h, const double *ww, const double *t, const double *mu);
int wrfb200_set_uv_r8(wrfb200_handle *h, const double *u, const double *v);
int wrfb200_download_outputs_r8(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                                double *ww, double *t, double *t_ave, double *mu, double *muave, double *muts,
                                double *mudf);

/* One advance_mu_t over the tile its:ite x jts:jte (kts:kte as the Fortran), asynchronous on the stream. */
int wrfb200_step(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte);
/* `nsteps` back-to-back steps replayed from a CUDA graph captured on first use for this tile. */
int wrfb200_step_graph(wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte, int nsteps);
int wrfb200_sync(wrfb200_handle *h);

/* real*8 handles: the verbs above that carry a precision, with double arrays / scalars.  create_r8 pads rows to
 * a multiple of 16 doubles (128 bytes); pitches are in doubles.  step, step_graph, sync, set_stream,
 * set_kernel, destroy, launch_count and last_kernel work on handles of either precision. */
int wrfb200_create_r8(wrfb200_handle **out, const wrfb200_domain *dom, int device, int allocate);
int wrfb200_set_scalars_r8(wrfb200_handle *h, double rdx, double rdy, double dts, double epssm);
int wrfb200_bind_device_r8(wrfb200_handle *h, int field, double *device_ptr, long pitch);
int wrfb200_device_ptr_r8(wrfb200_handle *h, int field, double **device_ptr, long *pitch);
int wrfb200_upload_r8(wrfb200_handle *h, int field, const double *host);
int wrfb200_download_r8(wrfb200_handle *h, int field, double *host);
int wrfb200_upload_range_r8(wrfb200_handle *h, int field, const double *host, int i0, int i1, int k0, int k1, int j0, int j1);
int wrfb200_download_range_r8(wrfb200_handle *h, int field, double *host, int i0, int i1, int k0, int k1, int j0, int j1);

/* Number of kernels this library has launched on behalf of `h` since creation (bench accounting). */
int wrfb200_launch_count(wrfb200_handle *h, long *count);
/* Kernel of the most recent launch on `h` (a wrfb200_kernel id; AUTO resolved to what actually ran). */
int wrfb200_last_kernel(wrfb200_handle *h, int *kernel);

/* ------------------------------------------------------------------------------------------------
 * 3. Halo support for the 2-D (i,j) decomposition (one patch per rank).
 *    pack:   copy the `width` cells just INSIDE the patch edge `side` of `field` into a dense buffer
 *    unpack: copy a dense buffer into the `width` halo cells just OUTSIDE that edge.
 *    Buffer layout is [j][k][i] over the packed sub-box (i fastest); ips..ipe/jps..jpe is the patch.
 *    Buffer sizes: WEST/EAST width*nk*(jpe-jps+1) floats, SOUTH/NORTH (ipe-ips+1)*nk*width floats
 *    (nk = kme-kms+1 for 3-D fields, 1 for 2-D).
 *    The caller moves the buffers between ranks with its own transport (MPI or NCCL send/recv, a device copy),
 *    so ranks may sit on different hosts.  Asynchronous on the handle's stream.
 * ---------------------------------------------------------------------------------------------- */
int wrfb200_pack_halo(wrfb200_handle *h, int field, int side, int width,
                      int ips, int ipe, int jps, int jpe, float *device_buf);
int wrfb200_unpack_halo(wrfb200_handle *h, int field, int side, int width,
                        int ips, int ipe, int jps, int jpe, const float *device_buf);
/* The same on a real*8 handle: same box, layout and sizes, counted in doubles.  On a real*4 handle they return
 * WRFB200_ERR_STATE; the two verbs above return WRFB200_ERR_UNSUPPORTED on a real*8 one. */
int wrfb200_pack_halo_r8(wrfb200_handle *h, int field, int side, int width,
                         int ips, int ipe, int jps, int jpe, double *device_buf);
int wrfb200_unpack_halo_r8(wrfb200_handle *h, int field, int side, int width,
                           int ips, int ipe, int jps, int jpe, const double *device_buf);

/* Deterministic stand-in for advance_uv (which in WRF updates u,v between two advance_mu_t calls but is
 * not part of the reference): field = WRFB200_U: u(i,k,j) += c*(mudf(i,j)-mudf(i-1,j));
 * field = WRFB200_V: v(i,k,j) += c*(mudf(i,j)-mudf(i,j-1)); over i0..i1 x all memory levels x j0..j1.
 * It makes the multi-step loop and the halo exchange load-bearing in tests (SURVEY.md section 8d). */
int wrfb200_standin_advance_uv(wrfb200_handle *h, int field, float c, int i0, int i1, int j0, int j1);
/* The same on a real*8 handle, every operation rounded once in binary64. */
int wrfb200_standin_advance_uv_r8(wrfb200_handle *h, int field, double c, int i0, int i1, int j0, int j1);

/* ------------------------------------------------------------------------------------------------
 * 3b. Multi-GPU behind the boundary: one rank per GPU of one NVLink box, 2-D (i,j) patches, the one-cell
 *     halo exchange fused into the kernels over peer-mapped memory (csrc/comm.cu).  Replaces the j-slab
 *     plan + per-call host re-upload + per-device launch loop of advance_mu_t_no_async.cu:87-162,
 *     :276-298, :329-357.  The handle must own its mirrors (wrfb200_create(..., allocate=1)) with
 *     memory = patch + halo (>= 1 cell) and the GLOBAL ids..jde, so the boundary clamps of
 *     module_small_step_em.f90:91-106 fire on edge ranks only.  Rank r sits at (r % px, r / px).
 *
 *     Bootstrap (transport-agnostic, like an ncclUniqueId): every rank calls wrfb200_comm_init, the caller
 *     all-gathers the WRFB200_COMM_INFO_BYTES blobs in rank order (MPI_Allgather, torch.distributed, a
 *     pipe ...), every rank calls wrfb200_comm_connect.  Ranks may be processes (CUDA IPC) or several
 *     handles of one process (peer access).
 *
 *     Per RK sub-step, after uploading:  wrfb200_comm_push_constants  (u_1, muu, msfuy, v_1, muv,
 *     msfvx_inv, t_1 edges into the neighbours' halos, bracketed by a stream-ordered neighbour barrier).
 *     Per acoustic step:  [caller's advance_uv]  ->  wrfb200_comm_push_uv  ->  wrfb200_comm_step.
 *     wrfb200_comm_step stores this patch's south row of v into the south neighbour's north halo (its
 *     south-row blocks do that before they start), waits -- in the blocks that own the east column / north row
 *     only -- for its own east / north halo of u / v, and stores mu, muts, mudf of its east column / north row
 *     into the east / north neighbour's west / south halo for that neighbour's next advance_uv; a kernel that
 *     reads those halos must be preceded by wrfb200_comm_wait_outputs on the same stream.  Everything is
 *     asynchronous on the handle's stream; there is no host synchronisation and no NCCL call inside the loop.
 *     All ranks must issue the same sequence of steps (the flags are step counters).  A halo wait gives up
 *     after 5 s (WRFB200_FLAG_TIMEOUT_MS) and is reported by wrfb200_comm_status.  Each binary32 step runs the
 *     TMA pipe kernel, so wrfb200_comm_init fails with WRFB200_ERR_UNSUPPORTED when the patch has more than 337
 *     computed levels.
 *
 *     Real*8 ranks (wrfb200_create_r8, allocate=1): wrfb200_comm_init_r8 instead of wrfb200_comm_init, and the
 *     _r8 forms of the loop and the stand-in (double c).  connect, barrier, push_constants, push_uv,
 *     wait_outputs, step and status take no floating-point argument and serve both precisions.  Each step runs
 *     the double2 tile kernel with the exchange fused in, so wrfb200_comm_init_r8 fails with
 *     WRFB200_ERR_UNSUPPORTED when the patch has more than 220 computed levels.  All ranks must hold the same
 *     precision: connect rejects a neighbour's blob of the other one with WRFB200_ERR_INVALID_ARG.
 *
 *     Periodic domains (WRF's periodic_x, and periodic_x + periodic_y on an open domain): call
 *     wrfb200_comm_set_wrap before wrfb200_comm_init[_r8] to make the exchange cyclic across the domain edge, so
 *     the ring of a periodic domain is refreshed inside the loop as WRF refreshes it every small step
 *     (u(ide) = u(ids), t_1(ids-1) = t_1(ide-1), t_1(ide) = t_1(ids), the same in j, and mu, muts, mudf after the
 *     step).  Without the call an edge rank's ring past the domain edge is never written.  wrap_x needs the
 *     domain's periodic_x; wrap_y needs specified == 0 and nested == 0.  The patches follow WRF's convention: the
 *     west-edge rank starts at ids, the east-edge rank ends at ide and computes at least one column (likewise in
 *     j); that rank's column ide (row jde) receives the wrap.  px = 1 (py = 1) makes a rank its own neighbour,
 *     which costs one extra copy launch per step.  comm_init fails with WRFB200_ERR_INVALID_ARG on a request that
 *     breaks these rules, connect on a neighbour with other wrap flags or other global extents.  The stand-in
 *     advance_uv then updates u from i_start (v from j_start) on a wrapped axis.
 * ---------------------------------------------------------------------------------------------- */
#define WRFB200_COMM_INFO_BYTES 2048
int wrfb200_comm_info_bytes(void);
/* periodic wrap of the exchange (0/1 each); before wrfb200_comm_init / _init_r8, kept for both precisions */
int wrfb200_comm_set_wrap(wrfb200_handle *h, int wrap_x, int wrap_y);
int wrfb200_comm_init(wrfb200_handle *h, int px, int py, int rank,
                      int ips, int ipe, int jps, int jpe, void *info_out /* WRFB200_COMM_INFO_BYTES */);
int wrfb200_comm_connect(wrfb200_handle *h, const void *all_infos /* nranks blobs, rank order */, int nranks);
int wrfb200_comm_barrier(wrfb200_handle *h);          /* stream-ordered barrier with the neighbours */
int wrfb200_comm_push_constants(wrfb200_handle *h);
int wrfb200_comm_push_uv(wrfb200_handle *h);          /* u west column -> west neighbour (px > 1, or wrap_x); the v
                                                         south row is pushed by wrfb200_comm_step itself, except to a
                                                         rank that is its own south neighbour (wrap_y, py = 1) */
int wrfb200_comm_wait_outputs(wrfb200_handle *h);     /* west / south halos of mu, muts, mudf have arrived */
int wrfb200_comm_step(wrfb200_handle *h);             /* advance_mu_t over the patch, fused with its exchange */
/* stand-in advance_uv (see wrfb200_standin_advance_uv) over this patch's share of the global update boxes,
 * preceded by wrfb200_comm_wait_outputs */
int wrfb200_comm_standin_advance_uv(wrfb200_handle *h, float c);
/* nsteps x (push_uv, step[, stand-in between steps]) -- the acoustic loop of one RK sub-step; with
 * use_graph the sequence is captured once and replayed from a CUDA graph. */
int wrfb200_comm_loop(wrfb200_handle *h, int nsteps, int standin, float c, int use_graph);
/* Synchronises the stream; flag_timeouts != 0 means some halo wait gave up (results are then invalid);
 * steps_done = advance_mu_t launches completed since wrfb200_comm_init. */
int wrfb200_comm_status(wrfb200_handle *h, int *flag_timeouts, long *steps_done);
/* real*8 ranks */
int wrfb200_comm_init_r8(wrfb200_handle *h, int px, int py, int rank,
                         int ips, int ipe, int jps, int jpe, void *info_out /* WRFB200_COMM_INFO_BYTES */);
int wrfb200_comm_standin_advance_uv_r8(wrfb200_handle *h, double c);
int wrfb200_comm_loop_r8(wrfb200_handle *h, int nsteps, int standin, double c, int use_graph);

/* ------------------------------------------------------------------------------------------------
 * 4. Harness utilities (host side; usable without a GPU).
 * ---------------------------------------------------------------------------------------------- */

/* Index sets of module_small_step_em.f90:91-106. */
int wrfb200_bounds(int periodic_x, int specified, int nested,
                   int ids, int ide, int jds, int jde,
                   int its, int ite, int jts, int jte, int kts, int kte,
                   int *i_start, int *i_end, int *j_start, int *j_end, int *k_start, int *k_end);

/* Deterministic atmosphere-like synthetic field (counter-based: the value of a cell depends only on
 * (seed, field, GLOBAL i,k,j, domain extents), so every decomposition generates the same global field).
 * Fills the dense host array of `field` for the patch described by `dom`.  dx_m (grid spacing in metres) is
 * accepted for interface stability and currently unused: the field magnitudes are grid-spacing independent;
 * rdx, rdy and dts are the caller's scalars. */
int wrfb200_synth_field(int field, uint64_t seed, const wrfb200_domain *dom, float dx_m, float *host_out);

/* The reference's comparison metrics (common.cu:68-164) over n floats: number of bit-equal values,
 * max relative error (|a-b|/max(|a|,|b|), or max(|a|,|b|) when either is zero, :117-120), max absolute
 * error, max ulp distance (:51-66), rmse.  Returns WRFB200_ERR_INVALID_ARG if either side holds a NaN
 * (the reference aborts, :108-115). */
typedef struct wrfb200_compare_result {
    long n, n_equal, n_different;
    float max_rel, max_abs, rmse;
    long max_ulp;
} wrfb200_compare_result;
int wrfb200_compare(const float *a, const float *b, long n, wrfb200_compare_result *out);
/* The same metrics over n doubles (real*8 fields), computed in binary64; the ulp distance is taken over the 64-bit
 * ordered bit patterns (saturating at LONG_MAX, which only opposite-signed values near the infinities reach). */
typedef struct wrfb200_compare_result_r8 {
    long n, n_equal, n_different;
    double max_rel, max_abs, rmse;
    long max_ulp;
} wrfb200_compare_result_r8;
int wrfb200_compare_r8(const double *a, const double *b, long n, wrfb200_compare_result_r8 *out);

/* Host-only description of the launch the TMA kernel makes for the tile its:ite x jts:jte of `dom` on a device with
 * `resident_blocks` resident blocks (0: a B200, 2 x 148): plan10 = {configuration TJ*10+STAGES, TJ, STAGES, tile
 * columns, block rows of 2-row tiles, block rows of 1-row tiles, remainder-strip blocks, first strip column (memory
 * index), grid size, dynamic shared memory in bytes}; configuration 62 is <1, 2> with the level tables read from
 * L2.  WRFB200_ERR_UNSUPPORTED past the pipe kernel's level limit (nk > 337).  Needs no GPU; the launch geometry is
 * unit-tested with it. */
int wrfb200_pipe_plan(const wrfb200_domain *dom, int its, int ite, int jts, int jte, int kts, int kte,
                      int resident_blocks, long long *plan10);

const char *wrfb200_last_error(void);
int wrfb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WRFB200_H */
