// amt_params.h -- kernel argument block and IEEE helpers shared by the advance_mu_t kernels.
//
// Semantics follow the reference Fortran, /root/reference/module_small_step_em.f90:91-250
// (restated in SURVEY.md section 8).  All indices in here are 0-based MEMORY indices
// (Fortran index minus ims / kms / jms); the host layer (capi.cu) does that shift, like the
// reference wrapper does at advance_mu_t_no_async.cu:57-79.
#pragma once
#include <cuda.h>            // CUtensorMap (types only; the driver is reached through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>

// Fused halo exchange of the multi-GPU path (comm.cu): everything a kernel needs to (a) wait for the halo
// cells a neighbour rank stores straight into this patch's memory over NVLink, (b) store its own edge
// values straight into the neighbours' halos, and (c) tell the neighbours when it is done with them.
// All flag words are monotonically increasing acoustic-step counters.  The step a launch computes is
// `*epoch + step_index + 1`: `epoch` (device memory of this rank) counts the steps completed before the current
// loop, `step_index` is the launch's position in the loop -- a kernel ARGUMENT, so a captured CUDA graph of the
// loop replays correctly (epoch moves on by one small kernel per loop, not per step).  enabled == 0: single GPU.
struct AmtHalo {
    int enabled;
    int ipe_mem, jpe_mem;              // memory index of the patch's east column / north row
    int ips_mem, jps_mem;              // ... west column / south row
    // waits: flags in THIS rank's memory, advanced by the east / north neighbour when its u / v edge is in
    // this patch's east / north halo (null: no such neighbour)
    const unsigned *uv_flag_east, *uv_flag_north;
    // peer stores of the 2-D outputs: cell (ipe, j) -> e_*[j * e_pitch2], cell (i, jpe) -> n_*[i]
    float *e_mu, *e_muts, *e_mudf;     // column ips_E - 1 of the east neighbour's arrays (null: none)
    long long e_pitch2;
    float *n_mu, *n_muts, *n_mudf;     // row jps_N - 1 of the north neighbour's arrays (null: none)
    // fused v push (j-slab neighbours): the blocks of the patch's SOUTH row store that row of v (all memory
    // levels) into the south neighbour's north halo before they start, after the neighbour has finished reading
    // it in its previous step (war_flag_south >= step - 1); the last of them releases `step`
    float *s_v;                        // south neighbour's v at (my memory column 0, level 0, row jps) (null: none)
    long long s_pitch3;
    const unsigned *war_flag_south;    // in THIS rank's memory
    unsigned *uv_flag_to_south;        // in the south neighbour's memory
    unsigned *push_counter;            // south-row blocks that have pushed in this launch
    int push_blocks;                   // tile blocks in the south row of the launch (set by the launcher)
    // "outputs of this step are in your halo, and I have finished reading the u / v halo you filled": released
    // to the east / north neighbour by the LAST of the blocks that own the patch's east column / north row --
    // exactly the blocks that store those outputs and read that halo; no other block pays anything
    unsigned *out_flag_to_east, *out_flag_to_north;   // in the neighbours' memory (null: none)
    unsigned *east_counter, *north_counter;           // in this rank's memory
    int east_blocks, north_blocks;                    // blocks owning column ipe / row jpe (set by the launcher)
    int north_second;                                 // dispatch the north block row right after the south row (amt_pipe.cu)
    const unsigned *epoch;             // steps completed before the current loop (this rank's memory)
    unsigned step_index;               // position of this launch in the loop
    unsigned *status;                  // != 0: a flag wait timed out (checked by the host)
    unsigned long long timeout_ns;     // a flag wait gives up after this long (never hang the GPU)
};

// Argument block of one launch, for element type T (float: the real*4 kernels; double: the real*8 kernels of a
// handle created with wrfb200_create_r8).  AmtParams / AmtParamsR8 below are the two instances; the float one keeps
// its own struct name so the float kernels' symbols do not change.
template <class T>
struct AmtFields {
    // 3-D fields, (i fastest, k, j): element (i,k,j) at  j*jstride + k*pitch + i
    T *ww;
    const T *ww_1, *u, *u_1, *v, *v_1;
    T *t;
    const T *t_1;
    T *t_ave;
    const T *ft;
    // 2-D fields: element (i,j) at  j*pitch2 + i
    T *mu;
    const T *mut;
    T *muave, *muts;
    const T *muu, *muv;
    T *mudf;
    const T *mu_tend, *msfuy, *msfvx_inv, *msftx, *msfty;
    // 1-D fields, index 0 = level kms
    const T *dnw, *fnm, *fnp, *rdnw;
    T rdx, rdy, dts, epssm;
    long long pitch;    // 3-D row stride in elements
    long long jstride;  // 3-D plane stride in elements (= pitch * kdim)
    long long pitch2;   // 2-D row stride in elements
    int i0, i1;         // computed i range (i_start..i_end), inclusive, memory index
    int j0, j1;         // computed j range
    int k0;             // memory index of level kts
    int nk;             // number of computed levels: k_start..k_end = kts..kte-1
    int kdim, jdim;     // memory extents in k and j (jstride == pitch * kdim)
    AmtHalo halo;       // fused multi-GPU halo exchange (enabled == 0 on a single GPU); for double its peer
                        // pointers address doubles (pitches stay in elements)
};
struct AmtParams : AmtFields<float> {};
struct AmtParamsR8 : AmtFields<double> {};

// Tensor maps of the TMA-staged kernel (amt_pipe.cu): boxes are [columns x 1 level x rows].
struct AmtTmaMaps {
    alignas(64) CUtensorMap u132;       // u    [132 x 1 x 1]
    alignas(64) CUtensorMap u1_132;     // u_1  [132 x 1 x 1]
    alignas(64) CUtensorMap v_2rows;    // v    [128 x 1 x 2]  rows j, j+1
    alignas(64) CUtensorMap v1_2rows;   // v_1  [128 x 1 x 2]
    alignas(64) CUtensorMap t1_136;     // t_1  [136 x 1 x 1]  both ring columns
    alignas(64) CUtensorMap t1_128;     // t_1  [128 x 1 x 1]
    const void *key_ptrs[5];            // what the maps were built for
    long long key_dims[3];
    int valid;
};

// Round-to-nearest single operations that the compiler may never contract into an FMA,
// whatever -fmad says: this is what keeps the result bit-identical to the Fortran's real*4
// arithmetic (the reference gets the same effect with `-fmad=false`, Makefile:12).
__device__ __forceinline__ float f_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float f_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float f_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float f_div(float a, float b) { return __fdiv_rn(a, b); }
// The same four in binary64 for the real*8 kernels.  Division stays the IEEE __ddiv_rn: its correctly rounded
// sequence is built from DFMA internally (as __fdiv_rn's is from FFMA), but no operation of the formula itself is
// ever contracted.
__device__ __forceinline__ double f_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double f_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double f_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double f_div(double a, double b) { return __ddiv_rn(a, b); }

// ---- cross-GPU flag helpers (system scope: the peer is another GPU on NVLink) ----
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Spin until *flag >= want (one thread; the caller follows with a block barrier).  A neighbour that never
// arrives must not hang the GPU: after kFlagTimeoutNs the wait gives up and records it in *status.
__device__ __forceinline__ void wait_flag(const unsigned *flag, unsigned want, unsigned *status,
                                          unsigned long long timeout_ns)
{
    if ((int)(ld_acquire_sys(flag) - want) >= 0) return;
    const unsigned long long t0 = global_timer_ns();
    while ((int)(ld_acquire_sys(flag) - want) < 0) {
        __nanosleep(64);
        if (global_timer_ns() - t0 > timeout_ns) { atomicAdd(status, 1u); return; }
    }
}

// Dynamic shared memory opt-in: raised ONCE per (kernel, device) to the architectural maximum and never
// lowered, so two handles or host threads with different level counts cannot interleave set(A), set(B<A),
// launch(A) into a spurious launch failure, and a captured graph never sees the limit shrink under it.
constexpr int kMaxDynSmemOptIn = 227 * 1024;
template <class K>
inline cudaError_t amt_raise_smem_limit(K kernel, bool (&done)[64])
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (done[dev]) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmemOptIn);
    if (e == cudaSuccess) done[dev] = true;
    return e;
}

// Dispatch order of the block rows in a fused multi-GPU launch: south row first (its blocks push v to the south
// neighbour before anything else), NORTH ROW SECOND, then the rest.  The north-row blocks are the ones that wait
// for the north neighbour's v (pushed by ITS first blocks, i.e. at about the same time) and the ones whose
// completion tells that neighbour "step done": run early, neither their wait nor their system-scope fence and
// flag store sit at the end of the launch, and the neighbour's write-after-read guard is released a whole
// launch ahead of its use.  Used by the binary32 pipe kernels and the fused real*8 tile kernel alike.
template <class T>
__device__ __forceinline__ int north_row_second(const AmtFields<T> &p, const int by, const int nby)
{
    if (!p.halo.enabled || !p.halo.north_second || !p.halo.out_flag_to_north || nby < 3) return by;
    return by == 0 ? 0 : (by == 1 ? nby - 1 : by - 1);
}

// Launchers (defined in the kernel translation units).
bool amt_pipe_plan(const AmtParams &p, int slots, long long out[10]);   // host-only launch description
cudaError_t amt_pipe_preload();                                         // load all kernels of amt_pipe.cu (see there)
// blocks of a fused launch that own the patch's east column / north row signal the neighbours when they finish
__device__ __forceinline__ void amt_halo_block_done(const AmtHalo &hx, bool owns_east, bool owns_north, unsigned step)
{
    __threadfence_system();
    if (owns_north && hx.out_flag_to_north && atomicAdd(hx.north_counter, 1u) == (unsigned)hx.north_blocks - 1u) {
        *hx.north_counter = 0u;
        __threadfence_system();
        st_release_sys(hx.out_flag_to_north, step);
    }
    if (owns_east && hx.out_flag_to_east && atomicAdd(hx.east_counter, 1u) == (unsigned)hx.east_blocks - 1u) {
        *hx.east_counter = 0u;
        __threadfence_system();
        st_release_sys(hx.out_flag_to_east, step);
    }
}
cudaError_t amt_launch_column(const AmtParams &p, cudaStream_t stream);
cudaError_t amt_launch_tile(const AmtParams &p, cudaStream_t stream);
bool amt_tile_supported(const AmtParams &p);
bool amt_pipe_supported(const AmtParams &p);
// Level limits: every kernel keeps a per-column slab of all p.nk levels in shared memory, so the level count decides
// whether a kernel can run at all.  true when p.nk fits; *max_levels (if given) receives the kernel's largest nk.
bool amt_pipe_levels_fit(const AmtParams &p, int *max_levels = nullptr);             // 337
bool amt_tile_levels_fit(const AmtParams &p, int *max_levels = nullptr);             // 223
bool amt_column_levels_fit(const AmtParams &p, int *max_levels = nullptr);           // 454
bool amt_tile_levels_fit(const AmtParamsR8 &p, int *max_levels = nullptr);           // 220
bool amt_column_levels_fit(const AmtParamsR8 &p, int *max_levels = nullptr);         // 227
bool amt_build_tma_maps(const AmtParams &p, AmtTmaMaps *maps);                    // cached: rebuilds only on change
cudaError_t amt_launch_pipe(const AmtParams &p, const AmtTmaMaps &maps, cudaStream_t stream);
// real*8 kernels (amt_column.cu, amt_tile_r8.cu)
cudaError_t amt_launch_column(const AmtParamsR8 &p, cudaStream_t stream);
cudaError_t amt_launch_tile(const AmtParamsR8 &p, cudaStream_t stream);       // p.halo.enabled: the multi-GPU kernel
bool amt_tile_supported(const AmtParamsR8 &p);
cudaError_t amt_tile_r8_preload();                                               // see amt_pipe_preload
