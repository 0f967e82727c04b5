// comm.cu -- multi-GPU advance_mu_t behind the C ABI: 2-D (i,j) patch decomposition whose one-cell halo
// exchange is FUSED into the kernels over peer-mapped memory (NVLink / NVSwitch), one rank per GPU.
//
// The reference's multi-GPU path lives inside its one C call: a 1-D j-slab plan over three hard-coded
// devices (/root/reference/advance_mu_t_no_async.cu:12, :87-162), every slab re-uploaded from the host with
// three rows of overlap on every call (:276-298), one launch per device (:329-357), no GPU<->GPU traffic.
// Here a rank owns a patch ips:ipe x jps:jpe of the global domain (device-resident, wrfb200_create) and
//   * learns its neighbours' device buffers once (wrfb200_comm_init -> the caller all-gathers the opaque
//     info blobs with whatever transport it has: MPI_Allgather in WRF, torch.distributed in bench.py, a
//     pipe in tests/c_comm_harness.c -> wrfb200_comm_connect maps them: CUDA IPC between processes, plain
//     peer access inside one process);
//   * pushes the halo cells its neighbours read STRAIGHT INTO THEIR ARRAYS with ordinary stores:
//       - the v south row (read at j+1, module_small_step_em.f90:143-144) by the south-row blocks of the
//         advance_mu_t kernel itself before they start; the u west column (read at i+1, :145-146; only for
//         px > 1) by the small kernel `push_kernel`,
//       - mu, muts, mudf east column / north row (what the neighbour's next advance_uv reads) by the
//         advance_mu_t kernel itself, from the scan thread that has just computed them (amt_pipe.cu; real*8:
//         amt_tile_r8.cu),
//       - the loop constants u_1, muu, msfuy, v_1, muv, msfvx_inv, t_1 once per RK sub-step;
//   * orders everything with monotonically increasing epoch flags in device memory (st.release.sys /
//     ld.acquire.sys): only the blocks of advance_mu_t that own the patch's east column / north row wait
//     -- at their start, for the neighbour's u / v push of this step -- while every other block runs
//     immediately, so the exchange overlaps the interior compute inside ONE launch per step; a one-thread
//     signal kernel behind it releases "outputs of step n are in your halo" to the east / north neighbours,
//     which is also the write-after-read guard of their next u / v push.
// No pack / send / recv / unpack launches and no host synchronisation inside the acoustic loop; the whole
// n-step loop replays from one CUDA graph per rank.  A flag wait that exceeds its time-out gives up and is
// reported by wrfb200_comm_status (a stuck neighbour must never hang the GPU).
//
// Epochs: a step is numbered `epoch + index + 1`, where `epoch` (a device word of each rank) counts the steps
// completed before the current loop and `index` is the step's position in the loop -- a kernel argument, so the
// captured graph of a loop replays unchanged; one tiny kernel per LOOP moves the epoch on.  All ranks run the
// same sequence, so step numbers agree.  Flags live in the READER's memory and are written by the neighbour:
//   uv_from_east / uv_from_north  = n : the u / v halo for step n is in place
//                                       (u: push_kernel; v: the south-row blocks of the neighbour's step n)
//   out_from_west / out_from_south = n : the west / south neighbour's blocks that own its east column / north
//                                       row have all finished step n: its mu, muts, mudf edges are in my halo AND
//                                       it no longer reads the u / v halo I filled for step n
//
// Real*8 ranks (wrfb200_create_r8 + wrfb200_comm_init_r8) run the same protocol with the same flags: the step is
// the double2 tile kernel with the exchange fused in (amt_tile_kernel_r8<TJ, true>, amt_tile_r8.cu), the peer
// addresses are computed with the element size, and push_kernel moves double edges as pairs of 4-byte words.  Both
// ranks of a pair must hold the same precision (checked at connect).
//
// Periodic wrap (wrfb200_comm_set_wrap): on a wrapped axis the neighbours are cyclic and the edge rank's column ide
// (row jde) is the cell that receives the wrap -- WRF's u(ide) = u(ids) -- so that rank exchanges over ips..ide-1
// (jps..jde-1) as if its patch ended there.  A peer then addresses a cell at my Fortran index + (di, dj), the period
// on a wrapped side and 0 otherwise.  A rank can be its own neighbour (px = 1 or py = 1): no flag wait may depend on
// a block of the same launch, so a self side is served by stream order alone -- its u / v edge goes through
// push_kernel before the step, its outputs are plain stores into this rank's own arrays, and it has no wait and no
// signal.  With px = 2 (py = 2) the same rank sits on both sides and uses the two per-side flag slots.
#include <unistd.h>

#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "capi_internal.h"

namespace {

enum FlagWord {
    F_UV_E = 0, F_UV_N = 1, F_OUT_W = 2, F_OUT_S = 3,
    F_BAR = 4,                       // 4..7: neighbour-barrier slots, indexed by the side the neighbour is on
    F_EPOCH = 9, F_STATUS = 10, F_PUSH_DONE = 11, F_VPUSH_DONE = 12, F_EAST_DONE = 13, F_NORTH_DONE = 14,
    F_WORDS = 32
};

// fields a neighbour stores into (order fixed: it is part of the info blob)
const int kXf[] = {WRFB200_U, WRFB200_V, WRFB200_MU, WRFB200_MUTS, WRFB200_MUDF,
                   WRFB200_U_1, WRFB200_V_1, WRFB200_T_1, WRFB200_MUU, WRFB200_MUV,
                   WRFB200_MSFUY, WRFB200_MSFVX_INV};
constexpr int kNX = 12;
constexpr uint32_t kMagic = 0x57424332u;

struct CommInfo {
    uint32_t magic;
    int rank, px, py;
    int pid, device;
    int esize;                       // bytes per element: 4 (binary32) or 8 (real*8); neighbours must agree
    uint64_t host_id;
    int ims, ime, jms, jme, kms, kme;
    int ips, ipe, jps, jpe;          // exchange extents (ipe = ide-1 / jpe = jde-1 on a wrapped edge)
    int wrap_x, wrap_y;
    int ids, ide, jds, jde;
    long long pitch3, pitch2;
    uint64_t ptr[kNX + 1];           // device addresses in the exporting process (last: flag block)
    uint64_t offset[kNX + 1];        // address - base of its allocation (IPC handles name allocations)
    cudaIpcMemHandle_t ipc[kNX + 1];
};
static_assert(sizeof(CommInfo) <= WRFB200_COMM_INFO_BYTES, "info blob too small");

struct Peer {
    bool present = false;
    bool self = false;               // this rank is its own neighbour on that side: stream order, no flags
    int di = 0, dj = 0;              // the peer's Fortran index of my cell (i, j) is (i + di, j + dj)
    CommInfo info{};
    float *f[WRFB200_NUM_FIELDS] = {};
    unsigned *flags = nullptr;
};

inline bool is3(int f) { return f >= WRFB200_WW && f <= WRFB200_FT; }
inline int opposite(int side) { return side ^ 1; }     // WEST<->EAST, SOUTH<->NORTH

uint64_t host_id()
{
    char name[256] = {0};
    gethostname(name, sizeof(name) - 1);
    uint64_t h = 1469598103934665603ull;
    for (const char *c = name; *c; ++c) h = (h ^ (uint64_t)(unsigned char)*c) * 1099511628211ull;
    // processes in different containers / namespaces of one host cannot share IPC handles either
    char boot[64] = {0};
    if (FILE *fp = fopen("/proc/sys/kernel/random/boot_id", "r")) {
        if (fgets(boot, sizeof(boot), fp)) for (const char *c = boot; *c; ++c) h = (h ^ (uint64_t)(unsigned char)*c) * 1099511628211ull;
        fclose(fp);
    }
    return h;
}

// base address of the allocation holding `p` (cuMemGetAddressRange, reached through the runtime so the
// library has no link-time dependency on libcuda)
typedef int (*AddrRangeFn)(unsigned long long *, size_t *, unsigned long long);
bool alloc_base(const void *p, uint64_t *base)
{
    static AddrRangeFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return (AddrRangeFn)f;
    }();
    if (!fn) return false;
    unsigned long long b = 0;
    size_t n = 0;
    if (fn(&b, &n, (unsigned long long)(uintptr_t)p) != 0) return false;
    *base = b;
    return true;
}

// Process-wide cache of opened IPC allocations: a handle may be opened only once per process, and several
// small fields of one peer can share an allocation.
struct OpenedIpc { void *base; int refs; };
std::map<std::string, OpenedIpc> &ipc_cache()
{
    static std::map<std::string, OpenedIpc> m;
    return m;
}
std::mutex &ipc_mutex()
{
    static std::mutex m;
    return m;
}

}  // namespace

struct wrfb200_comm {
    int px = 1, py = 1, rank = 0, nranks = 1;
    int ips = 0, ipe = 0, jps = 0, jpe = 0;    // exchange extents
    int wrap_x = 0, wrap_y = 0;
    int nbr[4] = {-1, -1, -1, -1};
    Peer peer[4];
    unsigned *flags = nullptr;                 // this rank's flag block (device memory)
    cudaStream_t own_stream = nullptr;
    bool connected = false;
    unsigned bar_epoch = 0;
    unsigned long long timeout_ns = 5ull * 1000ull * 1000ull * 1000ull;
    AmtHalo halo{};
    std::vector<std::string> opened;           // keys into ipc_cache()
    struct LoopGraph { cudaGraphExec_t exec; long launches; };
    std::map<std::tuple<int, int, unsigned long long>, LoopGraph> graphs;   // (nsteps, standin, bits of c)
};

namespace {

#define CUC(call)                                                                                         \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return wrfb200_fail(WRFB200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                __FILE__, __LINE__);                                                      \
    } while (0)

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------
// element (i,k,j) of a box: src[j*sj + k*sp + i] -> dst[j*dj + k*dp + i]
struct Box {
    const float *src;
    float *dst;
    long long sp, sj, dp, dj;
    int ni, nk, nj;
};
struct PushArgs {
    Box box[4];
    int nbox;
    const unsigned *wait0, *wait1;      // wait until >= *epoch + index (the reader finished the previous step)
    unsigned *sig0, *sig1;              // then release *epoch + index + 1 to these (in the neighbours' memory)
    const unsigned *epoch;
    unsigned index;
    unsigned *done, *status;
    unsigned long long timeout_ns;
};

__global__ void __launch_bounds__(256) push_kernel(const __grid_constant__ PushArgs a)
{
    if (threadIdx.x == 0 && (a.wait0 || a.wait1)) {
        const unsigned want = *(volatile const unsigned *)a.epoch + a.index;
        if (a.wait0) wait_flag(a.wait0, want, a.status, a.timeout_ns);
        if (a.wait1) wait_flag(a.wait1, want, a.status, a.timeout_ns);
    }
    __syncthreads();
    for (int b = 0; b < a.nbox; ++b) {
        const Box &x = a.box[b];
        const long long n = (long long)x.ni * x.nk * x.nj;
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
             e += (long long)gridDim.x * blockDim.x) {
            const int i = (int)(e % x.ni);
            const long long r = e / x.ni;
            const int k = (int)(r % x.nk);
            const long long j = r / x.nk;
            x.dst[j * x.dj + k * x.dp + i] = x.src[j * x.sj + k * x.sp + i];       // NVLink store when dst is a peer
        }
    }
    if (a.sig0 || a.sig1) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();
            if (atomicAdd(a.done, 1u) == gridDim.x - 1u) {                          // last block of the launch
                __threadfence_system();
                *a.done = 0u;
                const unsigned v = *(volatile const unsigned *)a.epoch + a.index + 1u;
                if (a.sig0) st_release_sys(a.sig0, v);
                if (a.sig1) st_release_sys(a.sig1, v);
            }
        }
    }
}

// Behind every loop: move the epoch on by the number of steps the loop ran.
__global__ void epoch_kernel(unsigned *epoch, unsigned nsteps)
{
    if (threadIdx.x == 0) *(volatile unsigned *)epoch = *(volatile unsigned *)epoch + nsteps;
}

// stream-ordered wait for the west / south neighbours' outputs of the last completed step
__global__ void wait_outputs_kernel(const unsigned *w0, const unsigned *w1, const unsigned *epoch, unsigned done_index,
                                    unsigned *status, unsigned long long timeout_ns)
{
    const unsigned want = *(volatile const unsigned *)epoch + done_index;   // steps completed so far
    if (threadIdx.x == 0 && w0) wait_flag(w0, want, status, timeout_ns);
    if (threadIdx.x == 1 && w1) wait_flag(w1, want, status, timeout_ns);
}

// stream-ordered barrier with the (up to four) neighbours: everything this rank stored into their memory
// before this kernel (earlier launches on the stream) is visible to them once they pass their own barrier
struct BarrierArgs {
    unsigned *to[4];          // neighbour's slot for me (null: no neighbour on that side)
    const unsigned *from[4];  // my slot for the neighbour on that side
    unsigned epoch;
    unsigned *status;
    unsigned long long timeout_ns;
};
__global__ void barrier_kernel(const __grid_constant__ BarrierArgs a)
{
    const int s = threadIdx.x;
    if (s < 4 && a.to[s]) {
        __threadfence_system();
        st_release_sys(a.to[s], a.epoch);
        wait_flag(a.from[s], a.epoch, a.status, a.timeout_ns);
    }
}

// ---------------------------------------------------------------------------------------------------
// host helpers
// ---------------------------------------------------------------------------------------------------
// `verb` is the calling entry point.  typed: 4 for the verbs with a float argument, 8 for the _r8 verbs, 0 for the
// verbs without a floating-point argument, which serve a real*8 handle once wrfb200_comm_init_r8 made its comm state.
int need_comm(wrfb200_handle *h, bool connected, const char *verb, int typed = 0)
{
    if (!h) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null handle");
    if (typed == 8 && h->esize != 8)
        return wrfb200_fail(WRFB200_ERR_STATE, "%s: this is a real*4 handle (created by wrfb200_create); use the "
                            "binary32 verb without the _r8 suffix", verb);
    if (typed == 4)
        if (int rc = wrfb200_require_r4(h, verb)) return rc;
    if (!h->comm && h->esize == 8)
        return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "%s: the state of wrfb200_comm_init is binary32 only; a real*8 "
                            "handle needs wrfb200_comm_init_r8 first", verb);
    if (!h->comm) return wrfb200_fail(WRFB200_ERR_STATE, "wrfb200_comm_init has not been called on this handle");
    if (connected && !h->comm->connected) return wrfb200_fail(WRFB200_ERR_STATE, "wrfb200_comm_connect has not been called");
    return WRFB200_OK;
}

cudaError_t launch_push(const PushArgs &a, cudaStream_t s)
{
    long long n = 0;
    for (int b = 0; b < a.nbox; ++b) {
        const long long m = (long long)a.box[b].ni * a.box[b].nk * a.box[b].nj;
        if (m > n) n = m;
    }
    if (n <= 0) return cudaSuccess;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 4) blocks = 148 * 4;
    (void)cudaGetLastError();
    push_kernel<<<(unsigned)blocks, 256, 0, s>>>(a);
    return cudaGetLastError();
}

// The box of `field` that goes to the neighbour on `side`: this rank's edge column / row of the patch,
// addressed in both memories by its Fortran indices.  Boxes count 4-byte words: push_kernel moves a real*8 edge as
// pairs of words, bit for bit, with the extents and strides doubled.
Box edge_box(const wrfb200_handle *h, const Peer &pr, int field, int side)
{
    const int w = h->esize / 4;
    const wrfb200_comm *c = h->comm;
    const wrfb200_domain &d = h->dom;
    const CommInfo &q = pr.info;
    const bool f3 = is3(field);
    const int nk = f3 ? h->kdim : 1;
    const long long sp = f3 ? h->pitch3 : 0, sj = f3 ? h->pitch3 * (long long)h->kdim : h->pitch2;
    const long long dp = f3 ? q.pitch3 : 0, dj = f3 ? q.pitch3 * (long long)(q.kme - q.kms + 1) : q.pitch2;
    int i0, i1, j0, j1;
    switch (side) {
    case WRFB200_WEST:  i0 = i1 = c->ips; j0 = c->jps; j1 = c->jpe; break;
    case WRFB200_EAST:  i0 = i1 = c->ipe; j0 = c->jps; j1 = c->jpe; break;
    case WRFB200_SOUTH: j0 = j1 = c->jps; i0 = c->ips; i1 = c->ipe; break;
    default:            j0 = j1 = c->jpe; i0 = c->ips; i1 = c->ipe; break;
    }
    Box b{};
    b.src = h->d[field] + ((long long)(j0 - d.jms) * sj + (i0 - d.ims)) * w;
    b.dst = pr.f[field] + ((long long)(j0 + pr.dj - q.jms) * dj + (i0 + pr.di - q.ims)) * w;
    b.sp = sp * w; b.sj = sj * w; b.dp = dp * w; b.dj = dj * w;
    b.ni = (i1 - i0 + 1) * w; b.nk = nk; b.nj = j1 - j0 + 1;
    return b;
}

int close_ipc(wrfb200_comm *c)
{
    std::lock_guard<std::mutex> lock(ipc_mutex());
    auto &cache = ipc_cache();
    for (const std::string &k : c->opened) {
        auto it = cache.find(k);
        if (it == cache.end()) continue;
        if (--it->second.refs <= 0) {
            cudaIpcCloseMemHandle(it->second.base);
            cache.erase(it);
        }
    }
    c->opened.clear();
    (void)cudaGetLastError();
    return WRFB200_OK;
}

int map_peer(wrfb200_handle *h, Peer *pr)
{
    wrfb200_comm *c = h->comm;
    const CommInfo &q = pr->info;
    const bool same_process = (q.pid == (int)getpid() && q.host_id == host_id());
    if (q.host_id != host_id())
        return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "rank %d runs on another host: peer-mapped halos need one NVLink box", q.rank);
    for (int x = 0; x <= kNX; ++x) {
        void *mapped = nullptr;
        if (same_process) {
            mapped = (void *)(uintptr_t)q.ptr[x];
        } else {
            const std::string key((const char *)&q.ipc[x], sizeof(cudaIpcMemHandle_t));
            std::lock_guard<std::mutex> lock(ipc_mutex());
            auto &cache = ipc_cache();
            auto it = cache.find(key);
            if (it == cache.end()) {
                void *base = nullptr;
                cudaError_t e = cudaIpcOpenMemHandle(&base, q.ipc[x], cudaIpcMemLazyEnablePeerAccess);
                if (e != cudaSuccess) {
                    (void)cudaGetLastError();
                    return wrfb200_fail(WRFB200_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d, buffer %d) failed: %s", q.rank, x,
                                        cudaGetErrorString(e));
                }
                it = cache.emplace(key, OpenedIpc{base, 0}).first;
            }
            it->second.refs += 1;
            c->opened.push_back(key);
            mapped = (char *)it->second.base + q.offset[x];
        }
        if (x < kNX) pr->f[kXf[x]] = (float *)mapped;
        else pr->flags = (unsigned *)mapped;
    }
    if (same_process && q.device != h->device) {
        int can = 0;
        CUC(cudaDeviceCanAccessPeer(&can, h->device, q.device));
        if (!can) return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "device %d cannot access device %d", h->device, q.device);
        cudaError_t e = cudaDeviceEnablePeerAccess(q.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            return wrfb200_fail(WRFB200_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) failed: %s", q.device, cudaGetErrorString(e));
        (void)cudaGetLastError();
    }
    return WRFB200_OK;
}

// the advance_uv stand-in boxes of this patch: u over i_start+1..i_end, v over j_start+1..j_end of the
// GLOBAL computed range (tests/cases.py standin_boxes); on a wrapped axis from i_start / j_start, whose mudf at
// i-1 / j-1 is the wrapped ring
void standin_boxes(const wrfb200_handle *h, int ub[4], int vb[4])
{
    const wrfb200_domain &d = h->dom;
    const wrfb200_comm *c = h->comm;
    int gi0, gi1, gj0, gj1, k0, k1;
    wrfb200_bounds(d.periodic_x, d.specified, d.nested, d.ids, d.ide, d.jds, d.jde,
                   d.ids, d.ide, d.jds, d.jde, 1, d.kde, &gi0, &gi1, &gj0, &gj1, &k0, &k1);
    auto mx = [](int a, int b) { return a > b ? a : b; };
    auto mn = [](int a, int b) { return a < b ? a : b; };
    const int su = c->wrap_x ? 0 : 1, sv = c->wrap_y ? 0 : 1;
    ub[0] = mx(c->ips, gi0 + su); ub[1] = mn(c->ipe, gi1); ub[2] = mx(c->jps, gj0); ub[3] = mn(c->jpe, gj1);
    vb[0] = mx(c->ips, gi0); vb[1] = mn(c->ipe, gi1); vb[2] = mx(c->jps, gj0 + sv); vb[3] = mn(c->jpe, gj1);
}

int enqueue_push_uv(wrfb200_handle *h, cudaStream_t s, unsigned index)
{
    wrfb200_comm *c = h->comm;
    PushArgs a{};
    const Peer &w = c->peer[WRFB200_WEST];
    if (w.present) {
        a.box[a.nbox++] = edge_box(h, w, WRFB200_U, WRFB200_WEST);
        if (!w.self) {
            a.wait0 = c->flags + F_OUT_W;
            a.sig0 = w.flags + F_UV_E;
        }
    }
    // (the v south row goes to the south neighbour from inside advance_mu_t itself: its south-row blocks push it
    // before they start, amt_pipe.cu for binary32 and amt_tile_r8.cu for real*8 -- no separate launch for j-slab
    // decompositions.  A self south side cannot: its north-row blocks, which read that row, run in the same launch.)
    const Peer &so = c->peer[WRFB200_SOUTH];
    if (so.present && so.self) a.box[a.nbox++] = edge_box(h, so, WRFB200_V, WRFB200_SOUTH);
    if (a.nbox == 0) return WRFB200_OK;
    a.epoch = c->flags + F_EPOCH;
    a.index = index;
    a.done = c->flags + F_PUSH_DONE;
    a.status = c->flags + F_STATUS;
    a.timeout_ns = c->timeout_ns;
    cudaError_t e = launch_push(a, s);
    if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "u halo push launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    return WRFB200_OK;
}

int enqueue_wait_outputs(wrfb200_handle *h, cudaStream_t s, unsigned done_index)
{
    wrfb200_comm *c = h->comm;
    auto waits = [&](int side) { return c->peer[side].present && !c->peer[side].self; };   // a self side: stream order
    const unsigned *w0 = waits(WRFB200_WEST) ? c->flags + F_OUT_W : nullptr;
    const unsigned *w1 = waits(WRFB200_SOUTH) ? c->flags + F_OUT_S : nullptr;
    if (!w0 && !w1) return WRFB200_OK;
    (void)cudaGetLastError();
    wait_outputs_kernel<<<1, 32, 0, s>>>(w0, w1, c->flags + F_EPOCH, done_index, c->flags + F_STATUS, c->timeout_ns);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "halo wait launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
    return WRFB200_OK;
}

// binary32: the TMA pipe kernel; real*8: the fused tile kernel (amt_tile_r8.cu)
template <class P>
int enqueue_step_as(wrfb200_handle *h, cudaStream_t s, unsigned index)
{
    wrfb200_comm *c = h->comm;
    P p;
    bool empty = false;
    if (int rc = wrfb200_make_params(h, c->ips, c->ipe, c->jps, c->jpe, 1, h->dom.kde, &p, &empty)) return rc;
    if (empty) return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "rank %d: patch has no computed columns", c->rank);
    p.halo = c->halo;
    p.halo.step_index = index;
    return wrfb200_launch_params(h, p, s, WRFB200_KERNEL_PIPE);
}

int enqueue_step(wrfb200_handle *h, cudaStream_t s, unsigned index)
{
    return h->esize == 8 ? enqueue_step_as<AmtParamsR8>(h, s, index) : enqueue_step_as<AmtParams>(h, s, index);
}

int enqueue_epoch(wrfb200_handle *h, cudaStream_t s, unsigned nsteps)
{
    wrfb200_comm *c = h->comm;
    (void)cudaGetLastError();
    epoch_kernel<<<1, 32, 0, s>>>(c->flags + F_EPOCH, nsteps);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "epoch kernel launch failed: %s", cudaGetErrorString(err));
    h->launches += 1;
    return WRFB200_OK;
}

// cc: the caller's float (binary32 handle) or double (real*8 handle), exact in a double either way
int enqueue_standin(wrfb200_handle *h, cudaStream_t s, double cc, unsigned done_index)
{
    int ub[4], vb[4];
    standin_boxes(h, ub, vb);
    if (int rc = enqueue_wait_outputs(h, s, done_index)) return rc;          // the mudf halo the stand-in reads has arrived
    cudaStream_t keep = h->stream;
    h->stream = s;
    auto advance = [&](int field, const int *b) {
        return h->esize == 8 ? wrfb200_standin_advance_uv_r8(h, field, cc, b[0], b[1], b[2], b[3])
                             : wrfb200_standin_advance_uv(h, field, (float)cc, b[0], b[1], b[2], b[3]);
    };
    int rc = advance(WRFB200_U, ub);
    if (rc == WRFB200_OK) rc = advance(WRFB200_V, vb);
    h->stream = keep;
    return rc;
}

int enqueue_loop(wrfb200_handle *h, cudaStream_t s, int nsteps, int standin, double cc)
{
    for (int n = 0; n < nsteps; ++n) {
        if (int rc = enqueue_push_uv(h, s, (unsigned)n)) return rc;
        if (int rc = enqueue_step(h, s, (unsigned)n)) return rc;
        if (standin && n + 1 < nsteps)
            if (int rc = enqueue_standin(h, s, cc, (unsigned)n + 1u)) return rc;
    }
    return enqueue_epoch(h, s, (unsigned)nsteps);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
// exported
// ---------------------------------------------------------------------------------------------------
void wrfb200_comm_release(wrfb200_handle *h)
{
    if (!h || !h->comm) return;
    wrfb200_comm *c = h->comm;
    DevGuard g(h->device);
    for (auto &kv : c->graphs) cudaGraphExecDestroy(kv.second.exec);
    close_ipc(c);
    if (c->flags) cudaFree(c->flags);
    if (c->own_stream) {
        if (h->stream == c->own_stream) h->stream = nullptr;
        cudaStreamDestroy(c->own_stream);
    }
    (void)cudaGetLastError();
    delete c;
    h->comm = nullptr;
}

extern "C" int wrfb200_comm_info_bytes(void) { return WRFB200_COMM_INFO_BYTES; }

namespace {

// wrfb200_comm_init / _init_r8 after the precision checks
int comm_init(wrfb200_handle *h, int px, int py, int rank, int ips, int ipe, int jps, int jpe, void *info_out)
{
    if (px < 1 || py < 1 || rank < 0 || rank >= px * py)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "bad process grid %dx%d / rank %d", px, py, rank);
    const wrfb200_domain &d = h->dom;
    if (ips > ipe || jps > jpe || ips - 1 < d.ims || ipe + 1 > d.ime || jps - 1 < d.jms || jpe + 1 > d.jme)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG,
                            "patch i=%d..%d j=%d..%d needs a one-cell halo inside memory i=%d..%d j=%d..%d",
                            ips, ipe, jps, jpe, d.ims, d.ime, d.jms, d.jme);
    const int pi = rank % px, pj = rank / px;
    if (h->wrap_x) {
        if (!d.periodic_x)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "wrap_x needs a periodic_x domain");
        if ((pi == 0 && ips != d.ids) || (pi == px - 1 && (ipe != d.ide || ipe - 1 < ips)))
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "wrap_x: rank %d (i=%d..%d) must start at ids=%d when on the "
                                "west edge, and end at ide=%d with at least one computed column when on the east edge",
                                rank, ips, ipe, d.ids, d.ide);
    }
    if (h->wrap_y) {
        if (d.specified || d.nested)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "wrap_y needs specified == 0 and nested == 0: otherwise the "
                                "j range is clamped at the domain edge");
        if ((pj == 0 && jps != d.jds) || (pj == py - 1 && (jpe != d.jde || jpe - 1 < jps)))
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "wrap_y: rank %d (j=%d..%d) must start at jds=%d when on the "
                                "south edge, and end at jde=%d with at least one computed row when on the north edge",
                                rank, jps, jpe, d.jds, d.jde);
    }
    // on a wrapped axis the edge rank's column ide / row jde receives the wrap: it is halo to the exchange
    if (h->wrap_x && pi == px - 1) ipe = d.ide - 1;
    if (h->wrap_y && pj == py - 1) jpe = d.jde - 1;
    for (int x = 0; x < kNX; ++x)
        if (!h->d[kXf[x]] || !h->owned[kXf[x]])
            return wrfb200_fail(WRFB200_ERR_STATE, "field %d must be a handle-owned mirror (wrfb200_create with allocate=1): "
                                "neighbours map it through CUDA IPC", kXf[x]);
    DevGuard g(h->device);
    // whoever receives the info blob may store into this rank's arrays at once: earlier uploads must be done
    CUC(cudaStreamSynchronize(h->stream));
    wrfb200_comm_release(h);
    wrfb200_comm *c = new (std::nothrow) wrfb200_comm();
    if (!c) return wrfb200_fail(WRFB200_ERR_NOMEM, "out of host memory");
    h->comm = c;
    c->px = px; c->py = py; c->rank = rank; c->nranks = px * py;
    c->ips = ips; c->ipe = ipe; c->jps = jps; c->jpe = jpe;
    c->wrap_x = h->wrap_x; c->wrap_y = h->wrap_y;
    c->nbr[WRFB200_WEST] = pi > 0 ? rank - 1 : (c->wrap_x ? rank + px - 1 : -1);
    c->nbr[WRFB200_EAST] = pi + 1 < px ? rank + 1 : (c->wrap_x ? rank - px + 1 : -1);
    c->nbr[WRFB200_SOUTH] = pj > 0 ? rank - px : (c->wrap_y ? rank + px * (py - 1) : -1);
    c->nbr[WRFB200_NORTH] = pj + 1 < py ? rank + px : (c->wrap_y ? rank - px * (py - 1) : -1);
    if (const char *e = getenv("WRFB200_FLAG_TIMEOUT_MS")) {
        const long ms = atol(e);
        if (ms > 0) c->timeout_ns = (unsigned long long)ms * 1000000ull;
    }
    CUC(cudaMalloc(&c->flags, F_WORDS * sizeof(unsigned)));
    CUC(cudaMemset(c->flags, 0, F_WORDS * sizeof(unsigned)));
    if (!h->stream) {
        // ranks that share a device (tests) must not serialise on the legacy default stream: a waiting
        // kernel of one rank would block the neighbour's producer behind it
        CUC(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
        h->stream = c->own_stream;
    }

    CommInfo q{};
    q.magic = kMagic;
    q.rank = rank; q.px = px; q.py = py;
    q.pid = (int)getpid(); q.device = h->device; q.esize = h->esize; q.host_id = host_id();
    q.ims = d.ims; q.ime = d.ime; q.jms = d.jms; q.jme = d.jme; q.kms = d.kms; q.kme = d.kme;
    q.ips = ips; q.ipe = ipe; q.jps = jps; q.jpe = jpe;
    q.wrap_x = c->wrap_x; q.wrap_y = c->wrap_y;
    q.ids = d.ids; q.ide = d.ide; q.jds = d.jds; q.jde = d.jde;
    q.pitch3 = h->pitch3; q.pitch2 = h->pitch2;
    for (int x = 0; x <= kNX; ++x) {
        void *p = x < kNX ? (void *)h->d[kXf[x]] : (void *)c->flags;
        uint64_t base = (uint64_t)(uintptr_t)p;
        alloc_base(p, &base);
        q.ptr[x] = (uint64_t)(uintptr_t)p;
        q.offset[x] = (uint64_t)(uintptr_t)p - base;
        cudaError_t e = cudaIpcGetMemHandle(&q.ipc[x], (void *)(uintptr_t)base);
        if (e != cudaSuccess) {
            // not fatal: ranks inside one process do not need IPC; connect() reports it if they do
            (void)cudaGetLastError();
            std::memset(&q.ipc[x], 0, sizeof(q.ipc[x]));
        }
    }
    std::memset(info_out, 0, WRFB200_COMM_INFO_BYTES);
    std::memcpy(info_out, &q, sizeof(q));
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_comm_set_wrap(wrfb200_handle *h, int wrap_x, int wrap_y)
{
    if (!h) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null handle");
    h->wrap_x = wrap_x ? 1 : 0;
    h->wrap_y = wrap_y ? 1 : 0;
    return WRFB200_OK;
}

extern "C" int wrfb200_comm_init(wrfb200_handle *h, int px, int py, int rank,
                                 int ips, int ipe, int jps, int jpe, void *info_out)
{
    if (!h || !info_out) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (int rc = wrfb200_require_r4(h, "multi-GPU halo exchange (wrfb200_comm_*)")) return rc;
    // every step runs the TMA pipe kernel: refuse a level count it cannot hold now, before any neighbour connects,
    // rather than at the first step
    AmtParams p{};
    p.nk = h->dom.kde - 1;                                      // levels 1 .. kde-1
    int most = 0;
    if (!amt_pipe_levels_fit(p, &most))
        return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "the binary32 multi-GPU path runs the TMA pipe kernel, which holds "
                            "at most %d levels (nk=%d)", most, p.nk);
    return comm_init(h, px, py, rank, ips, ipe, jps, jpe, info_out);
}

extern "C" int wrfb200_comm_init_r8(wrfb200_handle *h, int px, int py, int rank,
                                    int ips, int ipe, int jps, int jpe, void *info_out)
{
    if (!h || !info_out) return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "null argument");
    if (h->esize != 8)
        return wrfb200_fail(WRFB200_ERR_STATE, "wrfb200_comm_init_r8: this is a real*4 handle (created by "
                            "wrfb200_create); use wrfb200_comm_init");
    // every step runs the fused tile kernel: refuse a patch it cannot take now rather than at the first step.
    // Handle-owned mirrors are 128-byte aligned with even pitches, so the level count is what can fail.
    AmtParamsR8 p{};
    wrfb200_fill_fields(h, &p);
    p.nk = h->dom.kde - 1;                                      // levels 1 .. kde-1
    if (!amt_tile_supported(p))
        return wrfb200_fail(WRFB200_ERR_UNSUPPORTED, "the real*8 multi-GPU path runs the double2 tile kernel, which "
                            "needs 16-byte aligned fields, pitches of an even number of doubles and at most 220 levels "
                            "(this patch computes %d)", p.nk);
    return comm_init(h, px, py, rank, ips, ipe, jps, jpe, info_out);
}

extern "C" int wrfb200_comm_connect(wrfb200_handle *h, const void *all_infos, int nranks)
{
    if (int rc = need_comm(h, false, "wrfb200_comm_connect")) return rc;
    wrfb200_comm *c = h->comm;
    if (!all_infos || nranks != c->nranks)
        return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "expected the info blobs of all %d ranks, in rank order", c->nranks);
    DevGuard g(h->device);
    // Every kernel of the loop is loaded NOW: a lazy load at first launch can wait for the device to drain,
    // and a kernel already running may itself be waiting on a flag for work this thread has yet to launch.
    {
        cudaFuncAttributes fa;
        CUC(cudaFuncGetAttributes(&fa, (const void *)push_kernel));
        CUC(cudaFuncGetAttributes(&fa, (const void *)wait_outputs_kernel));
        CUC(cudaFuncGetAttributes(&fa, (const void *)barrier_kernel));
        CUC(cudaFuncGetAttributes(&fa, (const void *)epoch_kernel));
        CUC(wrfb200_halo_preload());
        if (h->esize == 8) CUC(amt_tile_r8_preload());
        else CUC(amt_pipe_preload());
    }
    const wrfb200_domain &d = h->dom;
    const int kdim = h->kdim;
    for (int side = 0; side < 4; ++side) {
        Peer &pr = c->peer[side];
        pr = Peer{};
        if (c->nbr[side] < 0) continue;
        std::memcpy(&pr.info, (const char *)all_infos + (size_t)c->nbr[side] * WRFB200_COMM_INFO_BYTES, sizeof(CommInfo));
        const CommInfo &q = pr.info;
        if (q.magic != kMagic || q.rank != c->nbr[side] || q.px != c->px || q.py != c->py)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "info blob %d is not rank %d of a %dx%d grid", c->nbr[side], c->nbr[side], c->px, c->py);
        if (q.esize != h->esize)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "rank %d holds %s data and this rank %s: ranks of mixed "
                                "precision are not supported", q.rank, q.esize == 8 ? "real*8" : "binary32",
                                h->esize == 8 ? "real*8" : "binary32");
        if (q.kms != d.kms || q.kme - q.kms + 1 != kdim)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "rank %d has different vertical memory extents", q.rank);
        if (q.wrap_x != c->wrap_x || q.wrap_y != c->wrap_y || q.ids != d.ids || q.ide != d.ide || q.jds != d.jds ||
            q.jde != d.jde)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "rank %d has wrap (%d,%d) on i=%d..%d j=%d..%d, this rank (%d,%d) "
                                "on i=%d..%d j=%d..%d: all ranks must set the same wrap on the same domain", q.rank,
                                q.wrap_x, q.wrap_y, q.ids, q.ide, q.jds, q.jde, c->wrap_x, c->wrap_y, d.ids, d.ide,
                                d.jds, d.jde);
        // across the domain edge the peer's index of my cell is shifted by the period
        const int pi = c->rank % c->px, pj = c->rank / c->px;
        if (side == WRFB200_WEST && pi == 0) pr.di = d.ide - d.ids;
        if (side == WRFB200_EAST && pi == c->px - 1) pr.di = -(d.ide - d.ids);
        if (side == WRFB200_SOUTH && pj == 0) pr.dj = d.jde - d.jds;
        if (side == WRFB200_NORTH && pj == c->py - 1) pr.dj = -(d.jde - d.jds);
        const int ips = c->ips + pr.di, ipe = c->ipe + pr.di, jps = c->jps + pr.dj, jpe = c->jpe + pr.dj;
        bool adjacent = false;
        switch (side) {
        case WRFB200_WEST:  adjacent = q.ipe + 1 == ips && q.jps == jps && q.jpe == jpe && q.ime >= ips; break;
        case WRFB200_EAST:  adjacent = q.ips - 1 == ipe && q.jps == jps && q.jpe == jpe && q.ims <= ipe; break;
        case WRFB200_SOUTH: adjacent = q.jpe + 1 == jps && q.ips == ips && q.ipe == ipe && q.jme >= jps; break;
        default:            adjacent = q.jps - 1 == jpe && q.ips == ips && q.ipe == ipe && q.jms <= jpe; break;
        }
        if (!adjacent)
            return wrfb200_fail(WRFB200_ERR_INVALID_ARG, "rank %d (i=%d..%d j=%d..%d) is not the side-%d neighbour of i=%d..%d j=%d..%d",
                                q.rank, q.ips, q.ipe, q.jps, q.jpe, side, c->ips, c->ipe, c->jps, c->jpe);
        if (int rc = map_peer(h, &pr)) return rc;
        pr.present = true;
        pr.self = c->nbr[side] == c->rank;
    }

    // peer addresses: element offsets into the neighbour's arrays, scaled to 4-byte words (the kernels read the
    // float pointers of AmtHalo as double pointers on a real*8 rank; pitches stay in elements)
    const int w = h->esize / 4;
    AmtHalo hx{};
    hx.enabled = 1;
    hx.ipe_mem = c->ipe - d.ims;
    hx.jpe_mem = c->jpe - d.jms;
    hx.ips_mem = c->ips - d.ims;
    hx.jps_mem = c->jps - d.jms;
    // A self side keeps the output stores (into this rank's own ring, read by later launches only) and drops every
    // flag: its u / v edge is copied by push_kernel ahead of the step (enqueue_push_uv).
    const Peer &so = c->peer[WRFB200_SOUTH];
    if (so.present && !so.self) {
        const CommInfo &q = so.info;
        // south neighbour's v at (my memory column 0, level 0, Fortran row jps = its north halo row)
        hx.s_v = so.f[WRFB200_V] + ((long long)(c->jps + so.dj - q.jms) * (q.kme - q.kms + 1) * q.pitch3 +
                                    (d.ims + so.di - q.ims)) * w;
        hx.s_pitch3 = q.pitch3;
        hx.war_flag_south = c->flags + F_OUT_S;
        hx.uv_flag_to_south = so.flags + F_UV_N;
        hx.push_counter = c->flags + F_VPUSH_DONE;
    }
    const Peer &e = c->peer[WRFB200_EAST], &n = c->peer[WRFB200_NORTH];
    if (e.present) {
        const CommInfo &q = e.info;
        // my memory row 0, column ipe
        const long long o = ((long long)(d.jms + e.dj - q.jms) * q.pitch2 + (c->ipe + e.di - q.ims)) * w;
        hx.e_mu = e.f[WRFB200_MU] + o; hx.e_muts = e.f[WRFB200_MUTS] + o; hx.e_mudf = e.f[WRFB200_MUDF] + o;
        hx.e_pitch2 = q.pitch2;
    }
    if (n.present) {
        const CommInfo &q = n.info;
        // row jpe, my memory column 0
        const long long o = ((long long)(c->jpe + n.dj - q.jms) * q.pitch2 + (d.ims + n.di - q.ims)) * w;
        hx.n_mu = n.f[WRFB200_MU] + o; hx.n_muts = n.f[WRFB200_MUTS] + o; hx.n_mudf = n.f[WRFB200_MUDF] + o;
    }
    if (e.present && !e.self) {
        hx.uv_flag_east = c->flags + F_UV_E;
        hx.out_flag_to_east = e.flags + F_OUT_W; hx.east_counter = c->flags + F_EAST_DONE;
    }
    if (n.present && !n.self) {
        hx.uv_flag_north = c->flags + F_UV_N;
        hx.out_flag_to_north = n.flags + F_OUT_S; hx.north_counter = c->flags + F_NORTH_DONE;
    }
    hx.epoch = c->flags + F_EPOCH;
    {
        const char *e = getenv("WRFB200_NORTH_SECOND");               // A/B switch; default on
        hx.north_second = (e && atoi(e) == 0) ? 0 : 1;
    }
    hx.status = c->flags + F_STATUS;
    hx.timeout_ns = c->timeout_ns;
    c->halo = hx;
    for (auto &kv : c->graphs) cudaGraphExecDestroy(kv.second.exec);
    c->graphs.clear();
    c->connected = true;
    return WRFB200_OK;
}

extern "C" int wrfb200_comm_barrier(wrfb200_handle *h)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_barrier")) return rc;
    wrfb200_comm *c = h->comm;
    DevGuard g(h->device);
    BarrierArgs a{};
    bool any = false;
    for (int side = 0; side < 4; ++side) {
        if (!c->peer[side].present || c->peer[side].self) continue;    // stream order covers a self side
        a.to[side] = c->peer[side].flags + F_BAR + opposite(side);
        a.from[side] = c->flags + F_BAR + side;
        any = true;
    }
    if (!any) return WRFB200_OK;
    a.epoch = ++c->bar_epoch;
    a.status = c->flags + F_STATUS;
    a.timeout_ns = c->timeout_ns;
    (void)cudaGetLastError();
    barrier_kernel<<<1, 32, 0, h->stream>>>(a);
    CUC(cudaGetLastError());
    h->launches += 1;
    return WRFB200_OK;
}

extern "C" int wrfb200_comm_push_constants(wrfb200_handle *h)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_push_constants")) return rc;
    wrfb200_comm *c = h->comm;
    DevGuard g(h->device);
    // (field, side the edge goes to): what advance_mu_t reads across a patch edge and nobody changes inside
    // the acoustic loop -- u_1, muu, msfuy at i+1; v_1, muv, msfvx_inv at j+1; t_1 on all four sides
    static const int plan[][2] = {
        {WRFB200_U_1, WRFB200_WEST}, {WRFB200_MUU, WRFB200_WEST}, {WRFB200_MSFUY, WRFB200_WEST}, {WRFB200_T_1, WRFB200_WEST},
        {WRFB200_V_1, WRFB200_SOUTH}, {WRFB200_MUV, WRFB200_SOUTH}, {WRFB200_MSFVX_INV, WRFB200_SOUTH}, {WRFB200_T_1, WRFB200_SOUTH},
        {WRFB200_T_1, WRFB200_EAST}, {WRFB200_T_1, WRFB200_NORTH}};
    // neighbours may still be uploading the arrays this rank is about to store into: meet them first
    if (int rc = wrfb200_comm_barrier(h)) return rc;
    PushArgs a{};
    auto flush = [&]() -> int {
        if (a.nbox == 0) return WRFB200_OK;
        cudaError_t e = launch_push(a, h->stream);
        if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "constant halo push launch failed: %s", cudaGetErrorString(e));
        h->launches += 1;
        a = PushArgs{};
        return WRFB200_OK;
    };
    for (const auto &fs : plan) {
        const Peer &pr = c->peer[fs[1]];
        if (!pr.present) continue;
        a.box[a.nbox++] = edge_box(h, pr, fs[0], fs[1]);
        if (a.nbox == 4) if (int rc = flush()) return rc;
    }
    if (int rc = flush()) return rc;
    return wrfb200_comm_barrier(h);
}

extern "C" int wrfb200_comm_push_uv(wrfb200_handle *h)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_push_uv")) return rc;
    DevGuard g(h->device);
    return enqueue_push_uv(h, h->stream, 0u);
}

extern "C" int wrfb200_comm_wait_outputs(wrfb200_handle *h)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_wait_outputs")) return rc;
    DevGuard g(h->device);
    return enqueue_wait_outputs(h, h->stream, 0u);     // the epoch already counts every completed step here
}

extern "C" int wrfb200_comm_step(wrfb200_handle *h)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_step")) return rc;
    DevGuard g(h->device);
    if (int rc = enqueue_step(h, h->stream, 0u)) return rc;
    return enqueue_epoch(h, h->stream, 1u);
}

extern "C" int wrfb200_comm_standin_advance_uv(wrfb200_handle *h, float c)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_standin_advance_uv", 4)) return rc;
    DevGuard g(h->device);
    return enqueue_standin(h, h->stream, c, 0u);
}

extern "C" int wrfb200_comm_standin_advance_uv_r8(wrfb200_handle *h, double c)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_standin_advance_uv_r8", 8)) return rc;
    DevGuard g(h->device);
    return enqueue_standin(h, h->stream, c, 0u);
}

namespace {

// wrfb200_comm_loop / _loop_r8 after the checks; cc is the caller's float or double, held exactly
int comm_loop(wrfb200_handle *h, int nsteps, int standin, double cc, int use_graph)
{
    if (nsteps <= 0) return WRFB200_OK;
    wrfb200_comm *c = h->comm;
    DevGuard g(h->device);
    if (!use_graph) return enqueue_loop(h, h->stream, nsteps, standin, cc);
    unsigned long long cbits;
    std::memcpy(&cbits, &cc, 8);
    const auto key = std::make_tuple(nsteps, standin ? 1 : 0, standin ? cbits : 0ull);
    auto it = c->graphs.find(key);
    if (it == c->graphs.end()) {
        cudaStream_t cs;
        CUC(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        const long before = h->launches;
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        int rc = WRFB200_OK;
        if (e == cudaSuccess) {
            rc = enqueue_loop(h, cs, nsteps, standin, cc);
            e = cudaStreamEndCapture(cs, &graph);
        }
        cudaStreamDestroy(cs);
        const long per_replay = h->launches - before;      // counted again on every replay below
        h->launches = before;
        if (rc != WRFB200_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
        cudaGraphExec_t exec = nullptr;
        e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return wrfb200_fail(WRFB200_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
        it = c->graphs.emplace(key, wrfb200_comm::LoopGraph{exec, per_replay}).first;
    }
    CUC(cudaGraphLaunch(it->second.exec, h->stream));
    h->launches += it->second.launches;
    return WRFB200_OK;
}

}  // namespace

extern "C" int wrfb200_comm_loop(wrfb200_handle *h, int nsteps, int standin, float cc, int use_graph)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_loop", 4)) return rc;
    return comm_loop(h, nsteps, standin, cc, use_graph);
}

extern "C" int wrfb200_comm_loop_r8(wrfb200_handle *h, int nsteps, int standin, double cc, int use_graph)
{
    if (int rc = need_comm(h, true, "wrfb200_comm_loop_r8", 8)) return rc;
    return comm_loop(h, nsteps, standin, cc, use_graph);
}

extern "C" int wrfb200_comm_status(wrfb200_handle *h, int *flag_timeouts, long *steps_done)
{
    if (int rc = need_comm(h, false, "wrfb200_comm_status")) return rc;
    wrfb200_comm *c = h->comm;
    DevGuard g(h->device);
    unsigned host[F_WORDS];
    CUC(cudaStreamSynchronize(h->stream));
    CUC(cudaMemcpy(host, c->flags, sizeof(host), cudaMemcpyDeviceToHost));
    if (flag_timeouts) *flag_timeouts = (int)host[F_STATUS];
    if (steps_done) *steps_done = (long)host[F_EPOCH];
    return WRFB200_OK;
}
