// capi_internal.h -- the handle layout shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <tuple>

#include "../../include/wrfb200.h"
#include "amt_params.h"

struct wrfb200_comm;                   // comm.cu: peer-mapped halo exchange state of a multi-GPU patch

struct wrfb200_handle {
    wrfb200_domain dom{};
    int device = 0;
    cudaStream_t stream = nullptr;
    int esize = 4;                     // bytes per element: 4 (wrfb200_create) or 8 (wrfb200_create_r8)
    float *d[WRFB200_NUM_FIELDS] = {};   // device fields; they hold doubles when esize == 8
    bool owned[WRFB200_NUM_FIELDS] = {};
    long pitch3 = 0, pitch2 = 0;       // row strides in elements (0 = not yet known)
    int idim = 0, jdim = 0, kdim = 0;
    double rdx = 0, rdy = 0, dts = 0, epssm = 0;   // exact for either precision
    bool scalars_set = false;
    int kernel = WRFB200_KERNEL_AUTO;
    long launches = 0;
    int last_kernel = 0;               // wrfb200_kernel id of the most recent launch (AUTO resolved)
    AmtTmaMaps maps{};                 // tensor maps of the TMA kernel, rebuilt when the fields move
    // graphs keyed by (its, ite, jts, jte, kte, nsteps, kernel)
    std::map<std::tuple<int, int, int, int, int, int, int>, cudaGraphExec_t> graphs;
    wrfb200_comm *comm = nullptr;      // non-null after wrfb200_comm_init
    int wrap_x = 0, wrap_y = 0;        // periodic exchange across the domain edge (wrfb200_comm_set_wrap)
};

// capi.cu: kernel argument block for a tile / kernel launch (shared with comm.cu)
int wrfb200_make_params(const wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                        AmtParams *out, bool *empty);
int wrfb200_launch_params(wrfb200_handle *h, const AmtParams &p, cudaStream_t s, int kernel);
// ... and their real*8 twins (a block with p.halo.enabled runs the fused tile kernel whatever `kernel` says)
int wrfb200_make_params(const wrfb200_handle *h, int its, int ite, int jts, int jte, int kts, int kte,
                        AmtParamsR8 *out, bool *empty);
int wrfb200_launch_params(wrfb200_handle *h, const AmtParamsR8 &p, cudaStream_t s, int kernel);
// the handle's field pointers and strides into *p, whose element type must be the handle's (AmtParams or AmtParamsR8)
template <class P>
void wrfb200_fill_fields(const wrfb200_handle *h, P *p);
// comm.cu: called by wrfb200_destroy
void wrfb200_comm_release(wrfb200_handle *h);

// halo.cu: dense device rows -> pitched mirror rows
cudaError_t wrfb200_repitch_rows(float *dst, const float *src, long long pitch, int ni, long long nrows,
                                 cudaStream_t stream);

cudaError_t wrfb200_halo_preload();

// thread-local error message; returns `code`
int wrfb200_fail(int code, const char *fmt, ...);
// WRFB200_OK for a binary32 handle; WRFB200_ERR_UNSUPPORTED naming `what` for a real*8 one
int wrfb200_require_r4(const wrfb200_handle *h, const char *what);
