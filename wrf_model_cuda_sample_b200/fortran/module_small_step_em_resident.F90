!-----------------------------------------------------------------------------------------------------------
! module_small_step_em_resident.F90 -- ISO_C_BINDING interfaces of the DEVICE-RESIDENT and MULTI-GPU entry
! points of libwrfb200.so (include/wrfb200.h sections 1, 2, 3 and 3b), for a Fortran host that wants more than
! the one-call drop-in of module_small_step_em.F90:
!
!   (A) acoustic-loop residency with the UNCHANGED 48-argument call (smallest source change in solve_em):
!           CALL wrfb200_loop_begin()
!           DO iteration = 1, number_of_small_timesteps
!              CALL advance_uv( ... )                       ! host code, changes u, v only
!              CALL advance_mu_t( ww, ww1, u_2, ... )       ! module_small_step_em.F90 -> wrfb200_advance_mu_t
!           END DO
!           CALL wrfb200_loop_end()
!       The first call of the loop uploads all 26 arrays, later calls only u and v; every call downloads the
!       seven outputs.  Replaces the reference's H2D copy of every array on every call
!       (advance_mu_t_no_async.cu:245-306).
!
!   (B) an explicit patch handle with the three cadences spelled out (wrfb200_create, wrfb200_upload_constants
!       + wrfb200_upload_state once per RK sub-step, then per small step wrfb200_set_uv / wrfb200_step /
!       wrfb200_download_outputs) -- what replaces the allocate/copy/launch/copy/free body of
!       advance_mu_t_no_async.cu:178-423.
!
!   (C) one MPI rank per GPU: wrfb200_comm_init -> MPI_Allgather of the WRFB200_COMM_INFO_BYTES blobs ->
!       wrfb200_comm_connect, then per RK sub-step wrfb200_comm_push_constants and per small step
!       wrfb200_comm_push_uv + wrfb200_comm_step (or wrfb200_comm_loop for the whole loop).  Replaces the
!       j-slab plan and per-device launch loop of advance_mu_t_no_async.cu:87-162, :329-357.  Sketch:
!
!           TYPE(c_ptr) :: h
!           CHARACTER(KIND=c_char), TARGET :: mine(WRFB200_COMM_INFO_BYTES), everyone(WRFB200_COMM_INFO_BYTES*nproc)
!           st = wrfb200_create( h, dom, MOD(myrank, gpus_per_node), 1_c_int )
!           ...uploads...
!           st = wrfb200_comm_init( h, px, py, myrank, ips, ipe, jps, jpe, C_LOC(mine) )
!           CALL MPI_Allgather( mine, WRFB200_COMM_INFO_BYTES, MPI_BYTE, everyone, WRFB200_COMM_INFO_BYTES, MPI_BYTE, comm, ierr )
!           st = wrfb200_comm_connect( h, C_LOC(everyone), nproc )
!           st = wrfb200_comm_push_constants( h )
!           st = wrfb200_comm_loop( h, number_of_small_timesteps, 0_c_int, 0.0_c_float, 1_c_int )
!
!       A periodic domain refreshes its ring inside the loop only when the exchange wraps across the domain
!       edge: set it from the namelist before comm_init (wrap_y needs specified = nested = .FALSE.), with the
!       patches of WRF's own decomposition (the east-edge rank ends at ide, the north-edge rank at jde):
!
!           st = wrfb200_comm_set_wrap( h, MERGE(1_c_int, 0_c_int, config_flags%periodic_x),               &
!                                          MERGE(1_c_int, 0_c_int, config_flags%periodic_y) )
!
!       In a build configured with -r8 the same sequence uses the real*8 patch (section (B') below): create_r8,
!       the _r8 uploads, comm_init_r8 and comm_loop_r8; connect, push_constants, push_uv, step and status are
!       shared by both precisions.  All ranks must be built alike (connect rejects a rank of the other precision):
!
!           st = wrfb200_create_r8( h, dom, MOD(myrank, gpus_per_node), 1_c_int )
!           st = wrfb200_set_scalars_r8( h, rdx, rdy, dts, epssm )
!           st = wrfb200_upload_constants_r8( h, ww1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend, &
!                                             msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw )
!           st = wrfb200_upload_state_r8( h, ww, t_2, mu_2 )
!           st = wrfb200_set_uv_r8( h, u_2, v_2 )
!           st = wrfb200_comm_init_r8( h, px, py, myrank, ips, ipe, jps, jpe, C_LOC(mine) )
!           CALL MPI_Allgather( mine, WRFB200_COMM_INFO_BYTES, MPI_BYTE, everyone, WRFB200_COMM_INFO_BYTES, MPI_BYTE, comm, ierr )
!           st = wrfb200_comm_connect( h, C_LOC(everyone), nproc )
!           st = wrfb200_comm_push_constants( h )
!           st = wrfb200_comm_loop_r8( h, number_of_small_timesteps, 0_c_int, 0.0_c_double, 1_c_int )
!
!   (D) ranks on several hosts, or any transport of the caller's own (WRF's MPI): pack the edge a neighbour
!       needs into a dense DEVICE buffer, move it, unpack it into the halo (include/wrfb200.h section 3;
!       INTEGRATION.md section 4).  -r8 builds use the _r8 pair with REAL(c_double) buffers:
!
!           ! u's east halo: this rank's west column goes west, the east neighbour's west column arrives
!           ! (field 2 = u, side 0 = west, 1 = east; send_buf, recv_buf: n = 1*nk*(jpe-jps+1) doubles on the device)
!           st = wrfb200_pack_halo_r8( h, 2_c_int, 0_c_int, 1_c_int, ips, ipe, jps, jpe, C_LOC(send_buf) )
!           st = wrfb200_sync( h )                                  ! the pack runs on the handle's stream
!           CALL MPI_Sendrecv( send_buf, n, MPI_DOUBLE_PRECISION, west, 0, recv_buf, n, MPI_DOUBLE_PRECISION,  &
!                              east, 0, comm, stat, ierr )          ! CUDA-aware MPI
!           st = wrfb200_unpack_halo_r8( h, 2_c_int, 1_c_int, 1_c_int, ips, ipe, jps, jpe, C_LOC(recv_buf) )
!
! Source only: no Fortran compiler exists in the build image (INTEGRATION.md); tests/c_abi_harness.c,
! tests/c_comm_harness.c and tests/c_comm_harness_r8.c drive exactly these entry points from C, and tests/test_cabi_host.py checks that every
! NAME= below is an exported symbol of the built library.
!-----------------------------------------------------------------------------------------------------------
MODULE module_small_step_em_resident

USE, INTRINSIC :: iso_c_binding, ONLY : c_float, c_double, c_int, c_long, c_ptr, c_size_t

IMPLICIT NONE
PUBLIC

INTEGER, PARAMETER :: WRFB200_COMM_INFO_BYTES = 2048

! struct wrfb200_domain (include/wrfb200.h)
TYPE, BIND(C) :: wrfb200_domain
   INTEGER(c_int) :: ids, ide, jds, jde, kde
   INTEGER(c_int) :: ims, ime, jms, jme, kms, kme
   INTEGER(c_int) :: periodic_x, specified, nested
END TYPE wrfb200_domain

INTERFACE
   ! ---- (A) acoustic-loop residency of the 48-argument call ----
   FUNCTION wrfb200_acoustic_loop_begin() BIND(C, NAME="wrfb200_acoustic_loop_begin") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_acoustic_loop_end() BIND(C, NAME="wrfb200_acoustic_loop_end") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_set_host_pinning(enable) BIND(C, NAME="wrfb200_set_host_pinning") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int), VALUE :: enable
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_host_register(host, bytes) BIND(C, NAME="wrfb200_host_register") RESULT(status)
      IMPORT :: c_int, c_float, c_size_t
      REAL(c_float), DIMENSION(*), INTENT(IN) :: host
      INTEGER(c_size_t), VALUE :: bytes
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_release_cache() BIND(C, NAME="wrfb200_release_cache") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int) :: status
   END FUNCTION
   ! how this thread's last advance_mu_t call moved its arrays: 0 all direct (page-locked), 1 some staged through
   ! the library's pinned bounce buffers (pageable), 2 all staged
   FUNCTION wrfb200_default_last_transfer(route) BIND(C, NAME="wrfb200_default_last_transfer") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int), INTENT(OUT) :: route
      INTEGER(c_int) :: status
   END FUNCTION
   ! OpenMP builds (smpar, dm+sm): the tiles of the !$OMP PARALLEL DO share one device-resident patch.  Call once,
   ! after the rank has picked its GPU; the loop begin / end and the per-tile advance_mu_t calls are unchanged
   ! (INTEGRATION.md section 1)
   FUNCTION wrfb200_set_shared_tiles(enable) BIND(C, NAME="wrfb200_set_shared_tiles") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int), VALUE :: enable
      INTEGER(c_int) :: status
   END FUNCTION
   ! the host-array call split over several GPUs of the box: call once at start-up (e.g. ids 0..7 on an
   ! 8-GPU box), the advance_mu_t call itself is unchanged
   FUNCTION wrfb200_set_default_devices(devices, n) BIND(C, NAME="wrfb200_set_default_devices") RESULT(status)
      IMPORT :: c_int
      INTEGER(c_int), DIMENSION(*), INTENT(IN) :: devices
      INTEGER(c_int), VALUE :: n
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_host_split_plan(dom, its, ite, jts, jte, kts, kte, n, rows4)                      &
            BIND(C, NAME="wrfb200_host_split_plan") RESULT(status)
      IMPORT :: c_int, wrfb200_domain
      TYPE(wrfb200_domain), INTENT(IN) :: dom
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte, n
      INTEGER(c_int), DIMENSION(*), INTENT(OUT) :: rows4
      INTEGER(c_int) :: status
   END FUNCTION

   ! ---- (B) explicit device-resident patch ----
   FUNCTION wrfb200_create(handle, dom, device, allocate) BIND(C, NAME="wrfb200_create") RESULT(status)
      IMPORT :: c_int, c_ptr, wrfb200_domain
      TYPE(c_ptr), INTENT(OUT) :: handle
      TYPE(wrfb200_domain), INTENT(IN) :: dom
      INTEGER(c_int), VALUE :: device, allocate
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_destroy(handle) BIND(C, NAME="wrfb200_destroy") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_set_scalars(handle, rdx, rdy, dts, epssm) BIND(C, NAME="wrfb200_set_scalars") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      REAL(c_float), VALUE :: rdx, rdy, dts, epssm
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_upload_constants(handle, ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend,        &
                                     msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw)           &
            BIND(C, NAME="wrfb200_upload_constants") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      REAL(c_float), DIMENSION(*), INTENT(IN) :: ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend
      REAL(c_float), DIMENSION(*), INTENT(IN) :: msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_upload_state(handle, ww, t, mu) BIND(C, NAME="wrfb200_upload_state") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      REAL(c_float), DIMENSION(*), INTENT(IN) :: ww, t, mu
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_set_uv(handle, u, v) BIND(C, NAME="wrfb200_set_uv") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      REAL(c_float), DIMENSION(*), INTENT(IN) :: u, v
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_step(handle, its, ite, jts, jte, kts, kte) BIND(C, NAME="wrfb200_step") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_step_graph(handle, its, ite, jts, jte, kts, kte, nsteps)                          &
            BIND(C, NAME="wrfb200_step_graph") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte, nsteps
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_download_outputs(handle, its, ite, jts, jte, kts, kte,                            &
                                     ww, t, t_ave, mu, muave, muts, mudf)                            &
            BIND(C, NAME="wrfb200_download_outputs") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte
      REAL(c_float), DIMENSION(*), INTENT(INOUT) :: ww, t, t_ave, mu, muave, muts, mudf
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_sync(handle) BIND(C, NAME="wrfb200_sync") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION

   ! ---- (B') the same patch in double precision (WRF built with -r8); step / step_graph / sync / destroy
   !      above work on it too.  Field ids: enum wrfb200_field of include/wrfb200.h.
   FUNCTION wrfb200_create_r8(handle, dom, device, allocate) BIND(C, NAME="wrfb200_create_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, wrfb200_domain
      TYPE(c_ptr), INTENT(OUT) :: handle
      TYPE(wrfb200_domain), INTENT(IN) :: dom
      INTEGER(c_int), VALUE :: device, allocate
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_set_scalars_r8(handle, rdx, rdy, dts, epssm) BIND(C, NAME="wrfb200_set_scalars_r8")      &
            RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      REAL(c_double), VALUE :: rdx, rdy, dts, epssm
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_upload_r8(handle, field, host) BIND(C, NAME="wrfb200_upload_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field
      REAL(c_double), DIMENSION(*), INTENT(IN) :: host
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_download_r8(handle, field, host) BIND(C, NAME="wrfb200_download_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field
      REAL(c_double), DIMENSION(*), INTENT(INOUT) :: host
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_upload_range_r8(handle, field, host, i0, i1, k0, k1, j0, j1)                       &
            BIND(C, NAME="wrfb200_upload_range_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, i0, i1, k0, k1, j0, j1
      REAL(c_double), DIMENSION(*), INTENT(IN) :: host
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_download_range_r8(handle, field, host, i0, i1, k0, k1, j0, j1)                     &
            BIND(C, NAME="wrfb200_download_range_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, i0, i1, k0, k1, j0, j1
      REAL(c_double), DIMENSION(*), INTENT(INOUT) :: host
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_bind_device_r8(handle, field, device_ptr, pitch) BIND(C, NAME="wrfb200_bind_device_r8") &
            RESULT(status)
      IMPORT :: c_int, c_long, c_ptr
      TYPE(c_ptr), VALUE :: handle, device_ptr
      INTEGER(c_int), VALUE :: field
      INTEGER(c_long), VALUE :: pitch
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_device_ptr_r8(handle, field, device_ptr, pitch) BIND(C, NAME="wrfb200_device_ptr_r8")    &
            RESULT(status)
      IMPORT :: c_int, c_long, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field
      TYPE(c_ptr), INTENT(OUT) :: device_ptr
      INTEGER(c_long), INTENT(OUT) :: pitch
      INTEGER(c_int) :: status
   END FUNCTION

   FUNCTION wrfb200_upload_constants_r8(handle, ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend,     &
                                        msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw)        &
            BIND(C, NAME="wrfb200_upload_constants_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      REAL(c_double), DIMENSION(*), INTENT(IN) :: ww_1, u_1, v_1, t_1, ft, mut, muu, muv, mu_tend
      REAL(c_double), DIMENSION(*), INTENT(IN) :: msfuy, msfvx_inv, msftx, msfty, dnw, fnm, fnp, rdnw
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_upload_state_r8(handle, ww, t, mu) BIND(C, NAME="wrfb200_upload_state_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      REAL(c_double), DIMENSION(*), INTENT(IN) :: ww, t, mu
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_set_uv_r8(handle, u, v) BIND(C, NAME="wrfb200_set_uv_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      REAL(c_double), DIMENSION(*), INTENT(IN) :: u, v
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_download_outputs_r8(handle, its, ite, jts, jte, kts, kte,                         &
                                        ww, t, t_ave, mu, muave, muts, mudf)                         &
            BIND(C, NAME="wrfb200_download_outputs_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte
      REAL(c_double), DIMENSION(*), INTENT(INOUT) :: ww, t, t_ave, mu, muave, muts, mudf
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_standin_advance_uv_r8(handle, field, c, i0, i1, j0, j1)                           &
            BIND(C, NAME="wrfb200_standin_advance_uv_r8") RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field
      REAL(c_double), VALUE :: c
      INTEGER(c_int), VALUE :: i0, i1, j0, j1
      INTEGER(c_int) :: status
   END FUNCTION

   ! ---- (D) halo pack / unpack around the caller's own transport; buffers are device addresses ----
   FUNCTION wrfb200_pack_halo(handle, field, side, width, ips, ipe, jps, jpe, device_buf)             &
            BIND(C, NAME="wrfb200_pack_halo") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, side, width, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: device_buf                    ! REAL(c_float) on the device
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_unpack_halo(handle, field, side, width, ips, ipe, jps, jpe, device_buf)           &
            BIND(C, NAME="wrfb200_unpack_halo") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, side, width, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: device_buf                    ! REAL(c_float) on the device
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_pack_halo_r8(handle, field, side, width, ips, ipe, jps, jpe, device_buf)          &
            BIND(C, NAME="wrfb200_pack_halo_r8") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, side, width, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: device_buf                    ! REAL(c_double) on the device
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_unpack_halo_r8(handle, field, side, width, ips, ipe, jps, jpe, device_buf)        &
            BIND(C, NAME="wrfb200_unpack_halo_r8") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: field, side, width, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: device_buf                    ! REAL(c_double) on the device
      INTEGER(c_int) :: status
   END FUNCTION

   ! ---- (C) one rank per GPU: halo exchange fused into the kernels over peer-mapped memory ----
   FUNCTION wrfb200_comm_set_wrap(handle, wrap_x, wrap_y) BIND(C, NAME="wrfb200_comm_set_wrap") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: wrap_x, wrap_y             ! 0 / 1; before wrfb200_comm_init[_r8]
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_init(handle, px, py, rank, ips, ipe, jps, jpe, info_out)                     &
            BIND(C, NAME="wrfb200_comm_init") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: px, py, rank, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: info_out                      ! WRFB200_COMM_INFO_BYTES bytes
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_connect(handle, all_infos, nranks) BIND(C, NAME="wrfb200_comm_connect") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      TYPE(c_ptr), VALUE :: all_infos                     ! nranks blobs in rank order (MPI_Allgather)
      INTEGER(c_int), VALUE :: nranks
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_barrier(handle) BIND(C, NAME="wrfb200_comm_barrier") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_push_constants(handle) BIND(C, NAME="wrfb200_comm_push_constants") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_push_uv(handle) BIND(C, NAME="wrfb200_comm_push_uv") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_wait_outputs(handle) BIND(C, NAME="wrfb200_comm_wait_outputs") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_step(handle) BIND(C, NAME="wrfb200_comm_step") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_loop(handle, nsteps, standin, c, use_graph) BIND(C, NAME="wrfb200_comm_loop") RESULT(status)
      IMPORT :: c_int, c_ptr, c_float
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: nsteps, standin
      REAL(c_float), VALUE :: c
      INTEGER(c_int), VALUE :: use_graph
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_status(handle, flag_timeouts, steps_done) BIND(C, NAME="wrfb200_comm_status") RESULT(status)
      IMPORT :: c_int, c_ptr, c_long
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), INTENT(OUT) :: flag_timeouts
      INTEGER(c_long), INTENT(OUT) :: steps_done
      INTEGER(c_int) :: status
   END FUNCTION

   ! ---- (C') the same on real*8 ranks (-r8 builds); connect / barrier / push_* / wait_outputs / step / status
   !      above serve them too
   FUNCTION wrfb200_comm_init_r8(handle, px, py, rank, ips, ipe, jps, jpe, info_out)                  &
            BIND(C, NAME="wrfb200_comm_init_r8") RESULT(status)
      IMPORT :: c_int, c_ptr
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: px, py, rank, ips, ipe, jps, jpe
      TYPE(c_ptr), VALUE :: info_out                      ! WRFB200_COMM_INFO_BYTES bytes
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_standin_advance_uv_r8(handle, c) BIND(C, NAME="wrfb200_comm_standin_advance_uv_r8")  &
            RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      REAL(c_double), VALUE :: c
      INTEGER(c_int) :: status
   END FUNCTION
   FUNCTION wrfb200_comm_loop_r8(handle, nsteps, standin, c, use_graph) BIND(C, NAME="wrfb200_comm_loop_r8")   &
            RESULT(status)
      IMPORT :: c_int, c_ptr, c_double
      TYPE(c_ptr), VALUE :: handle
      INTEGER(c_int), VALUE :: nsteps, standin
      REAL(c_double), VALUE :: c
      INTEGER(c_int), VALUE :: use_graph
      INTEGER(c_int) :: status
   END FUNCTION
END INTERFACE

CONTAINS

SUBROUTINE wrfb200_loop_begin()
   INTEGER(c_int) :: st
   st = wrfb200_acoustic_loop_begin()
END SUBROUTINE wrfb200_loop_begin

SUBROUTINE wrfb200_loop_end()
   INTEGER(c_int) :: st
   st = wrfb200_acoustic_loop_end()
END SUBROUTINE wrfb200_loop_end

END MODULE module_small_step_em_resident
