!-----------------------------------------------------------------------------------------------------------
! module_small_step_em.F90 -- drop-in replacement for the reference module of the same name
! (lydia-schiff/wrf-model-cuda-sample, module_small_step_em.f90:1-254).
!
! SUBROUTINE advance_mu_t keeps the reference's dummy-argument list, order, ranks, bounds and INTENTs
! exactly (module_small_step_em.f90:7-70), so the caller -- the reference driver's
!     CALL advance_mu_t( grid_ww, ww1, grid_u_2, ... , its, ite, jts, jte, kts, kte )
! (advance_mu_t_driver.f90:193-205), or WRF's solve_em -- compiles and links unchanged.  The body does no
! arithmetic: it pulls the three logicals the routine reads out of config_flags
! (module_small_step_em.f90:97-106; module_configure.f90:434,436,447) and calls the C ABI of
! libwrfb200.so (include/wrfb200.h), which runs the CUDA path.
!
! The dummies are explicit-shape arrays, so they are contiguous and are passed by reference.  The C entry
! is reached through the generic interface wrfb200_amt, whose two specific bodies take REAL(c_float)
! (wrfb200_advance_mu_t) and REAL(c_double) (wrfb200_advance_mu_t_r8): the compiler picks the one that
! matches default REAL, so the same source builds for WRF's default real*4 and for `configure -r8`
! (-fdefault-real-8 / -r8), which then runs in binary64.  grid_config_rec_type is not BIND(C)-interoperable
! (1 796 components, 110 of them character*256): it never crosses the boundary.
!
! Build (any Fortran 2003 compiler; none is available in the build container, see INTEGRATION.md):
!     gfortran -c module_configure.f90 module_small_step_em.F90
!     gfortran advance_mu_t_driver.f90 module_small_step_em.o -L<repo>/wrf_model_cuda_sample_b200 -lwrfb200 \
!              -Wl,-rpath,<repo>/wrf_model_cuda_sample_b200
!-----------------------------------------------------------------------------------------------------------
MODULE module_small_step_em

USE module_configure, ONLY : grid_config_rec_type
USE, INTRINSIC :: iso_c_binding, ONLY : c_float, c_double, c_int, c_char, c_ptr, c_null_char, c_f_pointer, &
                                        c_size_t

IMPLICIT NONE
PRIVATE
PUBLIC :: advance_mu_t

INTERFACE wrfb200_amt
   ! int wrfb200_advance_mu_t(float *ww, const float *ww_1, ..., int kts, int kte);   include/wrfb200.h
   FUNCTION wrfb200_advance_mu_t( ww, ww_1, u, u_1, v, v_1, mu, mut, muave, muts, muu, muv,        &
                                  mudf, t, t_1, t_ave, ft, mu_tend,                               &
                                  rdx, rdy, dts, epssm, dnw, fnm, fnp, rdnw,                      &
                                  msfuy, msfvx_inv, msftx, msfty,                                 &
                                  periodic_x, specified, nested,                                  &
                                  ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme,          &
                                  its, ite, jts, jte, kts, kte )                                  &
            BIND(C, NAME="wrfb200_advance_mu_t") RESULT(status)
      IMPORT :: c_float, c_int
      REAL(c_float), DIMENSION(*), INTENT(INOUT) :: ww, mu, muave, muts, mudf, t, t_ave
      REAL(c_float), DIMENSION(*), INTENT(IN)    :: ww_1, u, u_1, v, v_1, mut, muu, muv, t_1, ft, mu_tend
      REAL(c_float), DIMENSION(*), INTENT(IN)    :: dnw, fnm, fnp, rdnw, msfuy, msfvx_inv, msftx, msfty
      REAL(c_float), VALUE :: rdx, rdy, dts, epssm
      INTEGER(c_int), VALUE :: periodic_x, specified, nested
      INTEGER(c_int), VALUE :: ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte
      INTEGER(c_int) :: status
   END FUNCTION wrfb200_advance_mu_t

   ! int wrfb200_advance_mu_t_r8(double *ww, const double *ww_1, ..., int kts, int kte);   include/wrfb200.h
   FUNCTION wrfb200_advance_mu_t_r8( ww, ww_1, u, u_1, v, v_1, mu, mut, muave, muts, muu, muv,     &
                                     mudf, t, t_1, t_ave, ft, mu_tend,                            &
                                     rdx, rdy, dts, epssm, dnw, fnm, fnp, rdnw,                   &
                                     msfuy, msfvx_inv, msftx, msfty,                              &
                                     periodic_x, specified, nested,                               &
                                     ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme,       &
                                     its, ite, jts, jte, kts, kte )                               &
            BIND(C, NAME="wrfb200_advance_mu_t_r8") RESULT(status)
      IMPORT :: c_double, c_int
      REAL(c_double), DIMENSION(*), INTENT(INOUT) :: ww, mu, muave, muts, mudf, t, t_ave
      REAL(c_double), DIMENSION(*), INTENT(IN)    :: ww_1, u, u_1, v, v_1, mut, muu, muv, t_1, ft, mu_tend
      REAL(c_double), DIMENSION(*), INTENT(IN)    :: dnw, fnm, fnp, rdnw, msfuy, msfvx_inv, msftx, msfty
      REAL(c_double), VALUE :: rdx, rdy, dts, epssm
      INTEGER(c_int), VALUE :: periodic_x, specified, nested
      INTEGER(c_int), VALUE :: ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme
      INTEGER(c_int), VALUE :: its, ite, jts, jte, kts, kte
      INTEGER(c_int) :: status
   END FUNCTION wrfb200_advance_mu_t_r8
END INTERFACE wrfb200_amt

INTERFACE
   ! const char *wrfb200_last_error(void);
   FUNCTION wrfb200_last_error() BIND(C, NAME="wrfb200_last_error") RESULT(msg)
      IMPORT :: c_ptr
      TYPE(c_ptr) :: msg
   END FUNCTION wrfb200_last_error
END INTERFACE

CONTAINS

SUBROUTINE advance_mu_t( ww, ww_1, u, u_1, v, v_1,            &
                         mu, mut, muave, muts, muu, muv,      &
                         mudf, t, t_1,                        &
                         t_ave, ft, mu_tend,                  &
                         rdx, rdy, dts, epssm,                &
                         dnw, fnm, fnp, rdnw,                 &
                         msfuy, msfvx_inv,                    &
                         msftx, msfty,                        &
                         config_flags,                        &
                         ids, ide, jds, jde, kde,             &
                         ims, ime, jms, jme, kms, kme,        &
                         its, ite, jts, jte, kts, kte        )

  IMPLICIT NONE

  TYPE(grid_config_rec_type), INTENT(IN   ) :: config_flags

  INTEGER,      INTENT(IN   )    :: ids,ide, jds,jde, kde
  INTEGER,      INTENT(IN   )    :: ims,ime, jms,jme, kms,kme
  INTEGER,      INTENT(IN   )    :: its,ite, jts,jte, kts,kte

  REAL, DIMENSION( ims:ime , kms:kme, jms:jme ), INTENT(IN   ) :: u, v, u_1, v_1, t_1, ft
  REAL, DIMENSION( ims:ime , kms:kme, jms:jme ), INTENT(INOUT) :: ww, ww_1, t, t_ave
  REAL, DIMENSION( ims:ime , jms:jme ),          INTENT(IN   ) :: muu, muv, mut, msfuy, msfvx_inv,  &
                                                                  msftx, msfty, mu_tend
  REAL, DIMENSION( ims:ime , jms:jme ),          INTENT(  OUT) :: muave, muts, mudf
  REAL, DIMENSION( ims:ime , jms:jme ),          INTENT(INOUT) :: mu
  REAL, DIMENSION( kms:kme ),                    INTENT(IN   ) :: fnm, fnp, dnw, rdnw
  REAL,                                          INTENT(IN   ) :: rdx, rdy, dts, epssm

  INTEGER(c_int) :: status, px, sp, ne

  px = MERGE(1_c_int, 0_c_int, config_flags%periodic_x)
  sp = MERGE(1_c_int, 0_c_int, config_flags%specified)
  ne = MERGE(1_c_int, 0_c_int, config_flags%nested)

  ! resolved at compile time by the kind of default REAL: c_float -> wrfb200_advance_mu_t,
  ! c_double (-r8) -> wrfb200_advance_mu_t_r8
  status = wrfb200_amt( ww, ww_1, u, u_1, v, v_1, mu, mut, muave, muts, muu, muv,                     &
                        mudf, t, t_1, t_ave, ft, mu_tend,                                             &
                        rdx, rdy, dts, epssm, dnw, fnm, fnp, rdnw,                                    &
                        msfuy, msfvx_inv, msftx, msfty, px, sp, ne,                                   &
                        INT(ids, c_int), INT(ide, c_int), INT(jds, c_int), INT(jde, c_int),           &
                        INT(kde, c_int), INT(ims, c_int), INT(ime, c_int), INT(jms, c_int),           &
                        INT(jme, c_int), INT(kms, c_int), INT(kme, c_int), INT(its, c_int),           &
                        INT(ite, c_int), INT(jts, c_int), INT(jte, c_int), INT(kts, c_int),           &
                        INT(kte, c_int) )

  IF ( status /= 0 ) CALL advance_mu_t_fail( status )

END SUBROUTINE advance_mu_t

! The reference CUDA layer prints and exit()s on any CUDA error (advance_mu_t_no_async.cu:22-32); the
! library returns a status instead, and the Fortran side decides: here, print the message and stop.
SUBROUTINE advance_mu_t_fail( status )
  INTEGER(c_int), INTENT(IN) :: status
  TYPE(c_ptr) :: cmsg
  CHARACTER(KIND=c_char), DIMENSION(:), POINTER :: chars
  INTEGER :: n
  cmsg = wrfb200_last_error()
  CALL c_f_pointer( cmsg, chars, [512] )
  n = 0
  DO WHILE ( n < 512 )
     IF ( chars(n+1) == c_null_char ) EXIT
     n = n + 1
  END DO
  WRITE(0,*) 'advance_mu_t (wrfb200): status ', status, ': ', chars(1:n)
  STOP 1
END SUBROUTINE advance_mu_t_fail

END MODULE module_small_step_em
