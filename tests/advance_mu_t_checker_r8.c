/*
 * tests/advance_mu_t_checker_r8.c -- TEST INFRASTRUCTURE: the binary64 checker of the real*8 kernels.
 *
 * It is oracle/advance_mu_t_oracle.c itself, unmodified, compiled with `float` read as `double`: the same
 * statements, each operation rounded once in binary64, in the same (Fortran) order.  The oracle's literals
 * (0.0f, 0.5f, 1.0f) are exact in either precision, so a float literal in a double expression is the double
 * value.  The three exported names get an _r8 suffix.  Built at test time by tests/r8_checkers.py with the
 * oracle's flags (-ffp-contract=off -fno-fast-math: no contraction, no reassociation).
 */
#include <stddef.h>             /* the oracle's headers first, so `float` is redefined for its code only */
#include <stdlib.h>
#include <string.h>

#define float double
#define oracle_advance_mu_t_bounds oracle_advance_mu_t_bounds_r8
#define oracle_advance_mu_t oracle_advance_mu_t_r8
#define oracle_advance_mu_t_tiled oracle_advance_mu_t_tiled_r8
#include "../oracle/advance_mu_t_oracle.c"
