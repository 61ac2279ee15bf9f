/*
 * hpgmg_solvers.h -- bottom solver.  Drop-in for /root/reference/finite-volume/source/solvers.h:9-10.
 * Two solvers are built and chosen at run time (hpgmg_b200_set_bottom_solver, hpgmg_b200.h): the diagonally preconditioned
 * BiCGStab of solvers/bicgstab.c:14-97 (the reference's default, -DUSE_BICGSTAB) and the diagonally preconditioned CG of
 * solvers/cg.c (-DUSE_CG).  The CA variants (-DUSE_CABICGSTAB, -DUSE_CACG) are not built.
 *
 * IterativeSolver_NumVectors() is 8 whichever solver is selected: MGBuild sizes the bottom level once and the selection may
 * change afterwards.  The reference built with -DUSE_CG allocates 5 (r0 r p Ap z); CG here uses the first 5 of the 8 and
 * leaves the other 3 untouched, so no result depends on the difference.
 */
#ifndef HPGMG_B200_SOLVERS_H
#define HPGMG_B200_SOLVERS_H
#include "hpgmg_level.h"
#ifdef __cplusplus
extern "C" {
#endif
void IterativeSolver(level_type *level, int u_id, int f_id, double a, double b, double desired_reduction_in_norm);
int  IterativeSolver_NumVectors(void);
#ifdef __cplusplus
}
#endif
#endif
