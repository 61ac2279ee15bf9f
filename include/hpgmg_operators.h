/*
 * hpgmg_operators.h -- the level-operator entry points (the hot path).
 *
 * Drop-in for /root/reference/finite-volume/source/operators.h:9-50: same names, same argument
 * order and meaning.  These are exactly the external symbols the reference's operators.fv4.o
 * defines (SURVEY.md 8b); here every one of them enqueues hand-written sm_100a kernels on the
 * level's CUDA stream.  Vectors are named by id (hpgmg_defines.h), never by pointer.
 *
 * Behavioural contract kept from the reference:
 *   - smooth() clobbers VECTOR_TEMP and leaves its result in x_id        (gsrb.c:24-132)
 *   - residual()/apply_op() fill the ghost zone of x_id in place          (residual.c:11-12)
 *   - zero_vector() zeroes ghost zones too; all other BLAS1 touch the interior only (misc.c)
 *   - functions returning double (dot/norm/mean/error) synchronise the stream
 *   - fatal conditions print to stderr and exit(0), as the reference does
 */
#ifndef HPGMG_B200_OPERATORS_H
#define HPGMG_B200_OPERATORS_H

#include "hpgmg_level.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RESTRICT_CELL   0
#define RESTRICT_FACE_I 1
#define RESTRICT_FACE_J 2
#define RESTRICT_FACE_K 3

int stencil_get_radius(void);   /* 2                         operators.fv4.c:138   (fv2 flavour: 1) */
int stencil_get_shape(void);    /* STENCIL_SHAPE_NO_CORNERS  operators.fv4.c:139   (fv2 flavour: STENCIL_SHAPE_STAR) */

/* operators/apply_op.c:9, residual.c:9, gsrb.c:24 | chebyshev.c:8, operators.fv4.c:145, rebuild.c:47 */
void apply_op(level_type *level, int Ax_id, int x_id, double a, double b);
void residual(level_type *level, int res_id, int x_id, int rhs_id, double a, double b);
void smooth(level_type *level, int phi_id, int rhs_id, double a, double b);
void rebuild_operator(level_type *level, level_type *fromLevel, double a, double b);
void rebuild_operator_blackbox(level_type *level, double a, double b, int colors_in_each_dim);

/* operators/restriction.c:104, interpolation_v2.c:210, interpolation_v4.c:276, interpolation_p0.c, operators.fv4.c:204-205
 * (vcycle = v2, fcycle = v4; in the fv2 flavour, operators.fv2.c: vcycle = p0, fcycle = v2).  v4 needs 2 ghost layers. */
void restriction(level_type *level_c, int id_c, level_type *level_f, int id_f, int restrictionType);
void interpolation_vcycle(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c);
void interpolation_fcycle(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c);
void interpolation_v2(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c);
void interpolation_v4(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c);
void interpolation_p0(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c);   /* fine = prescale*fine + coarse parent */

/* operators/exchange_boundary.c:12, operators.fv4.c:51, boundary_fv.c:6,101,262,573 */
void exchange_boundary(level_type *level, int id_a, int shape);
void apply_BCs(level_type *level, int x_id, int shape);
void apply_BCs_v1(level_type *level, int x_id, int shape);
void apply_BCs_v2(level_type *level, int x_id, int shape);
void apply_BCs_v4(level_type *level, int x_id, int shape);
void extrapolate_betas(level_type *level);

/* operators/misc.c */
double dot(level_type *level, int id_a, int id_b);
#if defined(__CUDACC__)
/* CUDA's math API already owns an extern "C" norm(int, const double*) in C++ translation units, so
 * inside .cu files the level max-norm is spelled hpgmg_level_norm; its link name is still `norm`. */
double hpgmg_level_norm(level_type *level, int id_a) __asm__("norm");
#else
double norm(level_type *level, int id_a);                /* max norm */
#endif
double mean(level_type *level, int id_a);
double error(level_type *level, int id_a, int id_b);
void   add_vectors(level_type *level, int id_c, double scale_a, int id_a, double scale_b, int id_b);
void   scale_vector(level_type *level, int id_c, double scale_a, int id_a);
void   zero_vector(level_type *level, int id_a);
void   shift_vector(level_type *level, int id_c, int id_a, double shift_a);
void   mul_vectors(level_type *level, int id_c, double scale, int id_a, int id_b);
void   invert_vector(level_type *level, int id_c, double scale_a, int id_a);
void   init_vector(level_type *level, int id_a, double scalar);
void   color_vector(level_type *level, int id, int colors, int icolor, int jcolor, int kcolor);
void   random_vector(level_type *level, int id);

/* operators/problem.fv.c:9,35,90 */
void   initialize_problem(level_type *level, double hLevel, double a, double b);
double evaluateBeta(double x, double y, double z, double h, int add_Bxx, int add_Byy, int add_Bzz);
double evaluateF(double x, double y, double z, double h, int add_Fxx, int add_Fyy, int add_Fzz);

#ifdef __cplusplus
}
#endif
#endif
