// ldu.h -- banded-order matrix operations shared by ldu.cu / solvers.cu / gamg.cu
#pragma once
#include "internal.h"

int matrix_set_diag(b200ldu_matrix *m, const double *diag_d); // banded diag + 1/diag; re-points diag_ext
int to_banded(b200ldu_addr *a, const double *x, double *xb);
int from_banded(b200ldu_addr *a, const double *xb, double *x);
int mat_halo(b200ldu_matrix *m, double *x, const int *stop, int *usedP2P);
// mode: see AmulOp in ops.cuh
int mat_amul(b200ldu_matrix *m, bool transpose, double *x, double *out, int mode, const double *aux,
             double *partials, const int *stop);
int mat_ainv(b200ldu_matrix *m, bool transpose, const double *r, double *w, bool fuseDot,
             const double *dotv, double *partials, const int *stop);
int mat_precondition(b200ldu_matrix *m, int kind, bool transpose, const double *r, double *w, bool fuseDot,
                     const double *dotv, double *partials, int *nPartials, const int *stop);
int mat_jacobi(b200ldu_matrix *m, double omega, double *x, const double *b, double *out, const int *stop);
int mat_residual(b200ldu_matrix *m, double *x, const double *b, double *out, bool fuseSumMag,
                 double *partials, const int *stop);
int mat_sumA(b200ldu_matrix *m, double *out, const int *stop);
int mat_H1(b200ldu_matrix *m, double *out);
int mat_H(b200ldu_matrix *m, const double *x, double *out);
int mat_interpolate(b200ldu_matrix *m, double *x, double *out, const int *stop);
int precond_kind(const char *name, char *printed);
int smoother_ok(const char *name);
