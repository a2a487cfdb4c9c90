// solvers.h -- per-solve state shared by solvers.cu and gamg.cu
#pragma once
#include "internal.h"

struct SolverScalars;

struct Solve {
    b200ldu_matrix *m = nullptr;
    b200ldu_ctx *ctx = nullptr;
    SolverScalars *sc = nullptr; // device
    double *partials = nullptr;  // device
    double *psi = nullptr, *src = nullptr; // banded device vectors
    b200ldu_controls c;
    double *hist = nullptr; // device
    int *pinnedFlags = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    double *resultBuf = nullptr;
    int fixedSweeps = 0;
    bool sweepParityUnknown = false;
    double *smoothBuf[2] = {nullptr, nullptr};
    bool noScalars = false;
    bool useGraph = false; // replay iteration chunks as a CUDA graph
    int gamgFinestSweeps = 0; // GAMG: finest-level sweeps per cycle (result-buffer parity)
    double *vec(int k); // workspace vector k < WORK_SOLVER_SLOTS of the matrix (allocated once, reused)
};

int solve_banded(b200ldu_matrix *m, const char *solver, const char *pre, const b200ldu_controls *controls,
                 b200ldu_gamg *gamg, double *psi_b, double *src_b, b200ldu_perf *perf, double *hist_h,
                 int histCap, double **resultBuf);
