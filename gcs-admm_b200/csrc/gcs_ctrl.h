// Control block of one problem (device memory; one per problem in batched mode).  Written by the control step
// (reference admm_solver_v3.py:697-713), read by every kernel.
#pragma once
#define NSUMS 10  // r2, dz2, x2, z2, mu2 (pre-scale), nonfinite | check variant (-1: not computed): inner residual^2 (perf mode), r2 and dz2 in
                  // GLOBAL coordinates (local frames: the reference's definition of the residuals) | spare

struct Ctrl {
    double rho, mu_scale;
    double pri, dual, eps_pri, eps_dual;
    double pri_g, dual_g;   // local frames: the residuals in global coordinates (the reference's definition :598 / :602); -1: not computed
    double inner;       // perf mode: |(M u + m0) - c| over all (point, flow) pairs — how far the vertex programs' own constraints are from being met
    double sums[NSUMS];
    double abs_tol;         // this problem's tolerance of the absolute stop rule (0: GcsParams.abs_tol)
    unsigned long long inner_iters, skipped;
    int it, stop, opt, diverged, inner_fail, ignore_stop;
    int inner_active;       // batched perf mode: this problem is near its tolerance, the edge kernel adds up its inner residual (set by gcsadmm_run)
};
