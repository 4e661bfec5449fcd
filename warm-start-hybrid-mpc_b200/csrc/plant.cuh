// plant.cuh -- the nonlinear benchmark plant on the device: cart-pole between two soft walls (plants.CartPoleWithWalls).
// One thread integrates one state.  Every product and sum is an explicit round-to-nearest intrinsic, in the operation
// order of plants.py (x_dot, contact_forces, the 2x2 solve by det), so that nvcc cannot contract them to FMAs: the result
// differs from the numpy plant only where CUDA's fp64 sin / cos differ from the host's (at most 2 ulp).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#define WS_PLANT_NPARAM 7          // mc, mp, l, d, stiffness, damping, g (CartPoleWithWalls.params())

// x <- state after n_sub explicit Euler sub-steps of length h with the cart force fc held constant
// (CartPoleWithWalls.simulate with h = dt / n_sub); x = (qc, qp, qc', qp')
__device__ __forceinline__ void cartpole_walls_step(const double *__restrict__ prm, double x[4], double fc, double h, int n_sub)
{
    const double mc = prm[0], mp = prm[1], l = prm[2], d = prm[3], k = prm[4], c = prm[5], g = prm[6];
    const double m11 = __dadd_rn(mc, mp);
    const double mpl = __dmul_rn(mp, l);
    const double m22 = __dmul_rn(mpl, l);
    const double mpgl = __dmul_rn(__dmul_rn(mp, g), l);
    for (int it = 0; it < n_sub; ++it) {
        double s, co;
        sincos(x[1], &s, &co);
        // contact_forces: gaps of the pole tip from the walls, tip velocity, one-sided spring-dampers
        const double tip = __dsub_rn(x[0], __dmul_rn(l, s));
        const double gl = __dadd_rn(tip, d), gr = __dsub_rn(d, tip);
        const double lc = __dmul_rn(l, co);
        const double vtip = __dsub_rn(x[2], __dmul_rn(lc, x[3]));
        const double cv = __dmul_rn(c, vtip);
        double fl = __dsub_rn(__dmul_rn(-k, gl), cv);
        double fr = __dadd_rn(__dmul_rn(-k, gr), cv);
        if (gl > 0. || fl < 0.) fl = 0.;
        if (gr > 0. || fr < 0.) fr = 0.;
        // x_dot: the 2x2 mass matrix solved by its determinant
        const double r1 = __dsub_rn(__dsub_rn(__dadd_rn(fc, fl), fr), __dmul_rn(__dmul_rn(mpl, s), __dmul_rn(x[3], x[3])));
        const double r2 = __dsub_rn(__dmul_rn(mpgl, s), __dmul_rn(lc, __dsub_rn(fl, fr)));
        const double m12 = __dmul_rn(-mpl, co);
        const double det = __dsub_rn(__dmul_rn(m11, m22), __dmul_rn(m12, m12));
        const double qcdd = __ddiv_rn(__dsub_rn(__dmul_rn(m22, r1), __dmul_rn(m12, r2)), det);
        const double qpdd = __ddiv_rn(__dsub_rn(__dmul_rn(m11, r2), __dmul_rn(m12, r1)), det);
        // explicit Euler: x + h * x_dot
        const double v0 = x[2], v1 = x[3];
        x[0] = __dadd_rn(x[0], __dmul_rn(h, v0));
        x[1] = __dadd_rn(x[1], __dmul_rn(h, v1));
        x[2] = __dadd_rn(x[2], __dmul_rn(h, qcdd));
        x[3] = __dadd_rn(x[3], __dmul_rn(h, qpdd));
    }
}

// the plant as the closed loop sees it: parameter sets, sub-steps, which input is the cart force, optional state log
struct PlantView {
    const double *prm;       // [n_sets][WS_PLANT_NPARAM]
    int n_sets;              // 1: one set for every instance; else set k for instance k
    int n_sub;
    double h;                // dt / n_sub
    int fc_index;
    double *log_x;           // [n_steps][n_inst][4] or null
    double *stage;           // [n_inst][4] device scratch: the model error e = x_meas - x_1|t handed to the warm start
};
