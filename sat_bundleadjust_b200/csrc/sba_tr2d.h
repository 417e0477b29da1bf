// Exact solution of the 2-D trust-region subproblem  min 0.5 p'Bp + g'p  s.t. |p| <= Delta.
// Same contract as scipy/optimize/_lsq/common.py:171-219 (solve_trust_region_2d): the Newton step if B
// is positive definite and the step is inside the region, otherwise the global minimiser on the
// boundary.  scipy finds the boundary minimiser through the roots of a quartic (numpy.roots); here it
// is found from the 2x2 eigen-decomposition and the secular equation, which has no LAPACK dependency
// and runs unchanged on the device.  Below it, the rule that turns one evaluated trial point into the next radius,
// a termination code and the accept/reject decision.
#pragma once
#include <math.h>

#ifndef SBA_HD
#ifdef __CUDACC__
#define SBA_HD __host__ __device__ __forceinline__
#else
#define SBA_HD inline
#endif
#endif

namespace sba {

// returns true when p is the (interior) Newton step
SBA_HD bool solve_trust_region_2d(double b00, double b01, double b11, double g0, double g1, double Delta,
                                  double p[2])
{
    // Cholesky attempt (LAPACK potrf semantics: fail on a non-positive pivot)
    if (b00 > 0.0) {
        const double l00 = sqrt(b00), l10 = b01 / l00, t = b11 - l10 * l10;
        if (t > 0.0) {
            const double l11 = sqrt(t);
            const double y0 = g0 / l00, y1 = (g1 - l10 * y0) / l11;
            const double x1 = y1 / l11, x0 = (y0 - l10 * x1) / l00;
            p[0] = -x0; p[1] = -x1;
            if (p[0] * p[0] + p[1] * p[1] <= Delta * Delta) return true;
        }
    }
    const double gn = sqrt(g0 * g0 + g1 * g1);
    if (!(gn > 0.0)) {
        // no linear term: move along the eigenvector of the smallest eigenvalue
        const double h = 0.5 * (b00 - b11), th = 0.5 * atan2(b01, h);
        p[0] = -sin(th) * Delta; p[1] = cos(th) * Delta;
        return false;
    }
    const double m = 0.5 * (b00 + b11), h = 0.5 * (b00 - b11);
    const double r = sqrt(h * h + b01 * b01);
    if (r == 0.0) {   // B = m I
        p[0] = -Delta * g0 / gn; p[1] = -Delta * g1 / gn;
        return false;
    }
    const double th = 0.5 * atan2(b01, h);
    const double c = cos(th), s_ = sin(th);
    // v2 = (c, s) belongs to lambda2 = m + r, v1 = (-s, c) to lambda1 = m - r
    const double gh1 = -s_ * g0 + c * g1, gh2 = c * g0 + s_ * g1;
    const double lam1 = m - r, two_r = 2.0 * r;
    const double D2 = Delta * Delta;
    double lo = lam1 > 0.0 ? lam1 : 0.0;   // s = lambda1 + mu
    double hi = gn / Delta;
    if (hi < lo) hi = lo;
    double s;
    // hard case: no component along v1 and the v2-only step stays inside
    const double q2 = gh2 / two_r;
    if (lo == 0.0 && gh1 * gh1 <= 1e-300 && q2 * q2 <= D2) {
        double p1 = sqrt(D2 - q2 * q2), p2 = -q2;
        p[0] = -s_ * p1 + c * p2; p[1] = c * p1 + s_ * p2;
        return false;
    }
    s = 0.5 * (lo + hi);
    if (lo == 0.0) { s = fabs(gh1) / Delta; if (!(s > 0.0) || s > hi) s = 0.5 * hi; }
    for (int it = 0; it < 200; ++it) {
        const double a1 = gh1 / s, a2 = gh2 / (s + two_r);
        const double n2 = a1 * a1 + a2 * a2;
        const double f = n2 - D2;
        if (f > 0.0) lo = s; else hi = s;
        if (fabs(f) <= 4e-16 * D2 || hi - lo <= 1e-16 * hi) break;
        // Newton on phi(s) = 1/|p(s)| - 1/Delta
        const double n = sqrt(n2);
        const double dn2 = -2.0 * (a1 * a1 / s + a2 * a2 / (s + two_r));   // d(n2)/ds
        double s_new = s + (n - Delta) / Delta * (2.0 * n2 / (-dn2));
        if (!(s_new > lo && s_new < hi)) s_new = (lo > 0.0) ? sqrt(lo * hi) : 0.5 * (lo + hi);
        if (s_new == s) break;
        s = s_new;
    }
    double p1 = -gh1 / s, p2 = -gh2 / (s + two_r);
    const double nn = sqrt(p1 * p1 + p2 * p2);
    if (nn > 0.0) { p1 *= Delta / nn; p2 *= Delta / nn; }
    p[0] = -s_ * p1 + c * p2; p[1] = c * p1 + s_ * p2;
    return false;
}

// What one evaluated trial point does to the trust-region iteration: scipy's trf_no_bounds inner loop (trf.py:511-560)
// with update_tr_radius (common.py:222-245) and check_termination (common.py:705-717).  A non-finite cost_new shrinks
// the radius to |step_h| / 4 and is neither tested for termination nor accepted; the radius is kept when a termination
// test fires; the step is accepted iff it reduces the cost.
struct TrOutcome {
    double Delta;     // radius of the next trial point
    int status;       // termination: 2 ftol, 3 xtol, 4 both, -1 none
    bool accept;
};

SBA_HD TrOutcome tr_outcome(double cost, double cost_new, double predicted, double step_h_norm, double step_norm,
                            double x_norm, double Delta, double ftol, double xtol)
{
    TrOutcome r = {Delta, -1, false};
    if (!isfinite(cost_new)) { r.Delta = 0.25 * step_h_norm; return r; }
    const double actual = cost - cost_new;
    double ratio;
    if (predicted > 0.0) ratio = actual / predicted;
    else if (predicted == 0.0 && actual == 0.0) ratio = 1.0;
    else ratio = 0.0;
    const bool ftol_ok = actual < ftol * cost && ratio > 0.25;
    const bool xtol_ok = step_norm < xtol * (xtol + x_norm);
    if (ftol_ok && xtol_ok) r.status = 4; else if (ftol_ok) r.status = 2; else if (xtol_ok) r.status = 3;
    if (r.status < 0) {
        if (ratio < 0.25) r.Delta = 0.25 * step_h_norm;
        else if (ratio > 0.75 && step_h_norm > 0.95 * Delta) r.Delta = 2.0 * Delta;
    }
    r.accept = actual > 0.0;
    return r;
}

}  // namespace sba
