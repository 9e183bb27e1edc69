// oc_rk45.h -- Dormand-Prince 5(4) tableau as used by scipy's RK45 (scipy/integrate/_ivp/rk.py:538-565), and the
// host-side restatement of scipy's RK45 step-size controller shared by the single, batched and row-band HJB solves.
#pragma once
#include <algorithm>
#include <cmath>

#include "../../include/optimal_crowds.h"

namespace rk45 {
static const double A[6][5] = {{0, 0, 0, 0, 0},
                               {1.0 / 5, 0, 0, 0, 0},
                               {3.0 / 40, 9.0 / 40, 0, 0, 0},
                               {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
                               {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
                               {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
static const double B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
static const double E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
static const double P[7][4] = {
    {1, -8048581381.0 / 2820520608, 8663915743.0 / 2820520608, -12715105075.0 / 11282082432},
    {0, 0, 0, 0},
    {0, 131558114200.0 / 32700410799, -68118460800.0 / 10900136933, 87487479700.0 / 32700410799},
    {0, -1754552775.0 / 470086768, 14199869525.0 / 1410260304, -10690763975.0 / 1880347072},
    {0, 127303824393.0 / 49829197408, -318862633887.0 / 49829197408, 701980252875.0 / 199316789632},
    {0, -282668133.0 / 205662961, 2019193451.0 / 616988883, -1453857185.0 / 822651844},
    {0, 40617522.0 / 29380423, -110615467.0 / 29380423, 69997945.0 / 29380423}};

// scipy's RK45 controller (rk.py:111-176, common.py:109-134, base.py:179-210) for the solve from t = T back to
// t_bound = 0, with solve_ivp's t_eval cursor (ivp.py:617-621,715-728).  The caller evaluates the right-hand side and
// the error norms on the GPU and hands the norms in here; every operation is evaluated in scipy's order, so all solves
// built on it take the same accept/reject decisions bit for bit.
//
// t_eval is in the caller's (descending) order; "ascending index" ia counts from its end, sample column kd = nt-1-ia.
// The samples an attempt emits if accepted are the ascending indices [ia_lo, t_eval_i): sample e (0 = latest time)
// has column nt - t_eval_i + e.
struct Controller {
    static constexpr double t_bound = 0.0;
    const double *t_eval = nullptr;
    int nt = 0;
    double direction = 1.0;
    double t = 0, h_abs = 0, h = 0, t_new = 0, min_step = 0;
    bool rejected = false;
    int status = 1;  // solve_ivp: 1 running, 0 finished, -1 step too small
    int t_eval_i = 0, ia_lo = 0, n_out = 0;
    int n_accepted = 0, n_rejected = 0;

    Controller() = default;
    Controller(double T, const double *t_eval_, int nt_)
        : t_eval(t_eval_), nt(nt_), direction((t_bound != T) ? (t_bound > T ? 1.0 : -1.0) : 1.0), t(T), t_eval_i(nt_) {}

    // select_initial_step (common.py:109-134).  With T == t_bound there is nothing to integrate and h_abs stays 0;
    // otherwise h0 from the norms d0 = |y0|, d1 = |f0|, then h_abs from d2 = |f(y0 + h0 f0) - f0| / h0.
    bool needs_initial_step() const { return std::fabs(t_bound - t) != 0.0; }
    double initial_h0(double d0, double d1) const {
        const double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        return std::min(h0, std::fabs(t_bound - t));
    }
    void set_initial_step(double h0, double d1, double d2) {
        double h1;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = std::max(1e-6, h0 * 1e-3);
        else h1 = std::pow(0.01 / std::max(d1, d2), 1.0 / 5.0);
        h_abs = std::min(std::min(100 * h0, h1), std::fabs(t_bound - t));
    }

    // base.py:179-198 step(): false once the solve has ended
    bool begin_step() {
        if (status != 1) return false;
        if (t == t_bound) { status = 0; return false; }
        min_step = 10 * std::fabs(std::nextafter(t, direction * INFINITY) - t);
        if (h_abs < min_step) h_abs = min_step;
        rejected = false;
        return true;
    }
    // rk.py:120-131: the next attempt's h, t_new and samples; false (status -1) when the step has become too small.
    // forced_h[i] replaces the controller's h of attempt i < n_forced (teacher-forced parity tests).
    bool propose(const double *forced_h = nullptr, int n_forced = 0) {
        if (h_abs < min_step) { status = -1; return false; }
        h = h_abs * direction;
        if (forced_h && attempts() < n_forced) h = forced_h[attempts()];
        t_new = t + h;
        if (direction * (t_new - t_bound) > 0) t_new = t_bound;
        h = t_new - t;
        h_abs = std::fabs(h);
        ia_lo = std::min(lower_index(t_new), t_eval_i);
        return true;
    }
    int attempts() const { return n_accepted + n_rejected; }
    int n_emit() const { return t_eval_i - ia_lo; }
    int sample_column(int e) const { return nt - t_eval_i + e; }
    double sample_x(int e) const { return (t_eval[sample_column(e)] - t) / h; }  // RkDenseOutput: (t - t_old)/h

    // rk.py:146-165: true if the attempt is accepted
    bool judge(double error_norm) {
        const double error_exponent = -1.0 / 5.0;
        if (error_norm < 1) {
            double factor = (error_norm == 0) ? 10.0 : std::min(10.0, 0.9 * std::pow(error_norm, error_exponent));
            if (rejected) factor = std::min(1.0, factor);
            h_abs *= factor;
            n_accepted++;
            return true;
        }
        h_abs *= std::max(0.2, 0.9 * std::pow(error_norm, error_exponent));
        rejected = true;
        n_rejected++;
        return false;
    }
    // base.py:205-208, ivp.py:715-728: move to t_new past the attempt's samples
    void accept() {
        if (direction * (t_new - t_bound) >= 0) status = 0;
        n_out += n_emit();
        t_eval_i = ia_lo;
        t = t_new;
    }
    void report(oc_hjb_stats *s) const {
        s->status = status;
        s->n_out = n_out;
        s->n_accepted = n_accepted;
        s->n_rejected = n_rejected;
    }

    // first ascending index whose time is >= t (direction < 0)
    int lower_index(double tq) const {
        int lo = 0, hi = nt;
        while (lo < hi) {
            const int mid = (lo + hi) / 2;
            if (t_eval[nt - 1 - mid] < tq) lo = mid + 1; else hi = mid;
        }
        return lo;
    }
};
}  // namespace rk45
