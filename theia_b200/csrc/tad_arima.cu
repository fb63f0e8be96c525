// ARIMA detector (anomaly_detection.py:215-309): Box-Cox (MLE lambda) -> for every prefix of the
// series an ARIMA(1,1,1) state-space MLE fit and one-step forecast -> inverse Box-Cox -> flag.
//
// The per-fit algorithm is the one statsmodels 0.14 runs (see oracle/arima_oracle.py for the
// statement of it and for the parity status -- unpinned below ~1e-3 relative on algoCalc):
//   * 3-state Kalman filter likelihood, approximate-diffuse + stationary initialisation, burn 1;
//   * optimisation over the unconstrained parameters by L-BFGS with a More'-Thuente line search
//     (the unconstrained path of L-BFGS-B: m = 12, pgtol 1e-8, factr 1e2, maxiter 50,
//     forward-difference gradient with step 1e-8) on -loglike / nobs;
//   * Hannan-Rissanen start values.
// Compute-bound FP64 (about n^2/2 Kalman steps x ~100 likelihood evaluations per series), so the
// mapping is one WARP per series with one lane per prefix fit; the series lives in L1.
#include <cfloat>

#include "tad_kernels.h"

namespace tad {

inline namespace arima_core {

constexpr double kDiffuse = 1e6;
constexpr double kLog2Pi = 1.8378770664093454835606594728112;
constexpr int kLbfgsM = 12;

__device__ __forceinline__ SeriesEntry load_entry(const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase,
                                                  uint32_t B, uint32_t i)
{
    const uint32_t b = find_bucket(sbase, B, i);
    const uint4 *p = reinterpret_cast<const uint4 *>(entries + offsets[b] + (i - sbase[b]));
    const uint4 k = p[0], w = p[1];
    SeriesEntry e;
    e.a = ((uint64_t)k.y << 32) | k.x; e.b = ((uint64_t)k.w << 32) | k.z;
    e.proto = w.x; e.n = w.y; e.off = w.z; e.pad = w.w;
    return e;
}

// ------------------------------------------------------------------------------------------
// Box-Cox: llf(lambda) = (lambda - 1) sum(log x) - N/2 log var(x^lambda / lambda)   (scipy.stats.boxcox_llf)
// ------------------------------------------------------------------------------------------
// The variance of x^lambda / lambda is evaluated in log space (var = e^{2m} var(e^{z - m}) / lambda^2 with
// z = lambda log x, m = max z), so the likelihood stays finite for any lambda and Brent converges to the
// true optimum even when the transform itself would overflow (the caller then drops the series).
__host__ __device__ double boxcox_neg_llf(double lmb, const double *__restrict__ logx, uint32_t n, double sumlog)
{
    double logvar;
    if (lmb == 0.0) {
        double mean = 0.0;
        for (uint32_t i = 0; i < n; i++) mean += logx[i];
        mean /= n;
        double var = 0.0;
        for (uint32_t i = 0; i < n; i++) { const double d = logx[i] - mean; var += d * d; }
        logvar = log(var / n);
    } else {
        double m = -DBL_MAX;
        for (uint32_t i = 0; i < n; i++) m = fmax(m, lmb * logx[i]);
        double mean = 0.0;
        for (uint32_t i = 0; i < n; i++) mean += exp(lmb * logx[i] - m);
        mean /= n;
        double var = 0.0;
        for (uint32_t i = 0; i < n; i++) { const double d = exp(lmb * logx[i] - m) - mean; var += d * d; }
        logvar = log(var / n) + 2.0 * m - 2.0 * log(fabs(lmb));
    }
    return -((lmb - 1.0) * sumlog - 0.5 * n * logvar);
}

// scipy.optimize.brent(f, brack=(-2, 2)): bracket() followed by Brent's parabolic/golden iteration, tol 1.48e-8
__host__ __device__ double boxcox_mle_lambda(const double *__restrict__ logx, uint32_t n, double sumlog)
{
    auto f = [&](double l) { return boxcox_neg_llf(l, logx, n, sumlog); };
    const double gold = 1.618034, verysmall = 1e-21, grow = 110.0;
    double xa = -2.0, xb = 2.0;
    double fa = f(xa), fb = f(xb);
    if (fa < fb) { double t = xa; xa = xb; xb = t; t = fa; fa = fb; fb = t; }
    double xc = xb + gold * (xb - xa), fc = f(xc);
    int iter = 0;
    while (fc < fb && iter < 1000) {
        const double tmp1 = (xb - xa) * (fb - fc), tmp2 = (xb - xc) * (fb - fa);
        const double val = tmp2 - tmp1;
        const double denom = fabs(val) < verysmall ? 2.0 * verysmall : 2.0 * val;
        double w = xb - ((xb - xc) * tmp2 - (xb - xa) * tmp1) / denom;
        const double wlim = xb + grow * (xc - xb);
        double fw;
        iter++;
        if ((w - xc) * (xb - w) > 0.0) {
            fw = f(w);
            if (fw < fc) { xa = xb; xb = w; fa = fb; fb = fw; break; }
            else if (fw > fb) { xc = w; fc = fw; break; }
            w = xc + gold * (xc - xb); fw = f(w);
        } else if ((w - wlim) * (wlim - xc) >= 0.0) {
            w = wlim; fw = f(w);
        } else if ((w - wlim) * (xc - w) > 0.0) {
            fw = f(w);
            if (fw < fc) { xb = xc; xc = w; w = xc + gold * (xc - xb); fb = fc; fc = fw; fw = f(w); }
        } else {
            w = xc + gold * (xc - xb); fw = f(w);
        }
        xa = xb; xb = xc; xc = w; fa = fb; fb = fc; fc = fw;
    }
    const double mintol = 1.0e-11, cg = 0.3819660, tol = 1.48e-8;
    double x = xb, w = xb, v = xb, fx = fb, fw = fb, fv = fb;
    double a = xa < xc ? xa : xc, b = xa < xc ? xc : xa;
    double deltax = 0.0, rat = 0.0;
    for (iter = 0; iter < 500; iter++) {
        const double tol1 = tol * fabs(x) + mintol, tol2 = 2.0 * tol1, xmid = 0.5 * (a + b);
        if (fabs(x - xmid) < (tol2 - 0.5 * (b - a))) break;
        if (fabs(deltax) <= tol1) {
            deltax = x >= xmid ? a - x : b - x;
            rat = cg * deltax;
        } else {
            double tmp1 = (x - w) * (fx - fv), tmp2 = (x - v) * (fx - fw);
            double p = (x - v) * tmp2 - (x - w) * tmp1;
            tmp2 = 2.0 * (tmp2 - tmp1);
            if (tmp2 > 0.0) p = -p;
            tmp2 = fabs(tmp2);
            const double dx_temp = deltax;
            deltax = rat;
            if (p > tmp2 * (a - x) && p < tmp2 * (b - x) && fabs(p) < fabs(0.5 * tmp2 * dx_temp)) {
                rat = p / tmp2;
                const double u = x + rat;
                if ((u - a) < tol2 || (b - u) < tol2) rat = (xmid - x >= 0) ? tol1 : -tol1;
            } else {
                deltax = x >= xmid ? a - x : b - x;
                rat = cg * deltax;
            }
        }
        const double u = fabs(rat) < tol1 ? (rat >= 0 ? x + tol1 : x - tol1) : x + rat;
        const double fu = f(u);
        if (fu > fx) {
            if (u < x) a = u; else b = u;
            if (fu <= fw || w == x) { v = w; w = u; fv = fw; fw = fu; }
            else if (fu <= fv || v == x || v == w) { v = u; fv = fu; }
        } else {
            if (u >= x) a = x; else b = x;
            v = w; w = x; x = u; fv = fw; fw = fx; fx = fu;
        }
    }
    return x;
}

// ------------------------------------------------------------------------------------------
// ARIMA(1,1,1) likelihood (3-state Kalman filter, symmetric P as six scalars)
// ------------------------------------------------------------------------------------------
struct ArimaObj {
    const double *y;
    uint32_t n;
};

__host__ __device__ __forceinline__ void arima_transform(const double u[3], double &phi, double &theta, double &s2)
{
    phi = u[0] / sqrt(1.0 + u[0] * u[0]);
    theta = u[1] / sqrt(1.0 + u[1] * u[1]);
    s2 = u[2] * u[2];
}

// One filter: the state the recursion carries (a2 = p02 = 0, p12 = q12, p22 = q22 after every prediction step, so they are
// constants of the parameters) and one time step.  arima_loglike runs one of these; arima_fg runs FOUR side by side in one
// loop -- the objective at u and at its three forward-difference neighbours -- so that a lane has four independent FP64
// dependency chains in flight instead of one (the arithmetic of every chain is exactly that of the single filter).
struct Kalman {
    double phi, q11, q12, q22;
    double a0, a1, a2, p00, p01, p02, p11, p12, p22, ll;
    bool dead;                       // F <= 0 or not finite at some step: the likelihood is -1e300 (statsmodels raises)
};

__host__ __device__ __forceinline__ void kalman_init(Kalman &k, double phi, double theta, double s2)
{
    k.phi = phi;
    k.a0 = 0.0; k.a1 = 0.0; k.a2 = 0.0;
    k.p00 = kDiffuse; k.p01 = 0.0; k.p02 = 0.0;
    k.p11 = s2 * (1.0 + 2.0 * phi * theta + theta * theta) / (1.0 - phi * phi);
    k.p12 = s2 * theta; k.p22 = s2 * theta * theta;
    k.q11 = s2; k.q12 = s2 * theta; k.q22 = s2 * theta * theta;
    k.ll = 0.0;
    k.dead = false;
}

__host__ __device__ __forceinline__ void kalman_step(Kalman &k, double yt, bool count)
{
    const double v = yt - (k.a0 + k.a1);
    const double F = k.p00 + 2.0 * k.p01 + k.p11;
    if (!(F > 0.0) || !isfinite(F)) { k.dead = true; return; }
    if (count) k.ll += -0.5 * (kLog2Pi + log(F) + v * v / F);
    const double z0 = k.p00 + k.p01, z1 = k.p01 + k.p11, z2 = k.p02 + k.p12;
    const double g = v / F;
    const double f0 = k.a0 + z0 * g, f1 = k.a1 + z1 * g, f2 = k.a2 + z2 * g;
    const double c00 = k.p00 - z0 * z0 / F, c01 = k.p01 - z0 * z1 / F, c02 = k.p02 - z0 * z2 / F;
    const double c11 = k.p11 - z1 * z1 / F, c12 = k.p12 - z1 * z2 / F, c22 = k.p22 - z2 * z2 / F;
    k.a0 = f0 + f1; k.a1 = k.phi * f1 + f2; k.a2 = 0.0;
    k.p00 = c00 + 2.0 * c01 + c11;
    k.p01 = k.phi * (c01 + c11) + c02 + c12;
    k.p02 = 0.0;
    k.p11 = k.phi * k.phi * c11 + 2.0 * k.phi * c12 + c22 + k.q11;
    k.p12 = k.q12;
    k.p22 = k.q22;
}

__host__ __device__ double arima_loglike(const ArimaObj &o, double phi, double theta, double s2, double *forecast)
{
    Kalman k;
    kalman_init(k, phi, theta, s2);
    for (uint32_t t = 0; t < o.n && !k.dead; t++) kalman_step(k, o.y[t], t >= 1);
    if (k.dead) {
        if (forecast) *forecast = 0.0;
        return -1e300;
    }
    if (forecast) *forecast = k.a0 + k.a1;
    return k.ll;
}

__host__ __device__ __forceinline__ double arima_objective(const ArimaObj &o, const double u[3])
{
    double phi, theta, s2;
    arima_transform(u, phi, theta, s2);
    return -arima_loglike(o, phi, theta, s2, nullptr) / (double)o.n;
}

// f and the forward-difference gradient (step 1e-8, as SciPy's approx_fprime drives L-BFGS-B): four filters in one loop
__host__ __device__ void arima_fg(const ArimaObj &o, double u[3], double &f, double g[3])
{
    Kalman k[4];
    for (int c = 0; c < 4; c++) {
        double uc[3] = {u[0], u[1], u[2]};
        if (c > 0) uc[c - 1] = u[c - 1] + 1e-8;
        double phi, theta, s2;
        arima_transform(uc, phi, theta, s2);
        kalman_init(k[c], phi, theta, s2);
    }
    for (uint32_t t = 0; t < o.n; t++) {
        const double yt = o.y[t];
        const bool count = t >= 1;
#pragma unroll
        for (int c = 0; c < 4; c++)
            if (!k[c].dead) kalman_step(k[c], yt, count);
    }
    double fv[4];
    for (int c = 0; c < 4; c++) fv[c] = -(k[c].dead ? -1e300 : k[c].ll) / (double)o.n;
    f = fv[0];
    for (int c = 0; c < 3; c++) g[c] = (fv[c + 1] - f) / 1e-8;
}

// Least-squares solution of a two-regressor problem from its normal equations, following numpy.linalg.pinv:
// full rank -> the unique solution; rank one (singular value ratio below 1e-15) -> the minimum-norm solution
// b / trace(A); rank zero -> 0.
__host__ __device__ __forceinline__ void lstsq2(double s11, double s12, double s22, double r1, double r2, double &b1, double &b2)
{
    const double tr = s11 + s22, det = s11 * s22 - s12 * s12;
    b1 = 0.0; b2 = 0.0;
    if (!(tr > 0.0) || !isfinite(tr)) return;
    if (det > 1e-30 * tr * tr) {
        b1 = (r1 * s22 - r2 * s12) / det;
        b2 = (r2 * s11 - r1 * s12) / det;
    } else {
        b1 = r1 / tr;
        b2 = r2 / tr;
    }
}

// Hannan-Rissanen / conditional-sum-of-squares start values on the differenced data (k_ar = k_ma = 1)
__host__ __device__ void arima_start(const ArimaObj &o, double u[3])
{
    const double *y = o.y;
    const int m = (int)o.n - 1;                      // d[i] = y[i+1] - y[i]
    auto d = [&](int i) { return y[i + 1] - y[i]; };
    double phi0 = 0.0, th0 = 0.0, var = NAN;
    double dmean = 0.0;
    for (int i = 0; i < m; i++) dmean += d(i);
    dmean = m > 0 ? dmean / m : 0.0;
    double dvar = 0.0;
    for (int i = 0; i < m; i++) { const double e = d(i) - dmean; dvar += e * e; }
    dvar = m > 0 ? dvar / m : 0.0;
    if (m >= 4) {
        // AR(2) by least squares: d[t] ~ b1 d[t-1] + b2 d[t-2], t = 2..m-1
        double s11 = 0, s12 = 0, s22 = 0, r1 = 0, r2 = 0;
        for (int t = 2; t < m; t++) {
            const double x1 = d(t - 1), x2 = d(t - 2), yy = d(t);
            s11 += x1 * x1; s12 += x1 * x2; s22 += x2 * x2; r1 += x1 * yy; r2 += x2 * yy;
        }
        double b1, b2;
        lstsq2(s11, s12, s22, r1, r2, b1, b2);
        auto res = [&](int t) { return d(t) - b1 * d(t - 1) - b2 * d(t - 2); };      // residual at t >= 2
        // ARMA(1,1): d[t] ~ phi d[t-1] + theta res[t-1], t = 3..m-1
        s11 = s12 = s22 = r1 = r2 = 0;
        for (int t = 3; t < m; t++) {
            const double x1 = d(t - 1), x2 = res(t - 1), yy = d(t);
            s11 += x1 * x1; s12 += x1 * x2; s22 += x2 * x2; r1 += x1 * yy; r2 += x2 * yy;
        }
        lstsq2(s11, s12, s22, r1, r2, phi0, th0);
        if (m - 3 > 1) {
            double acc = 0.0;
            for (int t = 4; t < m; t++) { const double e = d(t) - phi0 * d(t - 1) - th0 * res(t - 1); acc += e * e; }
            var = acc / (m - 4);
        }
    }
    if (!(fabs(phi0) < 1.0)) phi0 = 0.0;
    if (!(fabs(th0) < 1.0)) th0 = 0.0;
    if (!isfinite(var) || var <= 1e-10 * dvar || var <= 0.0) var = dvar > 0.0 ? dvar : 1.0;
    u[0] = phi0 / sqrt(1.0 - phi0 * phi0);
    u[1] = th0 / sqrt(1.0 - th0 * th0);
    u[2] = sqrt(var);
}

// ------------------------------------------------------------------------------------------
// More'-Thuente line search (MINPACK-2 dcsrch / dcstep), as driven by L-BFGS-B's lnsrlb
// ------------------------------------------------------------------------------------------
struct LineSearch {
    bool brackt;
    int stage;
    double ginit, gtest, gx, gy, finit, fx, fy, stx, sty, stmin, stmax, width, width1;
};
enum { LS_FG = 0, LS_CONV = 1, LS_WARN = 2 };

__host__ __device__ void dcstep(double &stx, double &fx, double &dx, double &sty, double &fy, double &dy, double &stp, double fp, double dp,
                       bool &brackt, double stpmin, double stpmax)
{
    const double sgnd = dp * (dx / fabs(dx));
    double stpf;
    if (fp > fx) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
        if (stp < stx) gamma = -gamma;
        const double p = (gamma - dx) + theta, q = ((gamma - dx) + gamma) + dp, r = p / q;
        const double stpc = stx + r * (stp - stx);
        const double stpq = stx + ((dx / ((fx - fp) / (stp - stx) + dx)) / 2.0) * (stp - stx);
        stpf = fabs(stpc - stx) < fabs(stpq - stx) ? stpc : stpc + (stpq - stpc) / 2.0;
        brackt = true;
    } else if (sgnd < 0.0) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
        if (stp > stx) gamma = -gamma;
        const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dx, r = p / q;
        const double stpc = stp + r * (stx - stp);
        const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
        stpf = fabs(stpc - stp) > fabs(stpq - stp) ? stpc : stpq;
        brackt = true;
    } else if (fabs(dp) < fabs(dx)) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt(fmax(0.0, (theta / s) * (theta / s) - (dx / s) * (dp / s)));
        if (stp > stx) gamma = -gamma;
        const double p = (gamma - dp) + theta, q = (gamma + (dx - dp)) + gamma, r = p / q;
        double stpc;
        if (r < 0.0 && gamma != 0.0) stpc = stp + r * (stx - stp);
        else if (stp > stx) stpc = stpmax;
        else stpc = stpmin;
        const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
        if (brackt) {
            stpf = fabs(stpc - stp) < fabs(stpq - stp) ? stpc : stpq;
            if (stp > stx) stpf = fmin(stp + 0.66 * (sty - stp), stpf);
            else stpf = fmax(stp + 0.66 * (sty - stp), stpf);
        } else {
            stpf = fabs(stpc - stp) > fabs(stpq - stp) ? stpc : stpq;
            stpf = fmin(stpmax, stpf);
            stpf = fmax(stpmin, stpf);
        }
    } else {
        if (brackt) {
            const double theta = 3.0 * (fp - fy) / (sty - stp) + dy + dp;
            const double s = fmax(fabs(theta), fmax(fabs(dy), fabs(dp)));
            double gamma = s * sqrt((theta / s) * (theta / s) - (dy / s) * (dp / s));
            if (stp > sty) gamma = -gamma;
            const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dy, r = p / q;
            stpf = stp + r * (sty - stp);
        } else if (stp > stx) stpf = stpmax;
        else stpf = stpmin;
    }
    if (fp > fx) {
        sty = stp; fy = fp; dy = dp;
    } else {
        if (sgnd < 0.0) { sty = stx; fy = fx; dy = dx; }
        stx = stp; fx = fp; dx = dp;
    }
    stp = stpf;
}

__host__ __device__ void dcsrch_start(LineSearch &ls, double stp, double f, double g, double ftol, double stpmin, double stpmax)
{
    ls.brackt = false;
    ls.stage = 1;
    ls.finit = f; ls.ginit = g; ls.gtest = ftol * g;
    ls.width = stpmax - stpmin; ls.width1 = ls.width / 0.5;
    ls.stx = 0.0; ls.fx = f; ls.gx = g;
    ls.sty = 0.0; ls.fy = f; ls.gy = g;
    ls.stmin = 0.0; ls.stmax = stp + 4.0 * stp;
}

__host__ __device__ int dcsrch_step(LineSearch &ls, double &stp, double f, double g, double ftol, double gtol, double xtol, double stpmin,
                           double stpmax)
{
    const double ftest = ls.finit + stp * ls.gtest;
    if (ls.stage == 1 && f <= ftest && g >= 0.0) ls.stage = 2;
    int task = LS_FG;
    if (ls.brackt && (stp <= ls.stmin || stp >= ls.stmax)) task = LS_WARN;
    if (ls.brackt && ls.stmax - ls.stmin <= xtol * ls.stmax) task = LS_WARN;
    if (stp == stpmax && f <= ftest && g <= ls.gtest) task = LS_WARN;
    if (stp == stpmin && (f > ftest || g >= ls.gtest)) task = LS_WARN;
    if (f <= ftest && fabs(g) <= gtol * (-ls.ginit)) task = LS_CONV;
    if (task != LS_FG) return task;
    if (ls.stage == 1 && f <= ls.fx && f > ftest) {
        const double fm = f - stp * ls.gtest;
        double fxm = ls.fx - ls.stx * ls.gtest, fym = ls.fy - ls.sty * ls.gtest;
        const double gm = g - ls.gtest;
        double gxm = ls.gx - ls.gtest, gym = ls.gy - ls.gtest;
        dcstep(ls.stx, fxm, gxm, ls.sty, fym, gym, stp, fm, gm, ls.brackt, ls.stmin, ls.stmax);
        ls.fx = fxm + ls.stx * ls.gtest; ls.fy = fym + ls.sty * ls.gtest;
        ls.gx = gxm + ls.gtest; ls.gy = gym + ls.gtest;
    } else {
        dcstep(ls.stx, ls.fx, ls.gx, ls.sty, ls.fy, ls.gy, stp, f, g, ls.brackt, ls.stmin, ls.stmax);
    }
    if (ls.brackt) {
        if (fabs(ls.sty - ls.stx) >= 0.66 * ls.width1) stp = ls.stx + 0.5 * (ls.sty - ls.stx);
        ls.width1 = ls.width;
        ls.width = fabs(ls.sty - ls.stx);
    }
    if (ls.brackt) {
        ls.stmin = fmin(ls.stx, ls.sty);
        ls.stmax = fmax(ls.stx, ls.sty);
    } else {
        ls.stmin = stp + 1.1 * (stp - ls.stx);
        ls.stmax = stp + 4.0 * (stp - ls.stx);
    }
    stp = fmax(stp, stpmin);
    stp = fmin(stp, stpmax);
    if ((ls.brackt && (stp <= ls.stmin || stp >= ls.stmax)) || (ls.brackt && ls.stmax - ls.stmin <= xtol * ls.stmax)) stp = ls.stx;
    return LS_FG;
}

// ------------------------------------------------------------------------------------------
// L-BFGS (the unconstrained path of L-BFGS-B 3.0 as SciPy drives it), written as a resumable state machine:
// the caller evaluates (f, g) at x, lbfgs_advance() consumes them and either leaves the next trial point in x
// (returns false) or ends the fit (returns true, x = the solution).  The host driver below loops over it; the fit
// kernel lets all lanes of a warp evaluate TOGETHER (the Kalman-filter likelihood, >95 % of the work, then runs
// converged) and only the cheap bookkeeping between two evaluations diverges.
// ------------------------------------------------------------------------------------------
struct Lbfgs {
    double S[kLbfgsM][3], Y[kLbfgsM][3], rho[kLbfgsM];
    int col, head, iter, ifun, state;        // state 0: first evaluation pending, 1: line-search evaluation pending
    double theta, f, g[3], d[3], stp, fold, xold[3], gold[3], gdold, gd;
    LineSearch ls;
};

__host__ __device__ __forceinline__ void lbfgs_init(Lbfgs &s)
{
    s.col = 0; s.head = 0; s.iter = 0; s.ifun = 0; s.state = 0; s.theta = 1.0;
}

// start iterations from (s.f, s.g) at x until a line search has its first trial point in x (false) or the fit ends (true)
__host__ __device__ bool lbfgs_begin_iter(Lbfgs &s, double x[3])
{
    const double stpmx = 1e10, ftol = 1e-3;
    for (;;) {
        if (s.iter >= 50) return true;
        // ---- direction d = -H g (two-loop recursion, H0 = I / theta) ------------------------
        double d[3] = {s.g[0], s.g[1], s.g[2]}, alpha[kLbfgsM];
        for (int k = s.col - 1; k >= 0; k--) {
            const int i = (s.head + k) % kLbfgsM;
            alpha[k] = s.rho[i] * (s.S[i][0] * d[0] + s.S[i][1] * d[1] + s.S[i][2] * d[2]);
            for (int c = 0; c < 3; c++) d[c] -= alpha[k] * s.Y[i][c];
        }
        for (int c = 0; c < 3; c++) d[c] /= s.theta;
        for (int k = 0; k < s.col; k++) {
            const int i = (s.head + k) % kLbfgsM;
            const double beta = s.rho[i] * (s.Y[i][0] * d[0] + s.Y[i][1] * d[1] + s.Y[i][2] * d[2]);
            for (int c = 0; c < 3; c++) d[c] += s.S[i][c] * (alpha[k] - beta);
        }
        for (int c = 0; c < 3; c++) s.d[c] = -d[c];
        // ---- line search ----------------------------------------------------------------------
        const double dnorm = sqrt(s.d[0] * s.d[0] + s.d[1] * s.d[1] + s.d[2] * s.d[2]);
        s.stp = s.iter == 0 ? fmin(1.0 / dnorm, stpmx) : 1.0;
        s.fold = s.f;
        for (int c = 0; c < 3; c++) { s.xold[c] = x[c]; s.gold[c] = s.g[c]; }
        s.gdold = s.g[0] * s.d[0] + s.g[1] * s.d[1] + s.g[2] * s.d[2];
        s.gd = s.gdold;
        const bool ok = s.gdold < 0.0 && isfinite(s.gdold) && dnorm > 0.0;
        if (ok) {
            dcsrch_start(s.ls, s.stp, s.f, s.gdold, ftol, 0.0, stpmx);
            s.ifun = 0;
            for (int c = 0; c < 3; c++) x[c] = s.xold[c] + s.stp * s.d[c];
            s.state = 1;
            return false;
        }
        // no descent direction: with stored pairs restart from steepest descent, else stop (x, f, g are unchanged)
        if (s.col == 0) return true;
        s.col = 0; s.head = 0; s.theta = 1.0;
    }
}

__host__ __device__ bool lbfgs_advance(Lbfgs &s, double x[3], double f, const double g[3])
{
    const double pgtol = 1e-8, factr = 1e2, epsmch = DBL_EPSILON, stpmx = 1e10;
    const double ftol = 1e-3, gtol = 0.9, xtol = 0.1;
    s.f = f;
    for (int c = 0; c < 3; c++) s.g[c] = g[c];
    if (s.state == 0) {
        if (fmax(fabs(g[0]), fmax(fabs(g[1]), fabs(g[2]))) <= pgtol) return true;
        return lbfgs_begin_iter(s, x);
    }
    // ---- an evaluation of the running line search ---------------------------------------------
    s.ifun++;
    s.gd = g[0] * s.d[0] + g[1] * s.d[1] + g[2] * s.d[2];
    bool ok = isfinite(f) && isfinite(s.gd);
    if (ok) {
        const int task = dcsrch_step(s.ls, s.stp, f, s.gd, ftol, gtol, xtol, 0.0, stpmx);
        if (task == LS_FG) {
            if (s.ifun >= 20) ok = false;
            else {
                for (int c = 0; c < 3; c++) x[c] = s.xold[c] + s.stp * s.d[c];
                return false;
            }
        }
    }
    if (!ok) {
        // line search failed: restore; with stored pairs restart from steepest descent, else stop
        s.f = s.fold;
        for (int c = 0; c < 3; c++) { x[c] = s.xold[c]; s.g[c] = s.gold[c]; }
        if (s.col == 0) return true;
        s.col = 0; s.head = 0; s.theta = 1.0;
        return lbfgs_begin_iter(s, x);
    }
    s.iter++;
    if (fmax(fabs(g[0]), fmax(fabs(g[1]), fabs(g[2]))) <= pgtol) return true;
    const double ddum = fmax(fabs(s.fold), fmax(fabs(f), 1.0));
    if (s.fold - f <= epsmch * factr * ddum) return true;
    // ---- update the limited-memory matrices ---------------------------------------------------
    double r[3], sv[3], rr = 0.0;
    for (int c = 0; c < 3; c++) { r[c] = g[c] - s.gold[c]; sv[c] = x[c] - s.xold[c]; rr += r[c] * r[c]; }
    double dr, dd;
    if (s.stp == 1.0) { dr = s.gd - s.gdold; dd = -s.gdold; }
    else { dr = (s.gd - s.gdold) * s.stp; dd = -s.gdold * s.stp; }
    if (dr > epsmch * dd) {
        int slot;
        if (s.col < kLbfgsM) { slot = (s.head + s.col) % kLbfgsM; s.col++; }
        else { slot = s.head; s.head = (s.head + 1) % kLbfgsM; }
        for (int c = 0; c < 3; c++) { s.S[slot][c] = sv[c]; s.Y[slot][c] = r[c]; }
        s.rho[slot] = 1.0 / dr;
        s.theta = rr / dr;
    }
    return lbfgs_begin_iter(s, x);
}

// one fit, evaluated and advanced in place, on the host: the numerical reference the CPU tests check through
// tad_debug_arima_fit (arima_fit_sync_kernel runs the same steps per lane)
void arima_fit(const ArimaObj &o, double x[3])
{
    Lbfgs s;
    lbfgs_init(s);
    for (;;) {
        double f, g[3];
        arima_fg(o, x, f, g);
        if (lbfgs_advance(s, x, f, g)) return;
    }
}

}  // namespace arima_core

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
// one thread per series: validity, Box-Cox lambda, transformed series into yb[]
__global__ void __launch_bounds__(128) arima_boxcox_kernel(const SeriesEntry *__restrict__ entries, const uint32_t *__restrict__ offsets,
                                                           const uint32_t *__restrict__ sbase, uint32_t B, uint32_t S,
                                                           const uint64_t *__restrict__ csr_v, double *__restrict__ yb,
                                                           double *__restrict__ lam)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const SeriesEntry e = load_entry(entries, offsets, sbase, B, i);
    const uint64_t *v = csr_v + e.off;
    double *y = yb + e.off;
    const uint32_t n = e.n;
    bool valid = n > 3;                                   // anomaly_detection.py:232-234
    bool constant = true;
    double sumlog = 0.0;
    for (uint32_t q = 0; q < n && valid; q++) {
        if (v[q] == 0) valid = false;                     // Box-Cox needs positive data (:260-264 -> None)
        if (v[q] != v[0]) constant = false;
        const double lx = log(__ull2double_rn(v[q]));
        y[q] = lx;
        sumlog += lx;
    }
    if (!valid || constant) { lam[i] = NAN; return; }
    const double l = boxcox_mle_lambda(y, n, sumlog);
    bool finite = isfinite(l);
    for (uint32_t q = 0; q < n && finite; q++) {
        y[q] = l == 0.0 ? y[q] : expm1(l * y[q]) / l;     // scipy.special.boxcox
        finite = isfinite(y[q]);
    }
    lam[i] = finite ? l : NAN;                             // overflowing transform -> the series yields no rows
}

// Evaluation-synchronous fits, pred[] in Box-Cox space: one warp per series; the prefix fits t = n-1 .. 3 form a job list
// that the lanes work through dynamically (longest first, so the fits in flight have similar lengths).  Every round, all
// lanes that hold a job evaluate the objective and its forward-difference gradient TOGETHER -- the same Kalman-filter loop,
// each lane on its own prefix and parameters -- then each lane advances its own optimiser state (lbfgs_advance) to the next
// trial point; a lane whose fit has ended writes its forecast and takes the next job.  Per fit the arithmetic is the same
// as in arima_fit: only the scheduling differs.
__global__ void __launch_bounds__(128) arima_fit_sync_kernel(const SeriesEntry *__restrict__ entries, const uint32_t *__restrict__ offsets,
                                                             const uint32_t *__restrict__ sbase, uint32_t B, uint32_t S,
                                                             const double *__restrict__ yb, const double *__restrict__ lam,
                                                             double *__restrict__ pred)
{
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (i >= S) return;                                    // warp-uniform
    if (isnan(lam[i])) return;
    const SeriesEntry e = load_entry(entries, offsets, sbase, B, i);
    const double *y = yb + e.off;
    double *p = pred + e.off;
    for (uint32_t t = lane; t < min(e.n, 3u); t += 32) p[t] = y[t];      // train = first three points (:241,255)
    int next = (int)e.n - 1;                               // next job to hand out (warp-uniform), down to 3
    bool busy = false;
    ArimaObj o{y, 0};
    double u[3] = {0.0, 0.0, 0.0};
    Lbfgs st;
    for (;;) {
        // ---- hand the next jobs to the idle lanes --------------------------------------------
        const uint32_t idle = __ballot_sync(0xffffffffu, !busy);
        if (idle && next >= 3) {
            const int rank = __popc(idle & ((1u << lane) - 1u));
            if (!busy && next - rank >= 3) {
                o.n = (uint32_t)(next - rank);
                arima_start(o, u);
                lbfgs_init(st);
                busy = true;
            }
            next -= __popc(idle);
        }
        if (!__any_sync(0xffffffffu, busy)) break;
        // ---- all busy lanes evaluate together -------------------------------------------------
        double f = 0.0, g[3] = {0.0, 0.0, 0.0};
        if (busy) arima_fg(o, u, f, g);
        __syncwarp();
        // ---- every lane advances its own optimiser --------------------------------------------
        if (busy && lbfgs_advance(st, u, f, g)) {
            double phi, theta, s2, fc = 0.0;
            arima_transform(u, phi, theta, s2);
            arima_loglike(o, phi, theta, s2, &fc);
            p[o.n] = fc;
            busy = false;
        }
        __syncwarp();
    }
}

// stddev_samp as in the other detectors (Welford, sequential in time order)
__device__ __forceinline__ double arima_stddev(const uint64_t *__restrict__ v, uint32_t n, bool &has_sd)
{
    double cnt = 0.0, avg = 0.0, m2 = 0.0;
    for (uint32_t i = 0; i < n; i++) {
        const double x = __ull2double_rn(v[i]);
        cnt = __dadd_rn(cnt, 1.0);
        const double d = __dsub_rn(x, avg);
        const double dn = __ddiv_rn(d, cnt);
        avg = __dadd_rn(avg, dn);
        m2 = __dadd_rn(m2, __dmul_rn(d, __dsub_rn(d, dn)));
    }
    has_sd = n >= 2;
    return has_sd ? __dsqrt_rn(__ddiv_rn(m2, __dsub_rn(cnt, 1.0))) : __longlong_as_double(0x7ff8000000000000LL);
}

__device__ __forceinline__ double inv_boxcox_d(double y, double l)
{
    return l == 0.0 ? exp(y) : exp(log1p(l * y) / l);     // scipy.special.inv_boxcox
}

template <int NT>
__global__ void __launch_bounds__(NT) detect_arima_kernel(const SeriesEntry *__restrict__ entries, const uint32_t *__restrict__ offsets,
                                                          const uint32_t *__restrict__ sbase, uint32_t B, uint32_t S,
                                                          const uint64_t *__restrict__ csr_v, const uint32_t *__restrict__ csr_t,
                                                          const double *__restrict__ pred, const double *__restrict__ lam,
                                                          OutCols out, uint32_t out_cap, uint32_t *__restrict__ stats, int emit_all)
{
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t total_s, base_s;
    const uint32_t i = blockIdx.x * NT + threadIdx.x;
    SeriesEntry e;
    e.n = 0;
    const uint64_t *v = nullptr;
    const double *p = nullptr;
    bool has_sd = false;
    double sd = 0.0, l = 0.0;
    uint32_t count = 0;
    if (i < S && !isnan(lam[i])) {                         // calc None -> the series contributes no rows
        e = load_entry(entries, offsets, sbase, B, i);
        l = lam[i];
        v = csr_v + e.off;
        p = pred + e.off;
        bool finite = true;
        for (uint32_t q = 0; q < e.n; q++) finite = finite && isfinite(inv_boxcox_d(p[q], l));
        if (!finite) e.n = 0;
        sd = arima_stddev(v, e.n, has_sd);
        if (emit_all) count = e.n;
        else if (has_sd)
            for (uint32_t q = 0; q < e.n; q++)
                count += fabs(__ull2double_rn(v[q]) - inv_boxcox_d(p[q], l)) > sd ? 1u : 0u;
    }
    // block exclusive scan of the counts
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = count;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < NT / 32 ? warp_sums[lane] : 0u;
        uint32_t winc = w;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        if (lane < NT / 32) warp_sums[lane] = winc - w;
        if (lane == NT / 32 - 1) total_s = winc;
    }
    __syncthreads();
    const uint32_t pre = warp_sums[warp] + inc - count;
    if (threadIdx.x == 0) base_s = total_s ? atomicAdd(&stats[ST_OUTCOUNT], total_s) : 0u;
    __syncthreads();
    if (count == 0) return;
    uint32_t idx = base_s + pre;
    const uint32_t *t = csr_t + e.off;
    for (uint32_t q = 0; q < e.n; q++) {
        const double x = __ull2double_rn(v[q]);
        const double calc = inv_boxcox_d(p[q], l);
        const bool flag = has_sd && fabs(x - calc) > sd;
        if (flag || emit_all) {
            if (idx < out_cap) {
                out.src_ip[idx] = (uint32_t)(e.a >> 32); out.dst_ip[idx] = (uint32_t)e.a;
                out.flow_start[idx] = (uint32_t)(e.b >> 32);
                out.src_port[idx] = (uint16_t)(e.b >> 16); out.dst_port[idx] = (uint16_t)e.b;
                out.proto[idx] = (uint8_t)e.proto; out.flow_end[idx] = t[q];
                out.stddev[idx] = sd; out.algo_calc[idx] = calc; out.throughput[idx] = x;
                out.anomaly[idx] = flag ? 1 : 0;
            }
            idx++;
        }
    }
}

cudaError_t launch_detect_arima(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase,
                                uint32_t B, uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, double *scratch_y,
                                double *scratch_pred, double *scratch_lam, bool fit, const OutCols &out, uint32_t out_cap,
                                uint32_t *stats, int emit_all)
{
    if (S == 0) return cudaSuccess;
    if (fit) {
        arima_boxcox_kernel<<<(S + 127) / 128, 128, 0, st>>>(entries, offsets, sbase, B, S, csr_v, scratch_y, scratch_lam);
        const uint64_t threads = (uint64_t)S * 32;
        arima_fit_sync_kernel<<<(uint32_t)((threads + 127) / 128), 128, 0, st>>>(entries, offsets, sbase, B, S, scratch_y,
                                                                                scratch_lam, scratch_pred);
    }
    constexpr int NT = 128;
    detect_arima_kernel<NT><<<(S + NT - 1) / NT, NT, 0, st>>>(entries, offsets, sbase, B, S, csr_v, csr_t, scratch_pred,
                                                             scratch_lam, out, out_cap, stats, emit_all);
    return cudaGetLastError();
}

}  // namespace tad

// Host-side hook for the CPU tests of the numerical core (not part of the C ABI in theia_tad.h): runs the
// same start-value / L-BFGS / Kalman code the kernels run, on the host, for one history.
extern "C" int tad_debug_arima_fit(const double *y, uint32_t n, double *u_out, double *forecast, double *lambda_of_logx)
{
    if (lambda_of_logx) {        // y holds log(x): return the Box-Cox MLE lambda instead
        double sumlog = 0.0;
        for (uint32_t i = 0; i < n; i++) sumlog += y[i];
        *lambda_of_logx = tad::boxcox_mle_lambda(y, n, sumlog);
        return 0;
    }
    tad::ArimaObj o{y, n};
    double u[3];
    tad::arima_start(o, u);
    if (u_out) { u_out[3] = u[0]; u_out[4] = u[1]; u_out[5] = u[2]; }
    tad::arima_fit(o, u);
    double phi, theta, s2, fc = 0.0;
    tad::arima_transform(u, phi, theta, s2);
    const double ll = tad::arima_loglike(o, phi, theta, s2, &fc);
    if (u_out) { u_out[0] = u[0]; u_out[1] = u[1]; u_out[2] = u[2]; u_out[6] = -ll / n; }
    if (forecast) *forecast = fc;
    return 0;
}
