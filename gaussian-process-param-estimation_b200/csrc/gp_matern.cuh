// Matern correlation device functions shared by the dense generator, the sparse generator and the
// on-the-fly dK/drho reductions. Follows gaussian_proc/generate_correlation/_kernels.pyx:17-100 branch by branch.
#pragma once
#include <math.h>
#include <stdint.h>
#include <type_traits>

namespace gp {

enum MaternMode { MAT_05 = 0, MAT_15 = 1, MAT_25 = 2, MAT_GAUSS = 3, MAT_GENERAL = 4 };

// branch selection of _kernels.pyx:76-93 (exact comparisons on nu, as the reference does)
static inline int matern_mode_of(double nu) {
    if (nu == 0.5) return MAT_05;
    if (nu == 1.5) return MAT_15;
    if (nu == 2.5) return MAT_25;
    if (nu < 100) return MAT_GENERAL;
    return MAT_GAUSS;
}

#ifdef __CUDACC__
// Modified Bessel K_nu(x) and K_{nu+1}(x) for real nu >= 0, x > 0: Temme's series for x <= 2, Steed's
// continued fraction CF2 for x > 2, then upward recurrence from the fractional order mu in [-1/2, 1/2].
// (Published algorithm: Temme 1975; Numerical Recipes `bessik`.) Used only for the general-nu Matern branch, on the device
// and by the host evaluation that decides the sparse generator's borderline pairs and support radius (gp_sparse.cu).
__host__ __device__ inline void bessel_k_pair(double nu, double x, double* knu, double* knu1) {
    const double EPS = 1e-16;
    const int MAXIT = 100000;
    int nl = (int)(nu + 0.5);
    double xmu = nu - nl, xmu2 = xmu * xmu;
    double xi = 1.0 / x, xi2 = 2.0 * xi;
    double rkmu, rk1;
    if (x < 2.0) {
        double b = 0.5 * x, d = -log(b), e = xmu * d;
        double fact2 = (fabs(e) < EPS) ? 1.0 : sinh(e) / e;
        const double PI = 3.14159265358979323846;
        double pimu = PI * xmu;
        double fact = (fabs(pimu) < EPS) ? 1.0 : pimu / sin(pimu);
        // gam1 = (1/Gamma(1-mu) - 1/Gamma(1+mu)) / (2 mu), gam2 = (1/Gamma(1-mu) + 1/Gamma(1+mu)) / 2
        double gampl = 1.0 / tgamma(1.0 + xmu), gammi = 1.0 / tgamma(1.0 - xmu);
        double gam2 = 0.5 * (gammi + gampl);
        double gam1;
        if (fabs(xmu) < 1e-4) {
            // series of gam1 around mu = 0: -gamma_E + c2 mu^2 (avoids cancellation)
            gam1 = -0.5772156649015329 + xmu2 * 0.04200263503409524;
        } else {
            gam1 = (gammi - gampl) / (2.0 * xmu);
        }
        double ff = fact * (gam1 * cosh(e) + gam2 * fact2 * d);
        double sum = ff;
        e = exp(e);
        double p = 0.5 * e / gampl, q = 0.5 / (e * gammi);
        double c = 1.0, d2 = b * b, sum1 = p;
        for (int i = 1; i <= MAXIT; ++i) {
            ff = (i * ff + p + q) / (i * i - xmu2);
            c *= (d2 / i);
            p /= (i - xmu);
            q /= (i + xmu);
            double del = c * ff;
            sum += del;
            double del1 = c * (p - i * ff);
            sum1 += del1;
            if (fabs(del) < fabs(sum) * EPS) break;
        }
        rkmu = sum;
        rk1 = sum1 * xi2;
    } else {
        double b = 2.0 * (1.0 + x), d = 1.0 / b, h = d, delh = d;
        double q1 = 0.0, q2 = 1.0, a1 = 0.25 - xmu2;
        double q = a1, c = a1, a = -a1;
        double s = 1.0 + q * delh;
        for (int i = 2; i <= MAXIT; ++i) {
            a -= 2 * (i - 1);
            c = -a * c / i;
            double qnew = (q1 - b * q2) / a;
            q1 = q2;
            q2 = qnew;
            q += c * qnew;
            b += 2.0;
            d = 1.0 / (b + a * d);
            delh = (b * d - 1.0) * delh;
            h += delh;
            double dels = q * delh;
            s += dels;
            if (fabs(dels / s) < EPS) break;
        }
        h = a1 * h;
        rkmu = sqrt(3.14159265358979323846 / (2.0 * x)) * exp(-x) / s;
        rk1 = rkmu * (xmu + x + 0.5 - h) * xi;
    }
    for (int i = 1; i <= nl; ++i) {
        double rktemp = (xmu + i) * xi2 * rk1 + rkmu;
        rkmu = rk1;
        rk1 = rktemp;
    }
    *knu = rkmu;
    *knu1 = rk1;
}

struct MaternParams {
    double nu;
    double coef;    // 2^(1-nu) / Gamma(nu)            (general branch, _kernels.pyx:87)
    double sq2nu;   // sqrt(2 nu)
    double inv_rho; // 1 / rho for dK/drho (isotropic)
    double inv_scale[8]; // 1 / correlation_scale[k]
    int ddim = -1;       // >= 0: derivative with respect to correlation_scale[ddim] alone (anisotropic gradient; inv_rho = 1)
};

// The parameter checks of every entry point that takes scale_host and nu, made before anything is enqueued: -3 when a scale
// entry is not > 0 (NaN included), -4 when `isotropic` (a d/drho is requested) and the d entries are not all equal, -5 when
// nu selects the general branch and is not > 0. NaN nu takes the Gaussian branch, as in the reference. gp_kernel_threshold,
// host-only and defined for any d, uses these checks alone; every other entry point calls matern_params.
static inline int matern_check(const double* scale_host, int64_t d, double nu, bool isotropic) {
    for (int64_t k = 0; k < d; ++k)
        if (!(scale_host[k] > 0.0)) return -3;
    if (isotropic)
        for (int64_t k = 1; k < d; ++k)
            if (scale_host[k] != scale_host[0]) return -4;
    if (matern_mode_of(nu) == MAT_GENERAL && !(nu > 0.0)) return -5;
    return 0;
}

// matern_check, then the kernel parameters (d <= 8) and the branch: mode is the template argument of the kernels, passed
// through with_matern_mode. ddim stays -1.
static inline int matern_params(const double* scale_host, int64_t d, double nu, bool isotropic, MaternParams* mp, int* mode) {
    if (int rc = matern_check(scale_host, d, nu, isotropic)) return rc;
    *mp = MaternParams();
    *mode = matern_mode_of(nu);
    mp->nu = nu;
    if (*mode == MAT_GENERAL) {
        mp->coef = pow(2.0, 1.0 - nu) / tgamma(nu);
        mp->sq2nu = sqrt(2.0 * nu);
    }
    mp->inv_rho = 1.0 / scale_host[0];
    for (int64_t k = 0; k < d; ++k) mp->inv_scale[k] = 1.0 / scale_host[k];
    return 0;
}

// f(std::integral_constant<int, MODE>()) for the run-time branch `mode`: instantiates f for each of the five branches.
template <class F>
decltype(auto) with_matern_mode(int mode, F&& f) {
    switch (mode) {
        case MAT_05: return f(std::integral_constant<int, MAT_05>());
        case MAT_15: return f(std::integral_constant<int, MAT_15>());
        case MAT_25: return f(std::integral_constant<int, MAT_25>());
        case MAT_GAUSS: return f(std::integral_constant<int, MAT_GAUSS>());
        default: return f(std::integral_constant<int, MAT_GENERAL>());
    }
}

// correlation value only; x is the scaled distance (>= 0). x == 0 -> exactly 1 (_kernels.pyx:73-74).
template <int MODE>
__device__ __forceinline__ double matern_value(double x, const MaternParams& p) {
    if (x == 0.0) return 1.0;
    if (MODE == MAT_05) return exp(-x);
    if (MODE == MAT_15) {
        const double s3 = 1.7320508075688772;  // sqrt(3.0), correctly rounded
        return (1.0 + s3 * x) * exp(-s3 * x);
    }
    if (MODE == MAT_25) {
        const double s5 = 2.23606797749979;  // sqrt(5.0), correctly rounded
        return (1.0 + s5 * x + (5.0 / 3.0) * (x * x)) * exp(-s5 * x);
    }
    if (MODE == MAT_GAUSS) return exp(-0.5 * (x * x));
    double y = p.sq2nu * x, k, k1;
    bessel_k_pair(p.nu, y, &k, &k1);
    return p.coef * pow(y, p.nu) * k;
}

// value and derivative with respect to an isotropic correlation scale rho (x = r / rho)
template <int MODE>
__device__ __forceinline__ void matern_value_drho(double x, const MaternParams& p, double* val, double* dval) {
    if (x == 0.0) { *val = 1.0; *dval = 0.0; return; }
    if (MODE == MAT_05) {
        double e = exp(-x);
        *val = e; *dval = x * p.inv_rho * e;
    } else if (MODE == MAT_15) {
        const double s3 = 1.7320508075688772;
        double e = exp(-s3 * x);
        *val = (1.0 + s3 * x) * e; *dval = 3.0 * x * x * p.inv_rho * e;
    } else if (MODE == MAT_25) {
        const double s5 = 2.23606797749979;
        double e = exp(-s5 * x);
        *val = (1.0 + s5 * x + (5.0 / 3.0) * (x * x)) * e;
        *dval = (5.0 / 3.0) * x * x * p.inv_rho * (1.0 + s5 * x) * e;
    } else if (MODE == MAT_GAUSS) {
        double e = exp(-0.5 * (x * x));
        *val = e; *dval = x * x * p.inv_rho * e;
    } else {
        // d/dy [y^nu K_nu(y)] = -y^nu K_{nu-1}(y), dy/drho = -y/rho; K_{nu-1} = K_{nu+1} - (2 nu / y) K_nu
        double y = p.sq2nu * x, k, k1;
        bessel_k_pair(p.nu, y, &k, &k1);
        double ynu = pow(y, p.nu);
        double km1 = k1 - (2.0 * p.nu / y) * k;
        *val = p.coef * ynu * k;
        *dval = p.coef * ynu * y * km1 * p.inv_rho;
    }
}

// h(x) = -K'(x) / x, the radial factor of the gradient with respect to a point: with t_k = (p_k - q_k) / scale_k and
// x = ||t||, dK/dq_k = h(x) t_k / scale_k. Each branch is written without the division by x (x^2 for the closed forms).
// x == 0 returns exactly 0: there t = 0, so a coincident pair contributes 0 (nu > 1/2: the true derivative; nu = 1/2, where
// K has a kink: the symmetric one) and h = inf (nu = 1/2, general nu <= 1) is never multiplied by 0.
template <int MODE>
__device__ __forceinline__ double matern_h(double x, const MaternParams& p) {
    if (x == 0.0) return 0.0;
    if (MODE == MAT_05) return exp(-x) / x;
    if (MODE == MAT_15) return 3.0 * exp(-1.7320508075688772 * x);
    if (MODE == MAT_25) {
        const double s5 = 2.23606797749979;
        return (5.0 / 3.0) * (1.0 + s5 * x) * exp(-s5 * x);
    }
    if (MODE == MAT_GAUSS) return exp(-0.5 * (x * x));
    // h = coef 2 nu y^(nu-1) K_{nu-1}(y), y = sqrt(2 nu) x; K_{nu-1} = K_{nu+1} - (2 nu / y) K_nu
    double y = p.sq2nu * x, k, k1;
    bessel_k_pair(p.nu, y, &k, &k1);
    return p.coef * (2.0 * p.nu) * pow(y, p.nu - 1.0) * (k1 - (2.0 * p.nu / y) * k);
}
#endif  // __CUDACC__

}  // namespace gp
