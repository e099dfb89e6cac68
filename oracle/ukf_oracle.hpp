/*
 * oracle/ukf_oracle.hpp -- CPU ORACLE.  TEST INFRASTRUCTURE ONLY.
 *
 * A dependency-free C++17 restatement of the reference's UKF hot path:
 * the in-tree wrapper code of rock-slam/slam-pose_estimation plus the algorithm
 * of its un-vendored dependency `slam/mtk` (ukfom::ukf<>, MTK::SO3, MTK::vect;
 * no version is pinned by the reference: manifest.xml:13, src/CMakeLists.txt:25).
 *
 *   PARITY PARTLY PINNED.  The reference holds no test, golden vector or fixture
 *   for any UKF quantity (test/CMakeLists.txt:1-4 builds only the GDAL projection
 *   test; test/test_models.cpp:1-10 is a dead stub) and its own build cannot run
 *   here (Rock CMake macros, Eigen, Boost, base-types, GDAL, LAPACK and slam/mtk
 *   are all absent).  What is pinned: the WRAPPER layers (models, process-noise
 *   shaping with its quirks, time guards and latches) -- oracle/_ref compiles the
 *   reference's own PoseUKF.cpp, OrientationUKF.cpp and UnscentedKalmanFilter.hpp
 *   unmodified against stand-in headers (oracle/ref_shim, oracle/ref_recipe.mk)
 *   and this oracle equals it bit for bit (tests/test_ref_pin.py).  What stays
 *   UNPINNED: the ukfom / MTK engine underneath (sigma points, manifold mean and
 *   its tolerance, update / apply_delta, SO(3) conventions), which the reference
 *   does not vendor: pinned only by (i) analytic known-answer tests and (ii) an
 *   independent NumPy/LAPACK restatement (oracle/numpy_ukf.py); tests/test_oracle.py.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may include, link or execute this code.  The product
 * (slam_pose_estimation_b200/) never does.
 *
 * Everything is a template over the scalar T so that the same code runs with
 * `double` (the oracle proper), with `long double` (liboracle_ld.so, the
 * extended-precision reference of tests/precision.py) and with a counting scalar
 * (oracle/count_ops.cpp) that measures the algorithmic flop / special-function
 * counts of SURVEY.md section 8(d).  Only inputs stay `double` (dt, z, R, the
 * stored IMU / acceleration samples, tau, the earth rate): every intermediate of
 * Ukf<T,S>, the models and rotate_block is a T.
 *
 * Each function cites the reference file:line (or the upstream MTK file) it follows.
 */
#ifndef UKF_ORACLE_HPP
#define UKF_ORACLE_HPP

#include <cfloat>
#include <cmath>
#include <cstdint>
#include <functional>
#include <limits>
#include <stdexcept>
#include <type_traits>
#include <vector>

#include "../include/ukfb_constants.h"

namespace orc {

using std::atan;
using std::cos;
using std::sin;
using std::sqrt;

/* status bits, same values as include/ukf_batch.h UKFB_STATUS_* */
enum : uint32_t {
    ST_NEG_DT = 1u,
    ST_DT_TOO_LARGE = 2u,
    ST_NONFINITE_MEAS = 4u,
    ST_NOT_SPD = 8u,
    ST_MEAN_NO_CONVERGE = 16u,
};

template <class T>
inline bool is_finite(const T& x) { return std::isfinite(static_cast<double>(x)); }

/* a floating-point scalar wider than double (the extended-precision reference) */
template <class T>
constexpr bool kWiderThanDouble = std::is_floating_point<T>::value && (sizeof(T) > sizeof(double));

/* 1/k: the double constant for double and for the counting scalar, rounded in T itself when T is wider */
template <class T>
inline T recip(int k)
{
    if constexpr (kWiderThanDouble<T>)
        return T(1) / T(k);
    else
        return T(1. / k);
}

/* ------------------------------------------------------------------------- */
/* Quaternion, Eigen::Quaternion<double> semantics, storage (x,y,z,w).         */
/* ------------------------------------------------------------------------- */
template <class T>
struct Quat {
    T x, y, z, w;
};

template <class T>
inline Quat<T> quat_identity() { return Quat<T>{T(0), T(0), T(0), T(1)}; }

/* Eigen quat_product (generic path): Hamilton product a*b. */
template <class T>
inline Quat<T> quat_mul(const Quat<T>& a, const Quat<T>& b)
{
    Quat<T> r;
    r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
    r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
    r.y = a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z;
    r.z = a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x;
    return r;
}

template <class T>
inline Quat<T> quat_conj(const Quat<T>& a) { return Quat<T>{-a.x, -a.y, -a.z, a.w}; }

/* Eigen QuaternionBase::inverse(): conjugate / squaredNorm (used at
 * OrientationUKF.cpp:38,76). */
template <class T>
inline Quat<T> quat_inverse(const Quat<T>& a)
{
    T n2 = a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
    return Quat<T>{-a.x / n2, -a.y / n2, -a.z / n2, a.w / n2};
}

/* Eigen QuaternionBase::_transformVector: uv = 2 (q.vec x v); v + w*uv + q.vec x uv.
 * (`orientation * velocity` at PoseUKF.cpp:80-81, OrientationUKF.cpp:19,22.) */
template <class T>
inline void quat_rotate(const Quat<T>& q, const T v[3], T out[3])
{
    T uvx = q.y * v[2] - q.z * v[1];
    T uvy = q.z * v[0] - q.x * v[2];
    T uvz = q.x * v[1] - q.y * v[0];
    uvx = uvx + uvx;
    uvy = uvy + uvy;
    uvz = uvz + uvz;
    out[0] = v[0] + q.w * uvx + (q.y * uvz - q.z * uvy);
    out[1] = v[1] + q.w * uvy + (q.z * uvx - q.x * uvz);
    out[2] = v[2] + q.w * uvz + (q.x * uvy - q.y * uvx);
}

/* Eigen QuaternionBase::toRotationMatrix (`orientation.matrix()` at
 * PoseUKF.cpp:182, OrientationUKF.cpp:81).  Row-major 3x3. */
template <class T>
inline void quat_matrix(const Quat<T>& q, T R[9])
{
    const T tx = T(2) * q.x, ty = T(2) * q.y, tz = T(2) * q.z;
    const T twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
    const T txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
    const T tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
    R[0] = T(1) - (tyy + tzz);
    R[1] = txy - twz;
    R[2] = txz + twy;
    R[3] = txy + twz;
    R[4] = T(1) - (txx + tzz);
    R[5] = tyz - twx;
    R[6] = txz - twy;
    R[7] = tyz + twx;
    R[8] = T(1) - (txx + tyy);
}

/* ------------------------------------------------------------------------- */
/* MTK math (mtk/src/mtkmath.hpp).                                            */
/* ------------------------------------------------------------------------- */

/* cos_sinc_sqrt(x2): (cos sqrt(x2), sin sqrt(x2) / sqrt(x2)); 3-term Taylor pair
 * below x2 < DBL_EPSILON^(1/4). */
template <class T>
inline void cos_sinc_sqrt(const T& x2, T& c, T& sinc)
{
    if (x2 >= T(UKFB_TAYLOR_N_BOUND)) {
        T x = sqrt(x2);
        c = cos(x);
        sinc = sin(x) / x;
        return;
    }
    T cosi = T(1), si = T(1);
    T term = T(-1 / 2.) * x2;
    for (int i = 0; i < 3; ++i) {
        cosi = cosi + term;
        term = term * recip<T>(2 * i + 3);
        si = si + term;
        term = term * (-recip<T>(2 * i + 4) * x2);
    }
    c = cosi;
    sinc = si;
}

/* MTK::SO3::exp(vec, scale): w = cos, vec = sinc*(scale/2)*v with the angle
 * (scale/2)*|v|  (SOn.hpp exp -> mtkmath.hpp exp<scalar,3>). */
template <class T>
inline Quat<T> so3_exp(const T v[3], const T& scale)
{
    const T half = scale / T(2);
    const T norm2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    T c, sinc;
    cos_sinc_sqrt(half * half * norm2, c, sinc);
    const T mult = sinc * half;
    return Quat<T>{mult * v[0], mult * v[1], mult * v[2], c};
}

/* MTK::SO3::log(q): (2/nv) * atan(nv / w) * q.vec with nv floored at
 * MTK::tolerance (mtkmath.hpp log<scalar,3>, plus_minus_periodicity = true,
 * which makes q and -q equivalent). */
template <class T>
inline void so3_log(const Quat<T>& q, T out[3])
{
    T nv = sqrt(q.x * q.x + q.y * q.y + q.z * q.z);
    if (nv < T(UKFB_MTK_TOLERANCE)) nv = T(UKFB_MTK_TOLERANCE);
    const T s = T(2) / nv * atan(nv / q.w);
    out[0] = s * q.x;
    out[1] = s * q.y;
    out[2] = s * q.z;
}

/* MTK::SO3::boxplus / boxminus with the frame switch of ukfb_constants.h. */
template <class T>
inline void so3_boxplus(Quat<T>& q, const T v[3], const T& scale)
{
    const Quat<T> d = so3_exp(v, scale);
#if UKFB_SO3_BOXPLUS_LEFT
    q = quat_mul(d, q);
#else
    q = quat_mul(q, d);
#endif
}

template <class T>
inline void so3_boxminus(const Quat<T>& q, const Quat<T>& other, T res[3])
{
#if UKFB_SO3_BOXPLUS_LEFT
    so3_log(quat_mul(q, quat_conj(other)), res);
#else
    so3_log(quat_mul(quat_conj(other), q), res);
#endif
}

/* ------------------------------------------------------------------------- */
/* Manifolds.  MTK::vect boxplus: x += s*v; boxminus: x - o (mtk/types/vect.hpp). */
/* Compound manifolds apply member-wise in declaration order                   */
/* (mtk/build_manifold.hpp).                                                   */
/* ------------------------------------------------------------------------- */
template <class T, int M>
struct EuclidMeas { /* plain Eigen::Matrix<double,M,1> measurement */
    enum { DOF = M, EUCLID = 1 };
    T a[M];
    void boxplus(const T* d, const T& s = T(1))
    {
        for (int i = 0; i < M; ++i) a[i] = a[i] + s * d[i];
    }
    void boxminus(T* res, const EuclidMeas& o) const
    {
        for (int i = 0; i < M; ++i) res[i] = a[i] - o.a[i];
    }
};

template <class T>
struct RotMeas { /* RotationType = mtkwrap<MTK::SO3<double>> as a measurement */
    enum { DOF = 3, EUCLID = 0 };
    Quat<T> q;
    void boxplus(const T* d, const T& s = T(1)) { so3_boxplus(q, d, s); }
    void boxminus(T* res, const RotMeas& o) const { so3_boxminus(q, o.q, res); }
};

/* PoseWithVelocity (PoseWithVelocity.hpp:18-23). */
template <class T>
struct PoseState {
    enum { DOF = UKFB_POSE_DOF, MU = UKFB_POSE_MU };
    T position[3];
    Quat<T> orientation;
    T velocity[3];
    T angular_velocity[3];

    void boxplus(const T* d, const T& s = T(1))
    {
        for (int i = 0; i < 3; ++i) position[i] = position[i] + s * d[i];
        so3_boxplus(orientation, d + 3, s);
        for (int i = 0; i < 3; ++i) velocity[i] = velocity[i] + s * d[6 + i];
        for (int i = 0; i < 3; ++i) angular_velocity[i] = angular_velocity[i] + s * d[9 + i];
    }
    void boxminus(T* res, const PoseState& o) const
    {
        for (int i = 0; i < 3; ++i) res[i] = position[i] - o.position[i];
        so3_boxminus(orientation, o.orientation, res + 3);
        for (int i = 0; i < 3; ++i) res[6 + i] = velocity[i] - o.velocity[i];
        for (int i = 0; i < 3; ++i) res[9 + i] = angular_velocity[i] - o.angular_velocity[i];
    }
    void load(const double* m)
    {
        for (int i = 0; i < 3; ++i) position[i] = T(m[i]);
        orientation = Quat<T>{T(m[3]), T(m[4]), T(m[5]), T(m[6])};
        for (int i = 0; i < 3; ++i) velocity[i] = T(m[7 + i]);
        for (int i = 0; i < 3; ++i) angular_velocity[i] = T(m[10 + i]);
    }
    void store(double* m) const
    {
        for (int i = 0; i < 3; ++i) m[i] = double(position[i]);
        m[3] = double(orientation.x), m[4] = double(orientation.y);
        m[5] = double(orientation.z), m[6] = double(orientation.w);
        for (int i = 0; i < 3; ++i) m[7 + i] = double(velocity[i]);
        for (int i = 0; i < 3; ++i) m[10 + i] = double(angular_velocity[i]);
    }
};

/* OrientationState (OrientationState.hpp:20-26). */
template <class T>
struct OrientationState {
    enum { DOF = UKFB_ORI_DOF, MU = UKFB_ORI_MU };
    Quat<T> orientation;
    T velocity[3];
    T bias_gyro[3];
    T bias_acc[3];
    T gravity[1];

    void boxplus(const T* d, const T& s = T(1))
    {
        so3_boxplus(orientation, d, s);
        for (int i = 0; i < 3; ++i) velocity[i] = velocity[i] + s * d[3 + i];
        for (int i = 0; i < 3; ++i) bias_gyro[i] = bias_gyro[i] + s * d[6 + i];
        for (int i = 0; i < 3; ++i) bias_acc[i] = bias_acc[i] + s * d[9 + i];
        gravity[0] = gravity[0] + s * d[12];
    }
    void boxminus(T* res, const OrientationState& o) const
    {
        so3_boxminus(orientation, o.orientation, res);
        for (int i = 0; i < 3; ++i) res[3 + i] = velocity[i] - o.velocity[i];
        for (int i = 0; i < 3; ++i) res[6 + i] = bias_gyro[i] - o.bias_gyro[i];
        for (int i = 0; i < 3; ++i) res[9 + i] = bias_acc[i] - o.bias_acc[i];
        res[12] = gravity[0] - o.gravity[0];
    }
    void load(const double* m)
    {
        orientation = Quat<T>{T(m[0]), T(m[1]), T(m[2]), T(m[3])};
        for (int i = 0; i < 3; ++i) velocity[i] = T(m[4 + i]);
        for (int i = 0; i < 3; ++i) bias_gyro[i] = T(m[7 + i]);
        for (int i = 0; i < 3; ++i) bias_acc[i] = T(m[10 + i]);
        gravity[0] = T(m[13]);
    }
    void store(double* m) const
    {
        m[0] = double(orientation.x), m[1] = double(orientation.y);
        m[2] = double(orientation.z), m[3] = double(orientation.w);
        for (int i = 0; i < 3; ++i) m[4 + i] = double(velocity[i]);
        for (int i = 0; i < 3; ++i) m[7 + i] = double(bias_gyro[i]);
        for (int i = 0; i < 3; ++i) m[10 + i] = double(bias_acc[i]);
        m[13] = double(gravity[0]);
    }
};

/* ------------------------------------------------------------------------- */
/* Small dense helpers (row-major).                                            */
/* ------------------------------------------------------------------------- */

/* lapack::cholesky<n> (ukfom/lapack/cholesky.hpp) -> LAPACK dpotrf('L'); for
 * n = 12/13 that is the unblocked dpotf2: per column a dot-product update, a
 * sqrt, then a scale by the reciprocal (DSCAL with ONE/AJJ).  Upper triangle
 * zeroed.  Returns false when a pivot is not positive (not SPD). */
template <class T, int N>
inline bool cholesky_lower(const T* A, T* L)
{
    for (int i = 0; i < N * N; ++i) L[i] = T(0);
    for (int j = 0; j < N; ++j) {
        T ajj = A[j * N + j];
        for (int k = 0; k < j; ++k) ajj = ajj - L[j * N + k] * L[j * N + k];
        if (!(ajj > T(0)) || !is_finite(ajj)) return false;
        ajj = sqrt(ajj);
        L[j * N + j] = ajj;
        const T r = T(1) / ajj;
        for (int i = j + 1; i < N; ++i) {
            T s = A[i * N + j];
            for (int k = 0; k < j; ++k) s = s - L[i * N + k] * L[j * N + k];
            L[i * N + j] = s * r;
        }
    }
    return true;
}

/* Eigen fixed-size inverse() for 1x1 / 2x2 / 3x3 (compute_inverse_size{2,3}
 * helpers): closed-form cofactors over the determinant, not a factorisation. */
template <class T, int M>
inline void small_inverse(const T* S, T* Si)
{
    static_assert(M >= 1 && M <= 3, "measurement dimension 1..3");
    if (M == 1) {
        Si[0] = T(1) / S[0];
    } else if (M == 2) {
        const T det = S[0] * S[3] - S[1] * S[2];
        const T invdet = T(1) / det;
        Si[0] = S[3] * invdet;
        Si[1] = -S[1] * invdet;
        Si[2] = -S[2] * invdet;
        Si[3] = S[0] * invdet;
    } else {
        auto m = [&](int i, int j) -> const T& { return S[i * 3 + j]; };
        auto cof = [&](int i, int j) {
            const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
            return m(i1, j1) * m(i2, j2) - m(i1, j2) * m(i2, j1);
        };
        const T c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
        const T det = c00 * m(0, 0) + c10 * m(1, 0) + c20 * m(2, 0);
        const T invdet = T(1) / det;
        Si[0] = c00 * invdet;
        Si[1] = c10 * invdet;
        Si[2] = c20 * invdet;
        Si[3] = cof(0, 1) * invdet;
        Si[4] = cof(1, 1) * invdet;
        Si[5] = cof(2, 1) * invdet;
        Si[6] = cof(0, 2) * invdet;
        Si[7] = cof(1, 2) * invdet;
        Si[8] = cof(2, 2) * invdet;
    }
}

/* ------------------------------------------------------------------------- */
/* ukfom::ukf<state> (ukfom/ukf.hpp), SURVEY.md App. A.2 - A.4.                */
/* ------------------------------------------------------------------------- */
template <class T, class S>
class Ukf {
public:
    enum { n = S::DOF, NS = 2 * S::DOF + 1 };

    S mu;
    T sigma[n * n];
    /* the `accept` functor slot of ukfom::ukf::update.  The reference passes accept_any_mahalanobis_distance
     * (PoseUKF.cpp:116): accept_max_d2 = +inf.  A finite value models ukfom::accept_mahalanobis_distance(threshold):
     * a measurement with innov^T S^-1 innov > threshold leaves the filter untouched. */
    double accept_max_d2 = std::numeric_limits<double>::infinity();
    bool last_update_rejected = false;
    uint32_t status = 0;
    /* histogram of sigma_points_mean trip counts (number of mean passes) */
    uint64_t mean_iters[8] = {0, 0, 0, 0, 0, 0, 0, 0};

    /* A.2: X0 = mu + delta, X(2j+1) = mu + (delta + L[:,j]), X(2j+2) = mu + (delta - L[:,j]).
     * No sqrt(n+lambda) scaling.  Returns false (and flags) if sigma is not SPD. */
    bool generate_sigma_points(const T* delta, std::vector<S>& X)
    {
        T L[n * n];
        if (!cholesky_lower<T, n>(sigma, L)) {
            status |= ST_NOT_SPD;
            return false;
        }
        X.assign(NS, mu);
        T d[n];
        for (int i = 0; i < n; ++i) d[i] = delta ? delta[i] : T(0);
        X[0].boxplus(d);
        for (int j = 0; j < n; ++j) {
            T dp[n], dm[n];
            for (int i = 0; i < n; ++i) {
                dp[i] = d[i] + L[i * n + j];
                dm[i] = d[i] - L[i * n + j];
            }
            X[1 + 2 * j].boxplus(dp);
            X[2 + 2 * j].boxplus(dm);
        }
        return true;
    }

    /* A.3 sigma_points_mean: iterate ref += mean(X_i [-] ref) while |mean| > tol && ++i < max_it. */
    template <class M>
    M sigma_points_mean(const std::vector<M>& X)
    {
        constexpr int m = M::DOF;
        M ref = X[0];
        T mean_delta[m];
        std::size_t it = 0;
        std::size_t passes = 0;
        T norm;
        do {
            for (int k = 0; k < m; ++k) mean_delta[k] = T(0);
            for (const M& Xi : X) {
                T d[m];
                Xi.boxminus(d, ref);
                for (int k = 0; k < m; ++k) mean_delta[k] = mean_delta[k] + d[k];
            }
            const T cnt = T(double(X.size()));
            T n2 = T(0);
            for (int k = 0; k < m; ++k) {
                mean_delta[k] = mean_delta[k] / cnt;
                n2 = n2 + mean_delta[k] * mean_delta[k];
            }
            ref.boxplus(mean_delta);
            norm = sqrt(n2);
            ++passes;
        } while (norm > T(UKFB_MEAN_TOL) && ++it < std::size_t(UKFB_MEAN_MAX_IT));
        if (it >= std::size_t(UKFB_MEAN_MAX_IT)) status |= ST_MEAN_NO_CONVERGE;
        if (std::is_same<M, S>::value) mean_iters[passes < 7 ? passes : 7]++;
        return ref;
    }

    /* upstream's Euclidean special case: sum / N (UKFB_EUCLID_MEAS_DIRECT_MEAN = 1). */
    template <class M>
    M direct_mean(const std::vector<M>& Z)
    {
        constexpr int m = M::DOF;
        M r;
        for (int k = 0; k < m; ++k) r.a[k] = T(0);
        for (const M& Zi : Z)
            for (int k = 0; k < m; ++k) r.a[k] = r.a[k] + Zi.a[k];
        for (int k = 0; k < m; ++k) r.a[k] = r.a[k] / T(double(Z.size()));
        return r;
    }

    /* A.3 sigma_points_cov: 0.5 * sum (V_i [-] mean)(V_i [-] mean)^T, all 2n+1 points. */
    template <class M>
    void sigma_points_cov(const M& mean, const std::vector<M>& V, T* C)
    {
        constexpr int m = M::DOF;
        for (int i = 0; i < m * m; ++i) C[i] = T(0);
        for (const M& Vi : V) {
            T d[m];
            Vi.boxminus(d, mean);
            for (int a = 0; a < m; ++a)
                for (int b = 0; b < m; ++b) C[a * m + b] = C[a * m + b] + d[a] * d[b];
        }
        for (int i = 0; i < m * m; ++i) C[i] = T(0.5) * C[i];
    }

    /* A.4 sigma_points_cross_cov: 0.5 * sum (X_i [-] meanX)(Z_i [-] meanZ)^T. */
    template <class M>
    void sigma_points_cross_cov(const S& meanX, const M& meanZ, const std::vector<S>& X,
                                const std::vector<M>& Z, T* C)
    {
        constexpr int m = M::DOF;
        for (int i = 0; i < n * m; ++i) C[i] = T(0);
        for (std::size_t p = 0; p < X.size(); ++p) {
            T dx[n], dz[m];
            X[p].boxminus(dx, meanX);
            Z[p].boxminus(dz, meanZ);
            for (int a = 0; a < n; ++a)
                for (int b = 0; b < m; ++b) C[a * m + b] = C[a * m + b] + dx[a] * dz[b];
        }
        for (int i = 0; i < n * m; ++i) C[i] = T(0.5) * C[i];
    }

    /* A.3 predict(g, Q): sigma points -> g -> manifold mean -> cov + Q. */
    template <class G>
    void predict(G g, const T* Q)
    {
        std::vector<S> X;
        if (!generate_sigma_points(nullptr, X)) return;
        for (S& Xi : X) Xi = g(Xi);
        mu = sigma_points_mean(X);
        T C[n * n];
        sigma_points_cov(mu, X, C);
        for (int i = 0; i < n * n; ++i) sigma[i] = C[i] + Q[i];
    }

    /* A.4 apply_delta: re-draw sigma points around mu [+] delta with the updated sigma. */
    void apply_delta(const T* delta)
    {
        std::vector<S> X;
        if (!generate_sigma_points(delta, X)) return;
        mu = sigma_points_mean(X);
        sigma_points_cov(mu, X, sigma);
    }

    /* A.4 update(z, h, R, accept_any): K = Sxz S^-1, sigma -= K S K^T, apply_delta(K innov).
     * accept_any_mahalanobis_distance always accepts (PoseUKF.cpp:116). */
    template <class M, class H>
    void update(const M& z, H h, const T* R)
    {
        constexpr int m = M::DOF;
        std::vector<S> X;
        last_update_rejected = false;
        if (!generate_sigma_points(nullptr, X)) return;
        std::vector<M> Z(X.size());
        for (std::size_t p = 0; p < X.size(); ++p) Z[p] = h(X[p]);

        M meanZ;
        if (M::EUCLID && UKFB_EUCLID_MEAS_DIRECT_MEAN)
            meanZ = direct_mean_dispatch(Z);
        else
            meanZ = sigma_points_mean(Z);

        T Smat[m * m], Sxz[n * m], Sinv[m * m], K[n * m];
        sigma_points_cov(meanZ, Z, Smat);
        for (int i = 0; i < m * m; ++i) Smat[i] = Smat[i] + R[i];
        sigma_points_cross_cov(mu, meanZ, X, Z, Sxz);
        small_inverse<T, m>(Smat, Sinv);

        for (int a = 0; a < n; ++a)
            for (int b = 0; b < m; ++b) {
                T s = T(0);
                for (int k = 0; k < m; ++k) s = s + Sxz[a * m + k] * Sinv[k * m + b];
                K[a * m + b] = s;
            }

        T innov[m];
        z.boxminus(innov, meanZ);

        /* mahalanobis2 = innov^T Sinv innov; the reference's accept functor always accepts */
        {
            T d2 = T(0);
            for (int a = 0; a < m; ++a) {
                T s = T(0);
                for (int b = 0; b < m; ++b) s = s + Sinv[a * m + b] * innov[b];
                d2 = d2 + innov[a] * s;
            }
            last_update_rejected = double(d2) > accept_max_d2;
            if (last_update_rejected) return;
        }

        /* sigma -= (K * S) * K^T  (Eigen evaluates left to right) */
        T KS[n * m];
        for (int a = 0; a < n; ++a)
            for (int b = 0; b < m; ++b) {
                T s = T(0);
                for (int k = 0; k < m; ++k) s = s + K[a * m + k] * Smat[k * m + b];
                KS[a * m + b] = s;
            }
        for (int a = 0; a < n; ++a)
            for (int b = 0; b < n; ++b) {
                T s = T(0);
                for (int k = 0; k < m; ++k) s = s + KS[a * m + k] * K[b * m + k];
                sigma[a * n + b] = sigma[a * n + b] - s;
            }

        T delta[n];
        for (int a = 0; a < n; ++a) {
            T s = T(0);
            for (int k = 0; k < m; ++k) s = s + K[a * m + k] * innov[k];
            delta[a] = s;
        }
        apply_delta(delta);
    }

private:
    template <class M>
    M direct_mean_dispatch(const std::vector<M>& Z)
    {
        if constexpr (M::EUCLID)
            return direct_mean(Z);
        else
            return sigma_points_mean(Z);
    }
};

/* ------------------------------------------------------------------------- */
/* UnscentedKalmanFilter<Manifold> shell (UnscentedKalmanFilter.hpp:15-155).   */
/* ------------------------------------------------------------------------- */
template <class T, class S>
class FilterShell {
public:
    enum { n = S::DOF };

    /* :27-33 */
    FilterShell()
    {
        for (int i = 0; i < n * n; ++i) process_noise_cov[i] = T(0);
        last_measurement_time_us = 0;
        min_time_delta = UKFB_DEFAULT_MIN_DT;
        max_time_delta = std::numeric_limits<double>::max();
    }
    virtual ~FilterShell() {}

    /* :40-44 -- a fresh ukf and a reset time latch */
    void initializeFilter(const S& initial_state, const T* state_cov)
    {
        ukf = Ukf<T, S>();
        ukf.mu = initial_state;
        for (int i = 0; i < n * n; ++i) ukf.sigma[i] = state_cov[i];
        initialized = true;
        last_measurement_time_us = 0;
    }

    /* :51-60 */
    bool getCurrentState(S& state, T* state_cov) const
    {
        if (!initialized) return false;
        state = ukf.mu;
        for (int i = 0; i < n * n; ++i) state_cov[i] = ukf.sigma[i];
        return true;
    }

    /* :83-100 -- first call latches only; latch iff delta > min; forwards delta (also negative). */
    void predictionStepFromSampleTime(int64_t sample_time_us)
    {
        if (last_measurement_time_us == 0) {
            last_measurement_time_us = sample_time_us;
            return;
        }
        const double delta_t = double(sample_time_us - last_measurement_time_us) / UKFB_US_PER_S;
        if (delta_t > min_time_delta) last_measurement_time_us = sample_time_us;
        predictionStep(delta_t);
    }

    /* :107-125 */
    void predictionStep(double delta_t)
    {
        if (delta_t < 0.0)
            throw std::runtime_error("Delta time is negative!");
        else if (delta_t <= min_time_delta)
            return;
        else if (delta_t > max_time_delta)
            throw std::runtime_error("Delta time is greater then the allowed maximum!");
        predictionStepImpl(delta_t);
    }

    /* :142-147 */
    template <int DIM>
    static void checkMeasurment(const double* mu, const double* cov)
    {
        bool ok = true;
        for (int i = 0; i < DIM; ++i) ok = ok && std::isfinite(mu[i]);
        for (int i = 0; i < DIM * DIM; ++i) ok = ok && std::isfinite(cov[i]);
        if (!ok) throw std::runtime_error("Measurement or covariance contains non-finite values!");
    }

    bool initialized = false;
    Ukf<T, S> ukf;
    T process_noise_cov[n * n];
    int64_t last_measurement_time_us;
    double max_time_delta;
    double min_time_delta;

protected:
    virtual void predictionStepImpl(double delta_t) = 0;

    /* dst[off:off+3, off:off+3] = rot * src[off:off+3, off:off+3] * rot^T  (MTK::subblock) */
    static void rotate_block(T* dst, const T* src, const T* rot, int off)
    {
        T tmp[9];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                T s = T(0);
                for (int k = 0; k < 3; ++k) s = s + rot[i * 3 + k] * src[(off + k) * n + off + j];
                tmp[i * 3 + j] = s;
            }
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                T s = T(0);
                for (int k = 0; k < 3; ++k) s = s + tmp[i * 3 + k] * rot[j * 3 + k];
                dst[(off + i) * n + off + j] = s;
            }
    }
};

/* measurement kinds, same values as include/ukf_batch.h UKFB_MEAS_* */
enum MeasKind : int {
    MEAS_POSE_POSITION = 0,
    MEAS_POSE_XY = 1,
    MEAS_POSE_Z = 2,
    MEAS_POSE_ORIENTATION = 3,
    MEAS_POSE_VELOCITY = 4,
    MEAS_POSE_XY_VELOCITY = 5,
    MEAS_POSE_Z_VELOCITY = 6,
    MEAS_POSE_XVEL_YAWVEL = 7,
    MEAS_POSE_ANGULAR_VELOCITY = 8,
    MEAS_ORI_VELOCITY = 9,
};

inline int meas_dim(int kind)
{
    switch (kind) {
        case MEAS_POSE_XY:
        case MEAS_POSE_XY_VELOCITY:
        case MEAS_POSE_XVEL_YAWVEL: return 2;
        case MEAS_POSE_Z:
        case MEAS_POSE_Z_VELOCITY: return 1;
        default: return 3;
    }
}

/* ------------------------------------------------------------------------- */
/* PoseUKF (PoseUKF.hpp:17-93, PoseUKF.cpp).                                   */
/* ------------------------------------------------------------------------- */
template <class T>
class PoseFilter : public FilterShell<T, PoseState<T>> {
    typedef FilterShell<T, PoseState<T>> Base;
    typedef PoseState<T> S;
    enum { n = S::DOF };

public:
    double acc_mu[3];
    double acc_cov[9];

    /* PoseUKF.cpp:99-110 */
    PoseFilter(const S& initial_state, const T* state_cov)
    {
        this->initializeFilter(initial_state, state_cov);
        for (int i = 0; i < n * n; ++i) this->process_noise_cov[i] = T(0);
        for (int i = 0; i < 3; ++i) {
            this->process_noise_cov[(0 + i) * n + 0 + i] = T(UKFB_POSE_Q_POSITION);
            this->process_noise_cov[(3 + i) * n + 3 + i] = T(UKFB_POSE_Q_ORIENTATION);
            this->process_noise_cov[(6 + i) * n + 6 + i] = T(UKFB_POSE_Q_VELOCITY);
            this->process_noise_cov[(9 + i) * n + 9 + i] = T(UKFB_POSE_Q_ANGULAR_VELOCITY);
        }
        for (int i = 0; i < 3; ++i) acc_mu[i] = std::numeric_limits<double>::quiet_NaN();
        for (int i = 0; i < 9; ++i) acc_cov[i] = (i % 4 == 0) ? 1.0 : 0.0; /* Measurement.hpp:11 */
    }

    /* PoseUKF.cpp:175-178 -- stored without a finite check */
    void setAcceleration(const double* mu, const double* cov)
    {
        for (int i = 0; i < 3; ++i) acc_mu[i] = mu[i];
        for (int i = 0; i < 9; ++i) acc_cov[i] = cov[i];
    }

    /* The nine integrateMeasurement overloads, PoseUKF.cpp:112-173, selected by kind;
     * measurement models PoseUKF.cpp:7-69. */
    void integrateMeasurement(int kind, const double* zmu, const double* zcov)
    {
        switch (kind) {
            case MEAS_POSE_POSITION:
                upd<3>(zmu, zcov, [](const S& s, T* z) { z[0] = s.position[0], z[1] = s.position[1], z[2] = s.position[2]; });
                break;
            case MEAS_POSE_XY:
                upd<2>(zmu, zcov, [](const S& s, T* z) { z[0] = s.position[0], z[1] = s.position[1]; });
                break;
            case MEAS_POSE_Z:
                upd<1>(zmu, zcov, [](const S& s, T* z) { z[0] = s.position[2]; });
                break;
            case MEAS_POSE_ORIENTATION: {
                /* PoseUKF.cpp:133-138: z = SO3::exp(mu), h = state.orientation */
                T v[3] = {T(zmu[0]), T(zmu[1]), T(zmu[2])};
                RotMeas<T> z;
                z.q = so3_exp(v, T(1));
                T R[9];
                for (int i = 0; i < 9; ++i) R[i] = T(zcov[i]);
                this->ukf.update(z, [](const S& s) { RotMeas<T> r; r.q = s.orientation; return r; }, R);
                break;
            }
            case MEAS_POSE_VELOCITY:
                upd<3>(zmu, zcov, [](const S& s, T* z) { z[0] = s.velocity[0], z[1] = s.velocity[1], z[2] = s.velocity[2]; });
                break;
            case MEAS_POSE_XY_VELOCITY:
                upd<2>(zmu, zcov, [](const S& s, T* z) { z[0] = s.velocity[0], z[1] = s.velocity[1]; });
                break;
            case MEAS_POSE_Z_VELOCITY:
                upd<1>(zmu, zcov, [](const S& s, T* z) { z[0] = s.velocity[2]; });
                break;
            case MEAS_POSE_XVEL_YAWVEL:
                upd<2>(zmu, zcov, [](const S& s, T* z) { z[0] = s.velocity[0], z[1] = s.angular_velocity[2]; });
                break;
            case MEAS_POSE_ANGULAR_VELOCITY:
                upd<3>(zmu, zcov, [](const S& s, T* z) { z[0] = s.angular_velocity[0], z[1] = s.angular_velocity[1], z[2] = s.angular_velocity[2]; });
                break;
            default: throw std::invalid_argument("bad PoseUKF measurement kind");
        }
    }

    /* PoseUKF.cpp:75-83 -- both rotations use the input orientation. */
    static S processModel(const S& state, const T& dt)
    {
        S ns(state);
        T rv[3], rw[3];
        quat_rotate(ns.orientation, ns.velocity, rv);
        for (int i = 0; i < 3; ++i) ns.position[i] = ns.position[i] + dt * rv[i];
        quat_rotate(ns.orientation, ns.angular_velocity, rw);
        so3_boxplus(ns.orientation, rw, dt);
        return ns;
    }

    /* PoseUKF.cpp:88-97 */
    static S processModelWithAcceleration(const S& state, const T acc[3], const T& dt)
    {
        S ns(state);
        for (int i = 0; i < 3; ++i) ns.velocity[i] = ns.velocity[i] + dt * acc[i];
        T rv[3], rw[3];
        quat_rotate(ns.orientation, ns.velocity, rv);
        for (int i = 0; i < 3; ++i) ns.position[i] = ns.position[i] + dt * rv[i];
        quat_rotate(ns.orientation, ns.angular_velocity, rw);
        so3_boxplus(ns.orientation, rw, dt);
        return ns;
    }

protected:
    /* PoseUKF.cpp:180-196, including the shadowed `process_noise` of :190. */
    void predictionStepImpl(double delta) override
    {
        T rot[9];
        quat_matrix(this->ukf.mu.orientation, rot);
        T process_noise[n * n];
        for (int i = 0; i < n * n; ++i) process_noise[i] = this->process_noise_cov[i];
        Base::rotate_block(process_noise, this->process_noise_cov, rot, 0);
        Base::rotate_block(process_noise, this->process_noise_cov, rot, 3);
        for (int i = 0; i < n * n; ++i) process_noise[i] = T(delta) * process_noise[i];

        const bool acc_finite = std::isfinite(acc_mu[0]) && std::isfinite(acc_mu[1]) && std::isfinite(acc_mu[2]);
        if (acc_finite) {
            T pn[n * n]; /* the shadowing local: unrotated, unscaled Q */
            for (int i = 0; i < n * n; ++i) pn[i] = this->process_noise_cov[i];
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) pn[(6 + i) * n + 6 + j] = T(2.0) * T(acc_cov[i * 3 + j]);
            const T a[3] = {T(acc_mu[0]), T(acc_mu[1]), T(acc_mu[2])};
            const T dt = T(delta);
            this->ukf.predict([&](const S& s) { return processModelWithAcceleration(s, a, dt); }, pn);
        } else {
            const T dt = T(delta);
            this->ukf.predict([&](const S& s) { return processModel(s, dt); }, process_noise);
        }
    }

private:
    template <int M, class Sel>
    void upd(const double* zmu, const double* zcov, Sel sel)
    {
        EuclidMeas<T, M> z;
        T R[M * M];
        for (int i = 0; i < M; ++i) z.a[i] = T(zmu[i]);
        for (int i = 0; i < M * M; ++i) R[i] = T(zcov[i]);
        this->ukf.update(z, [&](const S& s) { EuclidMeas<T, M> r; sel(s, r.a); return r; }, R);
    }
};

/* ------------------------------------------------------------------------- */
/* OrientationUKF (OrientationUKF.hpp:20-59, OrientationUKF.cpp).              */
/* ------------------------------------------------------------------------- */
template <class T>
class OrientationFilter : public FilterShell<T, OrientationState<T>> {
    typedef FilterShell<T, OrientationState<T>> Base;
    typedef OrientationState<T> S;
    enum { n = S::DOF };

public:
    double rotation_rate_mu[3];
    double acceleration_mu[3];
    double earth_rotation[3];
    double gyro_bias_tau, acc_bias_tau;

    /* OrientationUKF.cpp:41-51 */
    OrientationFilter(const S& initial_state, const T* state_cov, double gyro_bias_tau_, double acc_bias_tau_,
                      double latitude)
        : gyro_bias_tau(gyro_bias_tau_), acc_bias_tau(acc_bias_tau_)
    {
        this->initializeFilter(initial_state, state_cov);
        earth_rotation[0] = UKFB_EARTHW * std::cos(latitude);
        earth_rotation[1] = 0.;
        earth_rotation[2] = UKFB_EARTHW * std::sin(latitude);
        for (int i = 0; i < 3; ++i) rotation_rate_mu[i] = 0.;
        acceleration_mu[0] = 0., acceleration_mu[1] = 0.;
        acceleration_mu[2] = double(initial_state.gravity[0]);
    }

    /* :53-57 */
    void setRotationRate(const double* mu, const double* cov)
    {
        Base::template checkMeasurment<3>(mu, cov);
        for (int i = 0; i < 3; ++i) rotation_rate_mu[i] = mu[i];
    }
    /* :59-63 */
    void setAcceleration(const double* mu, const double* cov)
    {
        Base::template checkMeasurment<3>(mu, cov);
        for (int i = 0; i < 3; ++i) acceleration_mu[i] = mu[i];
    }
    /* :65-72, measurement model :34-39  h = q^-1 * v */
    void integrateVelocity(const double* zmu, const double* zcov)
    {
        Base::template checkMeasurment<3>(zmu, zcov);
        EuclidMeas<T, 3> z;
        T R[9];
        for (int i = 0; i < 3; ++i) z.a[i] = T(zmu[i]);
        for (int i = 0; i < 9; ++i) R[i] = T(zcov[i]);
        this->ukf.update(z,
                         [](const S& s) {
                             EuclidMeas<T, 3> r;
                             quat_rotate(quat_inverse(s.orientation), s.velocity, r.a);
                             return r;
                         },
                         R);
    }
    /* :74-77 */
    void getRotationRate(double out[3]) const
    {
        T er[3] = {T(earth_rotation[0]), T(earth_rotation[1]), T(earth_rotation[2])};
        T r[3];
        quat_rotate(quat_inverse(this->ukf.mu.orientation), er, r);
        for (int i = 0; i < 3; ++i) out[i] = double(T(rotation_rate_mu[i]) - this->ukf.mu.bias_gyro[i] - r[i]);
    }

    /* :12-32 -- the acceleration is rotated with the UPDATED orientation. */
    static S processModel(const S& state, const T acc[3], const T omega[3], const T& gyro_bias_tau,
                          const T& acc_bias_tau, const T earth_rotation[3], const T& dt)
    {
        S ns(state);
        T w[3], av[3];
        for (int i = 0; i < 3; ++i) w[i] = omega[i] - ns.bias_gyro[i];
        quat_rotate(ns.orientation, w, av);
        for (int i = 0; i < 3; ++i) av[i] = av[i] - earth_rotation[i];
        so3_boxplus(ns.orientation, av, dt);

        T a[3], an[3];
        for (int i = 0; i < 3; ++i) a[i] = acc[i] - ns.bias_acc[i];
        quat_rotate(ns.orientation, a, an);
        an[0] = an[0] - T(0.);
        an[1] = an[1] - T(0.);
        an[2] = an[2] - ns.gravity[0];
        for (int i = 0; i < 3; ++i) ns.velocity[i] = ns.velocity[i] + dt * an[i];

        const T kg = T(-1.0) / gyro_bias_tau;
        for (int i = 0; i < 3; ++i) {
            const T d = kg * ns.bias_gyro[i];
            ns.bias_gyro[i] = ns.bias_gyro[i] + dt * d;
        }
        const T ka = T(-1.0) / acc_bias_tau;
        for (int i = 0; i < 3; ++i) {
            const T d = ka * ns.bias_acc[i];
            ns.bias_acc[i] = ns.bias_acc[i] + dt * d;
        }
        return ns;
    }

protected:
    /* :79-89 -- Q scaled by delta^2 (PoseUKF scales by delta). */
    void predictionStepImpl(double delta) override
    {
        T rot[9];
        quat_matrix(this->ukf.mu.orientation, rot);
        T process_noise[n * n];
        for (int i = 0; i < n * n; ++i) process_noise[i] = this->process_noise_cov[i];
        Base::rotate_block(process_noise, this->process_noise_cov, rot, 0);
        Base::rotate_block(process_noise, this->process_noise_cov, rot, 3);
        /* a scalar wider than double squares the exact delta; double keeps the reference's std::pow */
        T d2;
        if constexpr (kWiderThanDouble<T>)
            d2 = T(delta) * T(delta);
        else
            d2 = T(std::pow(delta, 2.));
        for (int i = 0; i < n * n; ++i) process_noise[i] = d2 * process_noise[i];

        const T a[3] = {T(acceleration_mu[0]), T(acceleration_mu[1]), T(acceleration_mu[2])};
        const T w[3] = {T(rotation_rate_mu[0]), T(rotation_rate_mu[1]), T(rotation_rate_mu[2])};
        const T er[3] = {T(earth_rotation[0]), T(earth_rotation[1]), T(earth_rotation[2])};
        const T tg = T(gyro_bias_tau), ta = T(acc_bias_tau), dt = T(delta);
        this->ukf.predict([&](const S& s) { return processModel(s, a, w, tg, ta, er, dt); }, process_noise);
    }
};

} /* namespace orc */

#endif /* UKF_ORACLE_HPP */
