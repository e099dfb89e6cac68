/*
 * oracle/oracle_capi.cpp -- CPU ORACLE, batch C interface.  TEST INFRASTRUCTURE ONLY
 * (see the header of ukf_oracle.hpp: parity unpinned; only tests/, smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this library).
 *
 * B independent oracle filter objects behind the same call shapes as
 * include/ukf_batch.h (prefix orc_ instead of ukfb_), so that a parity test can
 * drive the CUDA engine and the oracle with identical arguments.  OpenMP
 * `parallel for` over filters: this is also the CPU baseline that bench.py times.
 */
#include <omp.h>

#include <cstdint>
#include <cstring>
#include <memory>
#include <vector>

#include "ukf_oracle.hpp"

using namespace orc;

/* The filter objects behind the batch.  Default: the oracle's own restatement of the reference classes.  oracle/ref_capi.cpp
 * defines ORC_CUSTOM_IMPL, adapters over the REFERENCE'S OWN classes (compiled unmodified from /root/reference against
 * oracle/ref_shim) with the same member functions, and includes this file: the same batch interface then drives them. */
/* ORC_REAL: the filters' scalar.  `double` is the oracle proper; liboracle_ld.so builds with `long double` as an
 * extended-precision reference for the FP64 implementations.  The C interface stays `double` either way: inputs
 * widen exactly and results are rounded once on read-back. */
#ifndef ORC_REAL
#define ORC_REAL double
#endif

#ifndef ORC_CUSTOM_IMPL
typedef PoseFilter<ORC_REAL> PoseImpl;
typedef OrientationFilter<ORC_REAL> OriImpl;
namespace ax { /* access to what the reference keeps in protected members / inside ukfom::ukf */
template <class F> void store_mu(const F& f, double* mu) { f.ukf.mu.store(mu); }
template <class F> void copy_sigma(const F& f, double* sigma)
{
    const int nn = sizeof(f.ukf.sigma) / sizeof(f.ukf.sigma[0]);
    for (int k = 0; k < nn; ++k) sigma[k] = double(f.ukf.sigma[k]);
}
template <class F> void set_q(F& f, int k, double v) { f.process_noise_cov[k] = v; }
template <class F> void set_dt_bounds(F& f, double lo, double hi) { f.min_time_delta = lo, f.max_time_delta = hi; }
template <class F> void set_gate(F& f, double d2) { f.ukf.accept_max_d2 = d2; }
template <class F> bool rejected(const F& f) { return f.ukf.last_update_rejected; }
template <class F> void set_last_time(F& f, int64_t t) { f.last_measurement_time_us = t; }
template <class F> int64_t last_time(const F& f) { return f.last_measurement_time_us; }
template <class F> uint32_t status(const F& f) { return f.ukf.status; }
template <class F> void clear_status(F& f) { f.ukf.status = 0; }
template <class F> uint64_t mean_iters(const F& f, int k) { return f.ukf.mean_iters[k]; }
inline void set_ori_params(OriImpl& f, double tau_g, double tau_a, double latitude)
{
    f.gyro_bias_tau = tau_g;
    f.acc_bias_tau = tau_a;
    f.earth_rotation[0] = UKFB_EARTHW * std::cos(latitude);
    f.earth_rotation[1] = 0.;
    f.earth_rotation[2] = UKFB_EARTHW * std::sin(latitude);
}
} /* namespace ax */
#endif

namespace {

struct Batch {
    int kind;
    int64_t B;
    int n, MU;
    bool initialized = false;
    bool constructed = false; /* filter objects exist */
    std::vector<std::unique_ptr<PoseImpl>> pose;
    std::vector<std::unique_ptr<OriImpl>> ori;
    std::vector<uint32_t> status;
    /* parameters applied at construction / kept across re-initialisation */
    std::vector<double> Q; /* n*n or B*n*n */
    bool q_per_filter = false;
    bool q_set = false;
    double min_dt = UKFB_DEFAULT_MIN_DT;
    double max_dt = std::numeric_limits<double>::max();
    double tau_g = std::numeric_limits<double>::infinity();
    double tau_a = std::numeric_limits<double>::infinity();
    double latitude = 0.0;
};

template <class F>
void apply_common(Batch* b, F& f, int64_t i)
{
    const int nn = b->n * b->n;
    if (b->q_set) {
        const double* q = b->Q.data() + (b->q_per_filter ? i * nn : 0);
        for (int k = 0; k < nn; ++k) ax::set_q(f, k, q[k]);
    }
    ax::set_dt_bounds(f, b->min_dt, b->max_dt);
}

template <class Fn>
void guarded(Batch* b, int64_t i, Fn fn)
{
    try {
        fn();
    } catch (const std::runtime_error& e) {
        const char* w = e.what();
        if (std::strstr(w, "negative"))
            b->status[i] |= ST_NEG_DT;
        else if (std::strstr(w, "allowed maximum"))
            b->status[i] |= ST_DT_TOO_LARGE;
        else
            b->status[i] |= ST_NONFINITE_MEAS;
    }
}

} /* namespace */

extern "C" {

void* orc_create(int kind, int64_t B)
{
    if ((kind != 0 && kind != 1) || B <= 0) return nullptr;
    Batch* b = new Batch();
    b->kind = kind;
    b->B = B;
    b->n = kind == 0 ? UKFB_POSE_DOF : UKFB_ORI_DOF;
    b->MU = kind == 0 ? UKFB_POSE_MU : UKFB_ORI_MU;
    b->status.assign(B, 0u);
    return b;
}

void orc_destroy(void* h) { delete static_cast<Batch*>(h); }

void orc_set_threads(int t)
{
    if (t > 0) omp_set_num_threads(t);
}
int orc_max_threads(void) { return omp_get_max_threads(); }

int orc_initialize(void* h, const double* mu, const double* sigma)
{
    Batch* b = static_cast<Batch*>(h);
    const int nn = b->n * b->n;
    if (!b->constructed) {
        if (b->kind == 0)
            b->pose.resize(b->B);
        else
            b->ori.resize(b->B);
    }
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        ORC_REAL sg[UKFB_ORI_DOF * UKFB_ORI_DOF]; /* the larger of the two kinds */
        for (int k = 0; k < nn; ++k) sg[k] = sigma[i * nn + k];
        if (b->kind == 0) {
            PoseState<ORC_REAL> s;
            s.load(mu + i * b->MU);
            if (!b->constructed) {
                b->pose[i].reset(new PoseImpl(s, sg));
                apply_common(b, *b->pose[i], i);
            } else
                b->pose[i]->initializeFilter(s, sg);
        } else {
            OrientationState<ORC_REAL> s;
            s.load(mu + i * b->MU);
            if (!b->constructed) {
                b->ori[i].reset(new OriImpl(s, sg, b->tau_g, b->tau_a, b->latitude));
                apply_common(b, *b->ori[i], i);
            } else
                b->ori[i]->initializeFilter(s, sg);
        }
    }
    b->constructed = true;
    b->initialized = true;
    return 0;
}

int orc_get_state(void* h, double* mu, double* sigma)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
    const int nn = b->n * b->n;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        if (b->kind == 0) {
            ax::store_mu(*b->pose[i], mu + i * b->MU);
            if (sigma) ax::copy_sigma(*b->pose[i], sigma + i * nn);
        } else {
            ax::store_mu(*b->ori[i], mu + i * b->MU);
            if (sigma) ax::copy_sigma(*b->ori[i], sigma + i * nn);
        }
    }
    return 0;
}

int orc_set_process_noise(void* h, const double* Q, int per_filter)
{
    Batch* b = static_cast<Batch*>(h);
    const int nn = b->n * b->n;
    b->Q.assign(Q, Q + (per_filter ? b->B * nn : nn));
    b->q_per_filter = per_filter != 0;
    b->q_set = true;
    if (b->constructed) {
        for (int64_t i = 0; i < b->B; ++i) {
            if (b->kind == 0)
                apply_common(b, *b->pose[i], i);
            else
                apply_common(b, *b->ori[i], i);
        }
    }
    return 0;
}

int orc_set_time_bounds(void* h, double min_dt, double max_dt)
{
    Batch* b = static_cast<Batch*>(h);
    b->min_dt = min_dt;
    b->max_dt = max_dt;
    if (b->constructed)
        for (int64_t i = 0; i < b->B; ++i) {
            if (b->kind == 0)
                ax::set_dt_bounds(*b->pose[i], min_dt, max_dt);
            else
                ax::set_dt_bounds(*b->ori[i], min_dt, max_dt);
        }
    return 0;
}

/* the accept functor slot of ukfom::ukf::update (PoseUKF.cpp:116 passes accept_any = +inf) */
int orc_set_mahalanobis_gate(void* h, double max_d2)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->constructed) return -2;
    for (int64_t i = 0; i < b->B; ++i) {
        if (b->kind == 0)
            ax::set_gate(*b->pose[i], max_d2);
        else
            ax::set_gate(*b->ori[i], max_d2);
    }
    return 0;
}

int orc_set_orientation_params(void* h, double tau_g, double tau_a, double latitude)
{
    Batch* b = static_cast<Batch*>(h);
    if (b->kind != 1) return -1;
    b->tau_g = tau_g, b->tau_a = tau_a, b->latitude = latitude;
    if (b->constructed)
        for (int64_t i = 0; i < b->B; ++i) ax::set_ori_params(*b->ori[i], tau_g, tau_a, latitude);
    return 0;
}

int orc_set_orientation_params_per_filter(void* h, const double* tau_g, const double* tau_a, const double* latitude)
{
    Batch* b = static_cast<Batch*>(h);
    if (b->kind != 1) return -1;
    if (!b->constructed) return -2; /* the oracle's objects exist after the first initialize */
    for (int64_t i = 0; i < b->B; ++i) ax::set_ori_params(*b->ori[i], tau_g[i], tau_a[i], latitude[i]);
    return 0;
}

int orc_set_last_time(void* h, const int64_t* ts, int per_filter)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->constructed) return -2;
    for (int64_t i = 0; i < b->B; ++i) {
        const int64_t t = ts[per_filter ? i : 0];
        if (b->kind == 0)
            ax::set_last_time(*b->pose[i], t);
        else
            ax::set_last_time(*b->ori[i], t);
    }
    return 0;
}

int orc_get_last_time(void* h, int64_t* ts)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->constructed) return -2;
    for (int64_t i = 0; i < b->B; ++i)
        ts[i] = b->kind == 0 ? ax::last_time(*b->pose[i]) : ax::last_time(*b->ori[i]);
    return 0;
}

int orc_predict_dt(void* h, const double* dt, int per_filter)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        const double d = dt[per_filter ? i : 0];
        guarded(b, i, [&] {
            if (b->kind == 0)
                b->pose[i]->predictionStep(d);
            else
                b->ori[i]->predictionStep(d);
        });
    }
    return 0;
}

int orc_predict_time(void* h, const int64_t* ts, int per_filter)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        const int64_t t = ts[per_filter ? i : 0];
        guarded(b, i, [&] {
            if (b->kind == 0)
                b->pose[i]->predictionStepFromSampleTime(t);
            else
                b->ori[i]->predictionStepFromSampleTime(t);
        });
    }
    return 0;
}

int orc_meas_dim(int kind) { return meas_dim(kind); }

int orc_update(void* h, int meas_kind, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
    if (b->kind == 0 && (meas_kind < 0 || meas_kind > MEAS_POSE_ANGULAR_VELOCITY)) return -1;
    if (b->kind == 1 && meas_kind != MEAS_ORI_VELOCITY) return -1;
    const int m = meas_dim(meas_kind);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        if (mask && !mask[i]) continue;
        const double* zm = mu + i * m;
        const double* zc = cov + (cov_per_filter ? i * m * m : 0);
        guarded(b, i, [&] {
            if (b->kind == 0)
                { b->pose[i]->integrateMeasurement(meas_kind, zm, zc); if (ax::rejected(*b->pose[i])) b->status[i] |= 64u; }
            else
                { b->ori[i]->integrateVelocity(zm, zc); if (ax::rejected(*b->ori[i])) b->status[i] |= 64u; }
        });
    }
    return 0;
}

int orc_update_mixed(void* h, const int8_t* kinds, const double* mu3, const double* cov33)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        const int k = kinds[i];
        if (k < 0) continue;
        const int m = meas_dim(k);
        double zm[3], zc[9];
        for (int a = 0; a < m; ++a) zm[a] = mu3[i * 3 + a];
        for (int a = 0; a < m; ++a)
            for (int c = 0; c < m; ++c) zc[a * m + c] = cov33[i * 9 + a * 3 + c];
        guarded(b, i, [&] {
            if (b->kind == 0)
                { b->pose[i]->integrateMeasurement(k, zm, zc); if (ax::rejected(*b->pose[i])) b->status[i] |= 64u; }
            else
                { b->ori[i]->integrateVelocity(zm, zc); if (ax::rejected(*b->ori[i])) b->status[i] |= 64u; }
        });
    }
    return 0;
}

static const double kIdentity3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};

int orc_set_acceleration(void* h, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->constructed) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        if (mask && !mask[i]) continue;
        const double* c = cov ? cov + (cov_per_filter ? i * 9 : 0) : kIdentity3;
        guarded(b, i, [&] {
            if (b->kind == 0)
                b->pose[i]->setAcceleration(mu + i * 3, c);
            else
                b->ori[i]->setAcceleration(mu + i * 3, c);
        });
    }
    return 0;
}

int orc_set_rotation_rate(void* h, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    Batch* b = static_cast<Batch*>(h);
    if (b->kind != 1) return -1;
    if (!b->constructed) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        if (mask && !mask[i]) continue;
        const double* c = cov ? cov + (cov_per_filter ? i * 9 : 0) : kIdentity3;
        guarded(b, i, [&] { b->ori[i]->setRotationRate(mu + i * 3, c); });
    }
    return 0;
}

/* The reference's caller loop (one aggregator callback per sensor sample, in timestamp order):
 *     filter.predictionStepFromSampleTime(ts);  filter.integrateMeasurement(sample);
 * (UnscentedKalmanFilter.hpp:83-100, PoseUKF.cpp:112-178, OrientationUKF.cpp:53-72) run over the K queued samples of
 * every filter; same array shapes as ukfb_run_events. */
int orc_run_events(void* h, int K, const int64_t* ts, const int8_t* kinds, const double* mu3, const double* cov, int cov_mode)
{
    Batch* b = static_cast<Batch*>(h);
    if (!b->initialized) return -2;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < b->B; ++i) {
        for (int k = 0; k < K; ++k) {
            const int64_t e = int64_t(k) * b->B + i;
            const int kind = kinds[e];
            if (kind == -2) continue; /* idle slot */
            const bool pose = b->kind == 0;
            const bool known = kind >= -1 && kind <= 12 && (pose ? (kind != MEAS_ORI_VELOCITY && kind <= 10) : (kind == -1 || kind == MEAS_ORI_VELOCITY || kind >= 11));
            if (!known) {
                b->status[i] |= 32u;
                continue;
            }
            /* ONE guarded block per callback: a throw from predictionStep (negative / too large delta,
             * UnscentedKalmanFilter.hpp:110-122) leaves the callback, so that sample's integrateMeasurement never runs */
            guarded(b, i, [&] {
                if (pose)
                    b->pose[i]->predictionStepFromSampleTime(ts[e]);
                else
                    b->ori[i]->predictionStepFromSampleTime(ts[e]);
                if (kind < 0) return;
                const double* c33 = cov + (cov_mode ? e * 9 : int64_t(kind) * 9);
                const double* z = mu3 + e * 3;
                if (kind >= 10) {
                    if (pose)
                        b->pose[i]->setAcceleration(z, c33);
                    else if (kind == 11)
                        b->ori[i]->setRotationRate(z, c33);
                    else
                        b->ori[i]->setAcceleration(z, c33);
                    return;
                }
                const int m = meas_dim(kind);
                double zc[9];
                for (int a = 0; a < m; ++a)
                    for (int c = 0; c < m; ++c) zc[a * m + c] = c33[a * 3 + c];
                if (pose) {
                    b->pose[i]->integrateMeasurement(kind, z, zc);
                    if (ax::rejected(*b->pose[i])) b->status[i] |= 64u;
                } else {
                    b->ori[i]->integrateVelocity(z, zc);
                    if (ax::rejected(*b->ori[i])) b->status[i] |= 64u;
                }
            });
        }
    }
    return 0;
}

/* BodyStateMeasurement::fromRigidBodyState (BodyStateMeasurement.hpp:14-26): rbs B x 49 -> mu B x 13, sigma B x 12 x 12 */
void orc_from_body_states(const double* rbs, int64_t B, double* mu, double* sigma)
{
    for (int64_t i = 0; i < B; ++i) {
        const double* r = rbs + i * 49;
        for (int k = 0; k < 13; ++k) mu[i * 13 + k] = r[k]; /* position, orientation, velocity, angular_velocity */
        double* s = sigma + i * 144;
        for (int k = 0; k < 144; ++k) s[k] = 0.0; /* setZero() */
        for (int blk = 0; blk < 4; ++blk)
            for (int a = 0; a < 3; ++a)
                for (int c = 0; c < 3; ++c) s[(blk * 3 + a) * 12 + blk * 3 + c] = r[13 + blk * 9 + a * 3 + c];
    }
}

/* BodyStateMeasurement::toRigidBodyState (BodyStateMeasurement.hpp:28-39) */
void orc_to_body_states(const double* mu, const double* sigma, int64_t B, double* rbs)
{
    for (int64_t i = 0; i < B; ++i) {
        double* r = rbs + i * 49;
        const double* m = mu + i * 13;
        for (int k = 0; k < 13; ++k) r[k] = m[k];
        const Quat<double> q = {m[3], m[4], m[5], m[6]};
        quat_rotate(q, m + 7, r + 7); /* body_state.velocity = body_state.orientation * filter_state.velocity */
        const double* s = sigma + i * 144;
        for (int blk = 0; blk < 4; ++blk)
            for (int a = 0; a < 3; ++a)
                for (int c = 0; c < 3; ++c) r[13 + blk * 9 + a * 3 + c] = s[(blk * 3 + a) * 12 + blk * 3 + c];
    }
}

int orc_get_rotation_rate(void* h, double* out)
{
    Batch* b = static_cast<Batch*>(h);
    if (b->kind != 1) return -1;
    if (!b->initialized) return -2;
    for (int64_t i = 0; i < b->B; ++i) b->ori[i]->getRotationRate(out + i * 3);
    return 0;
}

int orc_step(void* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu, const double* cov,
             int cov_per_filter, const uint8_t* mask)
{
    int rc = orc_predict_dt(h, dt, dt_per_filter);
    if (rc) return rc;
    if (meas_kind < 0) return 0;
    return orc_update(h, meas_kind, mu, cov, cov_per_filter, mask);
}

int orc_get_status(void* h, uint32_t* flags)
{
    Batch* b = static_cast<Batch*>(h);
    for (int64_t i = 0; i < b->B; ++i) {
        uint32_t s = b->status[i];
        if (b->constructed) s |= b->kind == 0 ? ax::status(*b->pose[i]) : ax::status(*b->ori[i]);
        flags[i] = s;
    }
    return 0;
}

int orc_clear_status(void* h)
{
    Batch* b = static_cast<Batch*>(h);
    for (int64_t i = 0; i < b->B; ++i) {
        b->status[i] = 0;
        if (b->constructed) {
            if (b->kind == 0)
                ax::clear_status(*b->pose[i]);
            else
                ax::clear_status(*b->ori[i]);
        }
    }
    return 0;
}

int orc_get_mean_iter_hist(void* h, uint64_t hist[8])
{
    Batch* b = static_cast<Batch*>(h);
    for (int k = 0; k < 8; ++k) hist[k] = 0;
    if (!b->constructed) return 0;
    for (int64_t i = 0; i < b->B; ++i)
        for (int k = 0; k < 8; ++k)
            hist[k] += b->kind == 0 ? ax::mean_iters(*b->pose[i], k) : ax::mean_iters(*b->ori[i], k);
    return 0;
}

} /* extern "C" */
