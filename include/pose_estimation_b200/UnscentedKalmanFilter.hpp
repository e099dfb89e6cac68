/*
 * UnscentedKalmanFilter.hpp -- host-side mirror of pose_estimation::UnscentedKalmanFilter<Manifold>
 * (reference src/UnscentedKalmanFilter.hpp:15-155) on top of the C ABI in include/ukf_batch.h.
 *
 * Same member names, argument meaning and error behaviour as the reference class, minus its Eigen / MTK /
 * base-types dependencies (absent from this image): states and covariances are plain arrays, base::Time is an
 * int64 microsecond count.  One object drives `batch` independent filters (batch = 1 gives exactly the
 * reference's single-filter object), on one GPU or -- constructed with a device list -- split by filter index over
 * several GPUs of the box; every method applies to all of them.  The arithmetic runs in the CUDA
 * engine -- there is no host implementation behind this class.
 *
 * Error behaviour: the reference throws std::runtime_error from predictionStep / checkMeasurment.  The engine
 * records the same conditions as per-filter status bits; after each call this class turns new bits into the
 * same exception (same message) -- for batch > 1 the exception reports the first offending filter and the
 * other filters have been stepped normally, which is what a loop over reference objects with a try/catch per
 * object would have done.
 */
#ifndef POSE_ESTIMATION_B200_UKF_HPP
#define POSE_ESTIMATION_B200_UKF_HPP

#include <cstdint>
#include <limits>
#include <stdexcept>
#include <string>
#include <vector>

#include "../ukf_batch.h"

namespace pose_estimation_b200
{

template <int FILTER_KIND, int DOF_, int MU_>
class UnscentedKalmanFilter
{
public:
    enum { DOF = DOF_, MU = MU_ };
    /* State: MU doubles per filter (quaternion stored x, y, z, w like Eigen); Covariance: DOF x DOF row-major */
    struct State { double v[MU_]; };
    struct Covariance { double v[DOF_ * DOF_]; };

    explicit UnscentedKalmanFilter(int64_t batch = 1, int device = 0) : h(nullptr), batch_size(batch)
    {
        check(ukfb_create(FILTER_KIND, batch, device, &h));
    }
    /* the same `batch` filters split by filter index over several GPUs of the box behind one object (ukfb_create_sharded:
     * contiguous shards, one host worker and one set of streams per device, no inter-device traffic); every method below
     * then serves all devices at once and getCurrentState gathers all shards into the caller's arrays */
    UnscentedKalmanFilter(int64_t batch, const std::vector<int>& devices) : h(nullptr), batch_size(batch)
    {
        check(ukfb_create_sharded(FILTER_KIND, batch, devices.data(), int(devices.size()), &h));
    }
    virtual ~UnscentedKalmanFilter() { ukfb_destroy(h); }
    UnscentedKalmanFilter(const UnscentedKalmanFilter&) = delete; /* boost::noncopyable, :16 */
    UnscentedKalmanFilter& operator=(const UnscentedKalmanFilter&) = delete;

    int64_t batch() const { return batch_size; }
    ukfb_handle* handle() { return h; }

    /* (Re-)initializes the filters from given states (:40-44).  Arrays of `batch` entries. */
    void initializeFilter(const State* initial_state, const Covariance* state_cov)
    {
        check(ukfb_initialize(h, initial_state->v, state_cov->v));
    }
    /* the reference's signature: one filter.  On an object built with batch > 1 the C ABI would read `batch` states
     * behind the single struct, so that is refused rather than left to overrun. */
    void initializeFilter(const State& initial_state, const Covariance& state_cov)
    {
        single("initializeFilter(const State&, const Covariance&)");
        initializeFilter(&initial_state, &state_cov);
    }

    /* @returns false if the filter has not been initialized (:51-75) */
    bool getCurrentState(State* state, Covariance* state_cov) const
    {
        const int rc = ukfb_get_state(h, state->v, state_cov ? state_cov->v : nullptr);
        if (rc == UKFB_ERR_NOT_INITIALIZED) return false;
        check(rc);
        return true;
    }
    bool getCurrentState(State& state, Covariance& state_cov) const
    {
        single("getCurrentState(State&, Covariance&)");
        return getCurrentState(&state, &state_cov);
    }
    bool getCurrentState(State& state) const
    {
        single("getCurrentState(State&)");
        return getCurrentState(&state, nullptr);
    }

    /* The reference's single-filter calls for filter `index` of this object (a global index, also across devices): what a
     * caller owning N reference objects does to the one it needs, here without touching the others.  initializeFilter
     * resets that filter's time latch (:43) and leaves its status word alone. */
    void initializeFilter(int64_t index, const State& initial_state, const Covariance& state_cov)
    {
        check(ukfb_initialize_indexed(h, 1, &index, initial_state.v, state_cov.v));
    }
    bool getCurrentState(int64_t index, State& state, Covariance& state_cov) const
    {
        return getCurrentStates(1, &index, &state, &state_cov);
    }
    bool getCurrentState(int64_t index, State& state) const { return getCurrentStates(1, &index, &state, nullptr); }
    /* the same for n filters idx[0..n) at once: entry k of the arrays belongs to filter idx[k] (unique for initialize) */
    void initializeFilters(int64_t n, const int64_t* idx, const State* initial_states, const Covariance* state_covs)
    {
        check(ukfb_initialize_indexed(h, n, idx, n ? initial_states->v : nullptr, n ? state_covs->v : nullptr));
    }
    bool getCurrentStates(int64_t n, const int64_t* idx, State* states, Covariance* state_covs) const
    {
        const int rc = ukfb_get_state_indexed(h, n, idx, n ? states->v : nullptr, n && state_covs ? state_covs->v : nullptr);
        if (rc == UKFB_ERR_NOT_INITIALIZED) return false;
        check(rc);
        return true;
    }
    /* the filters whose condition the last exception reported (ascending), for getting them back with
     * initializeFilter(index, ...); empty after a call that threw nothing */
    const std::vector<int64_t>& lastFailedFilters() const { return failed; }

    /* :83-100; sample_time in microseconds (base::Time::microseconds) */
    void predictionStepFromSampleTime(int64_t sample_time_us)
    {
        check(ukfb_predict_time(h, &sample_time_us, 0));
        raise();
    }
    void predictionStepFromSampleTime(const int64_t* sample_time_us) /* one per filter */
    {
        check(ukfb_predict_time(h, sample_time_us, 1));
        raise();
    }

    /* :107-125 */
    void predictionStep(double delta_t)
    {
        check(ukfb_predict_dt(h, &delta_t, 0));
        raise();
    }
    void predictionStep(const double* delta_t) /* one per filter */
    {
        check(ukfb_predict_dt(h, delta_t, 1));
        raise();
    }

    unsigned getStateSize() const { return unsigned(DOF_); }                 /* :127 */
    bool isInitialized() const { return ukfb_is_initialized(h) != 0; }       /* :128 */
    Covariance getProcessNoiseCovariance() const                             /* :129, the first filter's */
    {
        std::vector<Covariance> q(static_cast<size_t>(batch_size));
        check(ukfb_get_process_noise(h, q[0].v, 1));
        return q[0];
    }
    void setProcessNoiseCovariance(const Covariance& noise_cov) { check(ukfb_set_process_noise(h, noise_cov.v, 0)); } /* :130 */
    void setProcessNoiseCovariance(const Covariance* noise_cov) { check(ukfb_set_process_noise(h, noise_cov->v, 1)); }
    int64_t getLastMeasurementTime() const                                   /* :131, the first filter's */
    {
        std::vector<int64_t> t(static_cast<size_t>(batch_size));
        check(ukfb_get_last_time(h, t.data()));
        return t[0];
    }
    void setLastMeasurementTime(int64_t t_us) { check(ukfb_set_last_time(h, &t_us, 0)); } /* :132-133 */
    double getMaxTimeDelta() const { double a, b; check(ukfb_get_time_bounds(h, &a, &b)); return b; }
    void setMaxTimeDelta(double max_time_delta) { check(ukfb_set_time_bounds(h, getMinTimeDelta(), max_time_delta)); }
    double getMinTimeDelta() const { double a, b; check(ukfb_get_time_bounds(h, &a, &b)); return a; }
    void setMinTimeDelta(double min_time_delta) { check(ukfb_set_time_bounds(h, min_time_delta, getMaxTimeDelta())); }

protected:
    /* the by-reference overloads carry ONE state: batch objects must use the pointer (array) overloads */
    void single(const char* what) const
    {
        if (batch_size != 1)
            throw std::logic_error(std::string("ukf_batch: ") + what + " serves a single filter; this object holds " +
                                   std::to_string(batch_size) + " -- pass arrays of `batch` entries to the pointer overload");
    }

    /* a failed C ABI call is API misuse or a CUDA failure, never a filter condition */
    static void check(int rc)
    {
        if (rc != UKFB_OK) throw std::logic_error(std::string("ukf_batch: ") + ukfb_last_error());
    }

    /* status bits -> the reference's exceptions; bits are cleared so that the next call starts clean */
    void raise()
    {
        int64_t n = 0;
        uint32_t bits = 0;
        failed.clear();
        check(ukfb_status_summary(h, &n, &bits));
        if (!bits) return;
        const uint32_t thrown = UKFB_STATUS_NEG_DT | UKFB_STATUS_DT_TOO_LARGE | UKFB_STATUS_NONFINITE_MEAS | UKFB_STATUS_NOT_SPD |
                                UKFB_STATUS_MEAN_NO_CONVERGE;
        if (bits & thrown) { /* which filters: before the status words are cleared */
            int64_t count = 0;
            check(ukfb_find_status(h, thrown, 0, nullptr, &count));
            failed.resize(size_t(count));
            check(ukfb_find_status(h, thrown, count, failed.data(), &count));
        }
        check(ukfb_clear_status(h));
        if (bits & UKFB_STATUS_NEG_DT) throw std::runtime_error("Delta time is negative!");                               /* :112 */
        if (bits & UKFB_STATUS_DT_TOO_LARGE) throw std::runtime_error("Delta time is greater then the allowed maximum!"); /* :121 */
        if (bits & UKFB_STATUS_NONFINITE_MEAS) throw std::runtime_error("Measurement or covariance contains non-finite values!"); /* :146 */
        if (bits & UKFB_STATUS_NOT_SPD) throw std::runtime_error("ukfom: covariance is not positive definite");           /* MTK assert */
        if (bits & UKFB_STATUS_MEAN_NO_CONVERGE) throw std::runtime_error("ukfom: sigma point mean did not converge");     /* MTK assert */
    }

    /* per_filter = false: `measurement` is one struct applied to every filter of the batch;
     * per_filter = true: an array of `batch` structs (mu and cov per filter).  Repacked to the ABI's separate
     * mu / cov arrays. */
    template <class M>
    void update(int meas_kind, const M* measurement, bool per_filter)
    {
        const int m = M::Dim;
        std::vector<double> mu(size_t(batch_size) * m), cov(size_t(per_filter ? batch_size : 1) * m * m);
        for (int64_t b = 0; b < batch_size; ++b)
            for (int i = 0; i < m; ++i) mu[size_t(b) * m + i] = measurement[per_filter ? b : 0].mu[i];
        for (int64_t b = 0; b < (per_filter ? batch_size : 1); ++b)
            for (int i = 0; i < m * m; ++i) cov[size_t(b) * m * m + i] = measurement[b].cov[i];
        check(ukfb_update(h, meas_kind, mu.data(), cov.data(), per_filter ? 1 : 0, nullptr));
        raise();
    }

    ukfb_handle* h;
    int64_t batch_size;
    std::vector<int64_t> failed; /* lastFailedFilters() */
};

}  // namespace pose_estimation_b200

#endif
