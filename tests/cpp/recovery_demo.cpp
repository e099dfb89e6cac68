// recovery_demo.cpp -- a batch PoseUKF object from C++ host code, as a caller of the reference classes recovers ONE of
// its filter objects: some filters are given a covariance that is not positive definite, the next prediction throws the
// same std::runtime_error as today, lastFailedFilters() names the filters behind it, initializeFilter(index, ...)
// re-initialises just those, and the batch carries on.  tests/test_indexed.py replays the calls on the oracle.
// usage: recovery_demo <batch>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <vector>

#include <pose_estimation_b200/PoseUKF.hpp>

using namespace pose_estimation_b200;

// deterministic per-filter values: tests/test_indexed.py restates this function
static double wobble(int64_t b, int k, int c) { return std::sin(0.37 * double(b) + 1.3 * double(k) + 0.71 * double(c)); }

static bool failing(int64_t b) { return b % 13 == 5; }  // the filters given a bad covariance

int main(int argc, char** argv)
{
    if (argc < 2) {
        fprintf(stderr, "usage: %s <batch>\n", argv[0]);
        return 64;
    }
    const int64_t B = atoll(argv[1]);
    const size_t n = size_t(B);
    std::vector<PoseUKF::State> x0(n);
    std::vector<PoseUKF::Covariance> p0(n);
    const double d0[12] = {1, 1, 1, 0.01, 0.01, 0.01, 0.1, 0.1, 0.1, 0.01, 0.01, 0.01};
    for (int64_t b = 0; b < B; ++b) {
        PoseUKF::State& x = x0[size_t(b)];
        memset(&x, 0, sizeof(x));
        memset(&p0[size_t(b)], 0, sizeof(PoseUKF::Covariance));
        const double yaw = 0.3 * wobble(b, 20, 0);
        x.v[0] = wobble(b, 21, 0), x.v[1] = wobble(b, 21, 1);
        x.v[5] = std::sin(0.5 * yaw), x.v[6] = std::cos(0.5 * yaw);
        x.v[7] = 1.0 + 0.1 * wobble(b, 22, 0);
        x.v[12] = 0.05;
        for (int i = 0; i < 12; ++i) p0[size_t(b)].v[i * 12 + i] = d0[i] * (1.0 + 0.2 * wobble(b, 23, i));
    }
    try {
        PoseUKF f(B, x0.data(), p0.data());
        for (int64_t b = 0; b < B; ++b)
            if (failing(b)) {
                PoseUKF::Covariance bad = p0[size_t(b)];
                bad.v[0] = -1.0;  // not positive definite: the next prediction's factorisation fails
                f.initializeFilter(b, x0[size_t(b)], bad);
            }
        f.predictionStepFromSampleTime(int64_t(1000000));  // first call only latches
        printf("after_latch_failed %zu\n", f.lastFailedFilters().size());
        try {
            f.predictionStepFromSampleTime(int64_t(1010000));
            printf("no_throw\n");
            return 1;
        } catch (const std::runtime_error& e) {
            printf("caught %s\n", e.what());
        }
        const std::vector<int64_t> failed = f.lastFailedFilters();
        printf("failed");
        for (int64_t b : failed) printf(" %lld", (long long)b);
        printf("\n");
        for (int64_t b : failed) f.initializeFilter(b, x0[size_t(b)], p0[size_t(b)]);  // back from where they started
        f.predictionStepFromSampleTime(int64_t(1020000));  // the re-initialised filters latch, the others predict
        std::vector<PoseUKF::AngularVelocityMeasurement> w(n);
        for (int64_t b = 0; b < B; ++b)
            for (int i = 0; i < 3; ++i) {
                w[size_t(b)].mu[i] = (i == 2 ? 0.05 : 0.0) + 1e-3 * wobble(b, 0, i);
                w[size_t(b)].cov[i * 3 + i] = 1e-6;
            }
        f.integrateMeasurements(UKFB_MEAS_POSE_ANGULAR_VELOCITY, w.data());
        f.predictionStepFromSampleTime(int64_t(1030000));
        PoseUKF::VelocityMeasurement v;
        v.mu[0] = 1.01;
        for (int i = 0; i < 3; ++i) v.cov[i * 3 + i] = 1e-4;
        f.integrateMeasurement(v);
        printf("after_steps_failed %zu\n", f.lastFailedFilters().size());
        std::vector<PoseUKF::State> xs(n);
        std::vector<PoseUKF::Covariance> ps(n);
        if (!f.getCurrentState(xs.data(), ps.data())) return 2;
        // the per-filter read-backs agree with the whole-batch one
        std::vector<int64_t> rev(n);
        for (int64_t b = 0; b < B; ++b) rev[size_t(b)] = B - 1 - b;
        std::vector<PoseUKF::State> xr(n);
        std::vector<PoseUKF::Covariance> pr(n);
        if (!f.getCurrentStates(B, rev.data(), xr.data(), pr.data())) return 2;
        bool same = true;
        for (int64_t b = 0; b < B; ++b) {
            PoseUKF::State s1, s2;
            PoseUKF::Covariance c1;
            if (!f.getCurrentState(b, s1, c1) || !f.getCurrentState(b, s2)) return 2;
            same = same && memcmp(&s1, &xs[size_t(b)], sizeof(s1)) == 0 && memcmp(&s2, &xs[size_t(b)], sizeof(s2)) == 0 &&
                   memcmp(&c1, &ps[size_t(b)], sizeof(c1)) == 0 && memcmp(&xr[size_t(B - 1 - b)], &xs[size_t(b)], sizeof(s1)) == 0 &&
                   memcmp(&pr[size_t(B - 1 - b)], &ps[size_t(b)], sizeof(c1)) == 0;
        }
        printf("indexed_equals_batch %d\n", int(same));
        for (int64_t b = 0; b < B; ++b) {
            printf("filter %lld", (long long)b);
            for (int i = 0; i < 13; ++i) printf(" %.17g", xs[size_t(b)].v[i]);
            for (int i = 0; i < 144; ++i) printf(" %.17g", ps[size_t(b)].v[i]);
            printf("\n");
        }
        return same ? 0 : 1;
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 3;
    }
}
