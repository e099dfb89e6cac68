// checkpoint_demo.cpp -- a batch PoseUKF object from C++ host code saved and brought back in a second object: some
// filters hold a stored acceleration (the predict then takes the reference's other branch, PoseUKF.cpp:188-192), the
// others the NaN sentinel; after restoreCheckpoint both objects step to bit-identical states.  tests/test_checkpoint.py
// runs it.
// usage: checkpoint_demo <batch>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <vector>

#include <pose_estimation_b200/PoseUKF.hpp>

using namespace pose_estimation_b200;

static double wobble(int64_t b, int k, int c) { return std::sin(0.37 * double(b) + 1.3 * double(k) + 0.71 * double(c)); }

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
    for (int64_t b = 0; b < B; ++b) {
        memset(&x0[size_t(b)], 0, sizeof(PoseUKF::State));
        memset(&p0[size_t(b)], 0, sizeof(PoseUKF::Covariance));
        const double yaw = 0.3 * wobble(b, 20, 0);
        x0[size_t(b)].v[0] = wobble(b, 21, 0);
        x0[size_t(b)].v[5] = std::sin(0.5 * yaw), x0[size_t(b)].v[6] = std::cos(0.5 * yaw);
        x0[size_t(b)].v[7] = 1.0 + 0.1 * wobble(b, 22, 0);
        for (int i = 0; i < 12; ++i) p0[size_t(b)].v[i * 12 + i] = (i < 3 ? 1.0 : 0.01) * (1.0 + 0.2 * wobble(b, 23, i));
    }
    try {
        PoseUKF f(B, x0.data(), p0.data());
        // a stored acceleration on the even filters only (the odd ones keep the NaN sentinel of PoseUKF.cpp:109)
        std::vector<double> acc(n * 3), cov(9, 0.0);
        std::vector<uint8_t> even(n);
        for (int64_t b = 0; b < B; ++b) {
            for (int i = 0; i < 3; ++i) acc[size_t(b) * 3 + i] = 0.1 * wobble(b, 30, i);
            even[size_t(b)] = uint8_t(b % 2 == 0);
        }
        for (int i = 0; i < 3; ++i) cov[size_t(i) * 4] = 1e-3;
        if (ukfb_set_acceleration(f.handle(), acc.data(), cov.data(), 0, even.data()) != UKFB_OK) throw std::runtime_error(ukfb_last_error());
        f.predictionStepFromSampleTime(int64_t(1000000));
        f.predictionStepFromSampleTime(int64_t(1010000));
        const std::vector<uint8_t> image = f.saveCheckpoint();
        printf("image_bytes %zu\n", image.size());

        std::vector<PoseUKF::State> other(n);
        for (auto& s : other) {
            memset(&s, 0, sizeof(s));
            s.v[6] = 1.0;
        }
        PoseUKF g(B, other.data(), p0.data());
        g.restoreCheckpoint(image);
        printf("resaved_equal %d\n", int(g.saveCheckpoint() == image));
        for (PoseUKF* u : {&f, &g}) {
            u->predictionStepFromSampleTime(int64_t(1020000));
            PoseUKF::VelocityMeasurement v;
            v.mu[0] = 1.01;
            for (int i = 0; i < 3; ++i) v.cov[i * 3 + i] = 1e-4;
            u->integrateMeasurement(v);
            u->predictionStepFromSampleTime(int64_t(1030000));
        }
        std::vector<PoseUKF::State> xf(n), xg(n);
        std::vector<PoseUKF::Covariance> pf(n), pg(n);
        if (!f.getCurrentState(xf.data(), pf.data()) || !g.getCurrentState(xg.data(), pg.data())) return 2;
        const bool same = memcmp(xf.data(), xg.data(), sizeof(PoseUKF::State) * n) == 0 &&
                          memcmp(pf.data(), pg.data(), sizeof(PoseUKF::Covariance) * n) == 0;
        printf("states_equal %d\n", int(same));
        return same ? 0 : 1;
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 3;
    }
}
