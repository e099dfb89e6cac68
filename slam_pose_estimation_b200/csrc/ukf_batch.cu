/*
 * ukf_batch.cu -- the C ABI of include/ukf_batch.h over the sm_100a kernels of
 * ukf_device.cuh.  CUDA only: there is no CPU path behind these entry points; every
 * call fails with UKFB_ERR_CUDA when no usable device is present.
 *
 * One handle = B filters of one kind on one device, one stream.  Filter records live in
 * HBM as fixed-size rows (PoseF::REC = 91 / OriF::REC = 105 doubles: mu, then the packed
 * lower triangle of sigma), so the record of a group of filters is one
 * contiguous, coalesced read for the warp that owns the group.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cassert>
#include <cfloat>
#include <cmath>
#include <vector>
#include <cstdarg>
#include <cstdio>
#include <cstddef>
#include <cstring>
#include <new>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <utility>

#include "ukf_device.cuh"
#include "ukf_thread.cuh"
#include "ukf_index.cuh"
#include "ukf_checkpoint.cuh"
#ifndef UKFB_DEFAULT_PREFETCH_BYTES
#define UKFB_DEFAULT_PREFETCH_BYTES 128
#endif
#ifndef UKFB_DEFAULT_WPB
#define UKFB_DEFAULT_WPB 1
#endif
#include "ukf_ori_fast.cuh"
#include "ukf_pose_fast.cuh"

using namespace ukfb;

/* ---- error plumbing ------------------------------------------------------------------ */
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail(UKFB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char* ukfb_last_error(void) { return g_err; }

/* ---- handle ------------------------------------------------------------------------------ */
struct ukfb_handle {
    int kind = 0, device = 0;
    long long B = 0;
    int n = 0, MU = 0, LP = 0, REC = 0;
    int G = 8, WPB = 4, MINB = 3; /* warp kernel launch shape: filters per warp, warps per block, resident blocks per SM */
    int tiled = 1;                /* 1: lane-per-filter kernel, tile-interleaved records; 0: warp-per-group kernel, AoS records */
    int fast = UKFB_SO3_BOXPLUS_LEFT; /* tiled: 1 = structure-exploiting kernels (ukf_pose_fast.cuh, ukf_ori_fast.cuh), 0 = literal kernel (ukf_thread.cuh) */
    cudaStream_t stream = nullptr;
    double* state = nullptr;
    double* Q = nullptr; /* LP (broadcast) or B x LP */
    int q_per_filter = 0;
    int q_diagonal = 0; /* the broadcast Q has no off-diagonal entry (StepParams::q_diagonal) */
    uint32_t* status = nullptr;
    long long* t_last = nullptr;
    unsigned long long* hist = nullptr;
    double* acc_mu = nullptr;
    double* acc_cov = nullptr;
    double gate_d2 = HUGE_VAL; /* accept_any_mahalanobis_distance */
    double* ori_params = nullptr; /* B x 5 per-filter (-1/tau_g, -1/tau_a, earth xyz), or null: the scalars above */
    bool tick_kinds_have_orientation = false; /* set by ukfb_run_dev from its host-side kinds */
    double* gyro_mu = nullptr;
    /* ukfb_set_measurement_cov: a kept covariance per measurement kind (m x m, or B x m x m) for calls that pass cov = NULL */
    double* meas_cov[UKFB_MEAS_KIND_COUNT] = {};
    int meas_cov_per_filter[UKFB_MEAS_KIND_COUNT] = {};
    bool initialized = false, first_init = true;
    double min_dt = UKFB_DEFAULT_MIN_DT, max_dt = DBL_MAX;
    double tau_g = INFINITY, tau_a = INFINITY, latitude = 0.0;
    double earth[3] = {UKFB_EARTHW, 0.0, 0.0};
    /* device staging for host-pointer entry points, grown on demand */
    char* stage = nullptr;
    size_t stage_bytes = 0;
    long long* summary = nullptr; /* 2 words */
    cudaEvent_t ev[16] = {};
    long long launches = 0;
    /* launch configuration of the two fast-kernel instances this handle can run (index = template flag), filled on first
     * use by the handle's single caller: nothing about a launch is shared between handles, so one host thread per handle
     * (the workers of a sharded handle) needs no lock */
    struct FastCfg {
        bool attr_set = false;
        long long prefetch_tiles = -1; /* -1 = not computed yet */
        long long resident_warps = 0;  /* of this kernel on the device (occupancy API) */
    } fast_cfg[2];
    /* consecutive launches of the fast kernels overlap at their ends (StepParams::tile_done): one counter per tile and the
     * number of fast launches made on this handle so far */
    unsigned long long* tile_done = nullptr;
    unsigned long long fast_launches = 0;
    /* ukfb_run_dev: the K tick kinds of the last call, on the device and on the host -- a caller streaming launches with the
     * same schedule then puts nothing but kernels into the stream (a copy between two launches is a full ordering point) */
    int8_t* tick_kinds_dev = nullptr;
    size_t tick_kinds_cap = 0;
    std::vector<int8_t> tick_kinds_last;
    /* sharded parent (ukfb_create_sharded): owns no device memory itself; shard i = filters first[i] .. first[i + 1] */
    std::vector<ukfb_handle*> shards;
    std::vector<long long> first;
    struct ShardPool* pool = nullptr;
    /* pipelined host-pointer calls (ukfb_step_async / ukfb_get_state_async): copy-in and copy-out streams beside the
     * compute stream, two staging slots each, events ordering slot reuse */
    struct Pipe {
        cudaStream_t s_in = nullptr, s_out = nullptr;
        char* in[2] = {nullptr, nullptr};
        char* out[2] = {nullptr, nullptr};
        size_t in_bytes[2] = {0, 0}, out_bytes[2] = {0, 0};
        cudaEvent_t in_ready[2] = {}, in_consumed[2] = {}, out_ready[2] = {}, out_drained[2] = {};
        unsigned long long n_in = 0, n_out = 0;
        bool made = false;
    } pipe;
};

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

/* ---- host-pointer calls: device staging ---------------------------------------------------------------------------- */
/* grows a staging buffer (h->stage, or a slot of h->pipe) to hold `bytes`, in whole MiB.  Whatever may still use the old
 * buffer is waited for before it is freed: h->stream for h->stage, h->stream and both copy streams for a pipe slot. */
static int stage_grow(ukfb_handle* h, char*& buf, size_t& have, size_t bytes, bool pipe_slot)
{
    if (bytes <= have) return UKFB_OK;
    CU(cudaStreamSynchronize(h->stream));
    if (pipe_slot) {
        CU(cudaStreamSynchronize(h->pipe.s_in));
        CU(cudaStreamSynchronize(h->pipe.s_out));
    }
    if (buf) CU(cudaFree(buf));
    buf = nullptr, have = 0;
    const size_t want = (bytes + (size_t(1) << 20)) & ~((size_t(1) << 20) - 1);
    cudaError_t e = cudaMalloc(&buf, want);
    if (e != cudaSuccess)
        return fail(UKFB_ERR_NOMEM, "%sstaging buffer of %zu bytes: %s", pipe_slot ? "pipeline " : "", want, cudaGetErrorString(e));
    have = want;
    return UKFB_OK;
}

static int pipe_make(ukfb_handle* h)
{
    if (h->pipe.made) return UKFB_OK;
    CU(cudaStreamCreateWithFlags(&h->pipe.s_in, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->pipe.s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        CU(cudaEventCreateWithFlags(&h->pipe.in_ready[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->pipe.in_consumed[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->pipe.out_ready[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->pipe.out_drained[i], cudaEventDisableTiming));
    }
    h->pipe.made = true;
    return UKFB_OK;
}

/* The device side of one host-pointer call on one device.  The call registers every part first: in() / in_rows() copy
 * host -> device, out() device -> host; a null host pointer skips its part and leaves its device pointer null.  Then
 * commit() reserves the buffer ONCE for all parts -- growing it frees the old one, so no pointer into it may exist
 * before --, sets the device pointers (256-byte aligned) and queues the host -> device copies.  After the call has
 * enqueued its work on h->stream, finish() queues the device -> host copies and ends the call.
 *   Blocking: h->stage, every copy on h->stream; finish() returns after cudaStreamSynchronize(h->stream).
 *   Pipelined (the _async calls): one of two slots of h->pipe and no synchronisation, but where a slot grows.  A call
 *   with inputs (ukfb_step_async, ukfb_run_events_async; counter pipe.n_in) copies them on s_in into slot n_in & 1 once
 *   the launch that last read that slot is done (in_consumed), and its launch waits for the copies (in_ready).  A call
 *   with outputs only (the _async getters; counter pipe.n_out) unpacks into slot n_out & 1 once the copies that last
 *   read that slot are done (out_drained), and its copies on s_out wait for the unpack (out_ready).
 * The host arrays of a pipelined call must stay valid and unchanged until ukfb_synchronize(). */
struct Staging {
    explicit Staging(ukfb_handle* h_, bool pipelined_) : h(h_), pipelined(pipelined_) {}

    template <class T>
    void in(T** dev, const void* src, size_t bytes) { add(dev, src, nullptr, bytes, 1, bytes); }
    /* `rows` rows of `width` bytes, `pitch` bytes apart on the host (a shard's slice of slot-major K x B arrays), dense on
     * the device */
    template <class T>
    void in_rows(T** dev, const void* src, size_t width, size_t rows, size_t pitch) { add(dev, src, nullptr, width, rows, pitch); }
    template <class T>
    void out(T** dev, void* dst, size_t bytes) { add(dev, nullptr, dst, bytes, 1, bytes); }
    /* device room without copies: the call moves the data itself, on h->stream (the checkpoint calls, whose sections go
     * to or come from several places of the caller's buffer) */
    template <class T>
    void scratch(T** dev, size_t bytes) { add(dev, nullptr, nullptr, bytes, 1, bytes, true); }

    int commit()
    {
        size_t end = 0;
        for (int i = 0; i < n; ++i) end = align256(end) + part[i].width * part[i].rows;
        char* base;
        if (!pipelined) {
            if (int rc = stage_grow(h, h->stage, h->stage_bytes, end, false)) return rc;
            base = h->stage;
            cs = h->stream;
        } else {
            if (int rc = pipe_make(h)) return rc;
            ukfb_handle::Pipe& p = h->pipe;
            for (int i = 0; i < n; ++i) inputs = inputs || part[i].src;
            slot = int((inputs ? p.n_in : p.n_out) & 1);
            char*& buf = inputs ? p.in[slot] : p.out[slot];
            if (int rc = stage_grow(h, buf, inputs ? p.in_bytes[slot] : p.out_bytes[slot], end, true)) return rc;
            base = buf;
            cs = inputs ? p.s_in : p.s_out;
            if (inputs && p.n_in >= 2) CU(cudaStreamWaitEvent(cs, p.in_consumed[slot], 0)); /* the launch that read this slot is done */
            if (!inputs && p.n_out >= 2) CU(cudaStreamWaitEvent(h->stream, p.out_drained[slot], 0)); /* the copies that read it are done */
        }
        size_t off = 0;
        for (int i = 0; i < n; ++i) {
            Part& q = part[i];
            off = align256(off);
            q.at = base + off;
            off += q.width * q.rows;
            q.set(q.dev, q.at);
            if (q.src && q.width == q.pitch)
                CU(cudaMemcpyAsync(q.at, q.src, q.width * q.rows, cudaMemcpyHostToDevice, cs));
            else if (q.src)
                CU(cudaMemcpy2DAsync(q.at, q.width, q.src, q.pitch, q.width, q.rows, cudaMemcpyHostToDevice, cs));
        }
        if (pipelined && inputs) {
            CU(cudaEventRecord(h->pipe.in_ready[slot], cs));
            CU(cudaStreamWaitEvent(h->stream, h->pipe.in_ready[slot], 0));
        }
        return UKFB_OK;
    }

    int finish()
    {
        ukfb_handle::Pipe& p = h->pipe;
        if (pipelined && inputs) {
            CU(cudaEventRecord(p.in_consumed[slot], h->stream));
            p.n_in++;
            return UKFB_OK;
        }
        if (pipelined) {
            CU(cudaEventRecord(p.out_ready[slot], h->stream));
            CU(cudaStreamWaitEvent(cs, p.out_ready[slot], 0));
        }
        for (int i = 0; i < n; ++i)
            if (part[i].dst) CU(cudaMemcpyAsync(part[i].dst, part[i].at, part[i].width, cudaMemcpyDeviceToHost, cs));
        if (!pipelined) {
            CU(cudaStreamSynchronize(h->stream));
            return UKFB_OK;
        }
        CU(cudaEventRecord(p.out_drained[slot], cs));
        p.n_out++;
        return UKFB_OK;
    }

private:
    struct Part {
        void* dev;                /* the caller's T* to set */
        void (*set)(void*, char*); /* stores the device address into it as a T* */
        const void* src;          /* host -> device */
        void* dst;                /* device -> host */
        size_t width, rows, pitch;
        char* at;                 /* device address, from commit() on */
    };
    template <class T>
    void add(T** dev, const void* src, void* dst, size_t width, size_t rows, size_t pitch, bool keep = false)
    {
        *dev = nullptr;
        if (!src && !dst && !keep) return;
        assert(n < MAX_PARTS);
        part[n++] = Part{dev, [](void* d, char* a) { *static_cast<T**>(d) = reinterpret_cast<T*>(a); }, src, dst, width, rows, pitch, nullptr};
    }
    static constexpr int MAX_PARTS = 4;
    ukfb_handle* h;
    bool pipelined;
    bool inputs = false; /* pipelined: the call uses the input side of the pipe */
    int slot = 0;
    cudaStream_t cs = nullptr; /* the stream of the copies */
    Part part[MAX_PARTS];
    int n = 0;
};

struct Bind { /* sets the device for the duration of a call */
    int prev = -1;
    bool ok = true;
    explicit Bind(const ukfb_handle* h)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != h->device) ok = cudaSetDevice(h->device) == cudaSuccess;
    }
    ~Bind()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

/* `who`: the entry point named in the error text */
#define CHECK_H_AS(h, who)                                                \
    if (!(h)) return fail(UKFB_ERR_INVALID, "%s: null handle", who);      \
    Bind bind_(h);                                                        \
    if (!bind_.ok) return fail(UKFB_ERR_CUDA, "%s: cudaSetDevice(%d) failed", who, (h)->device)
#define CHECK_H(h) CHECK_H_AS(h, __func__)

/* ---- sharded handles: one worker thread per shard ---------------------------------------------------------------- */
/* Filters share nothing (UnscentedKalmanFilter.hpp:150-154), so a sharded parent is just a list of one-device handles
 * over contiguous index ranges.  Every host-pointer entry point starts with UKFB_FAN: on a parent it hands the SAME
 * call, with the caller's arrays advanced to the shard's first filter, to each shard's worker and waits for all of them
 * (copies to / from the devices and the final synchronisations of the shards then run concurrently). */
struct ShardPool {
    struct Worker {
        std::thread th;
        int rc = 0;
        std::string err;
    };
    std::vector<Worker> w;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    std::function<int(int)> job;
    unsigned long long generation = 0;
    int pending = 0;
    bool quit = false;

    explicit ShardPool(int n) : w(size_t(n))
    {
        for (int i = 0; i < n; ++i) w[size_t(i)].th = std::thread([this, i] { loop(i); });
    }
    ~ShardPool()
    {
        {
            std::lock_guard<std::mutex> lock(mu);
            quit = true;
        }
        cv_job.notify_all();
        for (auto& x : w)
            if (x.th.joinable()) x.th.join();
    }
    void loop(int i)
    {
        unsigned long long seen = 0;
        for (;;) {
            std::function<int(int)> fn;
            {
                std::unique_lock<std::mutex> lock(mu);
                cv_job.wait(lock, [&] { return quit || generation != seen; });
                if (quit) return;
                seen = generation;
                fn = job;
            }
            const int rc = fn(i);
            std::string err = rc ? std::string(ukfb_last_error()) : std::string();
            {
                std::lock_guard<std::mutex> lock(mu);
                w[size_t(i)].rc = rc;
                w[size_t(i)].err.swap(err);
                if (--pending == 0) cv_done.notify_all();
            }
        }
    }
    /* runs fn(i) on every worker; returns the first non-zero result (its text in *err) */
    int run(const std::function<int(int)>& fn, std::string* err, int* who)
    {
        std::unique_lock<std::mutex> lock(mu);
        job = fn;
        pending = int(w.size());
        ++generation;
        cv_job.notify_all();
        cv_done.wait(lock, [&] { return pending == 0; });
        for (size_t i = 0; i < w.size(); ++i)
            if (w[i].rc) {
                *err = w[i].err;
                *who = int(i);
                return w[i].rc;
            }
        return 0;
    }
};

static inline bool is_sharded(const ukfb_handle* h) { return h && !h->shards.empty(); }

/* fn(shard handle, first filter of the shard, number of filters) on every shard, concurrently */
template <class Fn>
static int fan_out(ukfb_handle* h, Fn fn)
{
    std::string err;
    int who = -1;
    const int rc = h->pool->run([&](int i) { return fn(h->shards[size_t(i)], h->first[size_t(i)], h->first[size_t(i) + 1] - h->first[size_t(i)]); },
                                &err, &who);
    if (rc) return fail(rc, "shard %d (device %d): %s", who, h->shards[size_t(who)]->device, err.c_str());
    return UKFB_OK;
}

#define UKFB_FAN(h, call)                                                                                   \
    if (is_sharded(h)) return fan_out(h, [&](ukfb_handle* s_, long long f_, long long c_) -> int { (void)f_; (void)c_; return (call); })
/* `_dev` entry points take pointers of one device */
#define UKFB_NOT_SHARDED(h)                                                                                   \
    if (is_sharded(h)) return fail(UKFB_ERR_INVALID, "%s: device pointers belong to one device -- use the per-device handles of ukfb_shard()", __func__)

/* ---- small kernels ------------------------------------------------------------------------- */

/* rec_index (record entry e of filter b in either layout): ukf_index.cuh */

/* host layout (mu B x MU, sigma B x n x n) -> records */
__global__ void pack_kernel(double* __restrict__ state, const double* __restrict__ mu, const double* __restrict__ sigma,
                            long long B, int n, int MU, int LP, int REC, int tiled)
{
    const long long total = B * REC;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / REC;
        const int k = int(i - b * REC);
        double v = 0.0;
        if (k < MU)
            v = mu[b * MU + k];
        else {
            const int e = k - MU;
            int r = 0;
            while ((r + 1) * (r + 2) / 2 <= e) ++r;
            const int c = e - r * (r + 1) / 2;
            v = sigma[(b * n + r) * n + c];
        }
        state[rec_index(tiled, b, k, REC)] = v;
    }
}

__global__ void unpack_mu_kernel(const double* __restrict__ state, double* __restrict__ mu, long long B, int MU, int REC, int tiled)
{
    const long long total = B * MU;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / MU;
        const int k = int(i - b * MU);
        mu[i] = state[rec_index(tiled, b, k, REC)];
    }
}

__global__ void unpack_sigma_kernel(const double* __restrict__ state, double* __restrict__ sigma, long long B, int n, int MU, int REC, int tiled)
{
    const long long total = B * n * n;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / (n * n);
        const int e = int(i - b * n * n);
        int r = e / n, c = e - (e / n) * n;
        if (c > r) {
            const int t = r;
            r = c;
            c = t;
        }
        sigma[i] = state[rec_index(tiled, b, MU + tri(r, c), REC)];
    }
}

/* BodyStateMeasurement::fromRigidBodyState (BodyStateMeasurement.hpp:14-26): RigidBodyState records -> PoseUKF records */
__global__ void pack_rbs_kernel(double* __restrict__ state, const double* __restrict__ rbs, long long B, int tiled)
{
    const long long total = B * PoseF::REC;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / PoseF::REC;
        const int k = int(i - b * PoseF::REC);
        const double* r = rbs + b * UKFB_RBS_DOUBLES;
        double v = 0.0;
        if (k < PoseF::MU)
            v = r[k]; /* position, orientation, velocity, angular velocity: the same order as mu */
        else {
            const int e = k - PoseF::MU;
            int row = 0;
            while ((row + 1) * (row + 2) / 2 <= e) ++row;
            const int col = e - row * (row + 1) / 2;
            if (row / 3 == col / 3) v = r[13 + (row / 3) * 9 + (row % 3) * 3 + (col % 3)];
        }
        state[rec_index(tiled, b, k, PoseF::REC)] = v;
    }
}

/* BodyStateMeasurement::toRigidBodyState (BodyStateMeasurement.hpp:28-39) */
__global__ void unpack_rbs_kernel(const double* __restrict__ state, double* __restrict__ rbs, long long B, int tiled)
{
    const long long total = B * UKFB_RBS_DOUBLES;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / UKFB_RBS_DOUBLES;
        const int k = int(i - b * UKFB_RBS_DOUBLES);
        double v;
        if (k >= 7 && k < 10) { /* velocity: rotated into the navigation frame (:32) */
            double q[4], bv[3], nv[3];
            for (int j = 0; j < 4; ++j) q[j] = state[rec_index(tiled, b, 3 + j, PoseF::REC)];
            for (int j = 0; j < 3; ++j) bv[j] = state[rec_index(tiled, b, 7 + j, PoseF::REC)];
            quat_rotate(q, bv, nv);
            v = nv[k - 7];
        } else if (k < PoseF::MU)
            v = state[rec_index(tiled, b, k, PoseF::REC)];
        else {
            const int blk = (k - 13) / 9, e = (k - 13) % 9;
            int row = blk * 3 + e / 3, col = blk * 3 + e % 3;
            if (col > row) {
                const int t = row;
                row = col;
                col = t;
            }
            v = state[rec_index(tiled, b, PoseF::MU + tri(row, col), PoseF::REC)];
        }
        rbs[i] = v;
    }
}

/* packed lower triangle of Q from full n x n matrices */
__global__ void pack_q_kernel(double* __restrict__ Qp, const double* __restrict__ Q, long long count, int n, int LP)
{
    const long long total = count * LP;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / LP;
        const int e = int(i - b * LP);
        int r = 0;
        while ((r + 1) * (r + 2) / 2 <= e) ++r;
        const int c = e - r * (r + 1) / 2;
        Qp[i] = Q[(b * n + r) * n + c];
    }
}

__global__ void unpack_q_kernel(const double* __restrict__ Qp, double* __restrict__ Q, long long count, int n, int LP, long long q_stride)
{
    const long long total = count * n * n;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / (n * n);
        const int e = int(i - b * n * n);
        int r = e / n, c = e - (e / n) * n;
        if (c > r) {
            const int t = r;
            r = c;
            c = t;
        }
        Q[i] = Qp[b * q_stride + tri(r, c)];
    }
}

template <typename T>
__global__ void fill_kernel(T* __restrict__ dst, long long count, T v)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) dst[i] = v;
}

/* B identity 3x3 matrices (Measurement.hpp:11: cov = Identity) */
__global__ void eye3_kernel(double* __restrict__ dst, long long count)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
        dst[i] = ((i % 9) % 4 == 0) ? 1.0 : 0.0;
}

/* store a 3-vector measurement (and optionally its 3x3 covariance) per filter, masked;
 * check = 1: checkMeasurment (UnscentedKalmanFilter.hpp:142-147) -- a non-finite sample is
 * flagged and not stored, as the throw would have prevented the assignment. */
__global__ void store_vec3_kernel(double* __restrict__ dst_mu, double* __restrict__ dst_cov, const double* __restrict__ mu,
                                  const double* __restrict__ cov, long long cov_stride, const uint8_t* __restrict__ mask,
                                  uint32_t* __restrict__ status, int check, long long B)
{
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        if (mask && !mask[b]) continue;
        const double m0 = mu[b * 3], m1 = mu[b * 3 + 1], m2 = mu[b * 3 + 2];
        double c[9];
        for (int i = 0; i < 9; ++i) c[i] = cov ? cov[b * cov_stride + i] : ((i % 4 == 0) ? 1.0 : 0.0);
        if (check) {
            bool ok = isfinite(m0) && isfinite(m1) && isfinite(m2);
            for (int i = 0; i < 9; ++i) ok = ok && isfinite(c[i]);
            if (!ok) {
                status[b] |= UKFB_STATUS_NONFINITE_MEAS;
                continue;
            }
        }
        dst_mu[b * 3] = m0, dst_mu[b * 3 + 1] = m1, dst_mu[b * 3 + 2] = m2;
        if (dst_cov)
            for (int i = 0; i < 9; ++i) dst_cov[b * 9 + i] = c[i];
    }
}

/* OrientationUKF::getRotationRate (OrientationUKF.cpp:74-77) */
__global__ void rotation_rate_kernel(const double* __restrict__ state, const double* __restrict__ gyro, double e0, double e1,
                                     double e2, const double* __restrict__ ori_params, double* __restrict__ out, long long B, int tiled)
{
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        double q[4];
        for (int i = 0; i < 4; ++i) q[i] = state[rec_index(tiled, b, i, OriF::REC)];
        double e[3] = {e0, e1, e2};
        if (ori_params) e[0] = ori_params[b * 5 + 2], e[1] = ori_params[b * 5 + 3], e[2] = ori_params[b * 5 + 4];
        double r[3];
        quat_inv_rotate(q, e, r);
        for (int i = 0; i < 3; ++i) out[b * 3 + i] = gyro[b * 3 + i] - state[rec_index(tiled, b, 7 + i, OriF::REC)] - r[i];
    }
}

/* initial stored acceleration of OrientationUKF: (0, 0, gravity) (OrientationUKF.cpp:50) */
__global__ void ori_default_imu_kernel(const double* __restrict__ state, double* __restrict__ acc, double* __restrict__ gyro,
                                       long long B, int tiled)
{
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        acc[b * 3] = 0.0, acc[b * 3 + 1] = 0.0, acc[b * 3 + 2] = state[rec_index(tiled, b, 13, OriF::REC)];
        gyro[b * 3] = gyro[b * 3 + 1] = gyro[b * 3 + 2] = 0.0;
    }
}

__global__ void status_summary_kernel(const uint32_t* __restrict__ status, long long B, long long* __restrict__ out)
{
    long long n = 0;
    unsigned bits = 0;
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const uint32_t s = status[b];
        n += s != 0;
        bits |= s;
    }
    for (int o = 16; o; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        bits |= __shfl_xor_sync(0xffffffffu, bits, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (n) atomicAdd(reinterpret_cast<unsigned long long*>(out), (unsigned long long)n);
        if (bits) atomicOr(reinterpret_cast<unsigned long long*>(out + 1), (unsigned long long)bits);
    }
}

/* independent DFMA chains: the FP64 roofline denominator */
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = fma(x0, a, b), x1 = fma(x1, a, b), x2 = fma(x2, a, b), x3 = fma(x3, a, b);
            x4 = fma(x4, a, b), x5 = fma(x5, a, b), x6 = fma(x6, a, b), x7 = fma(x7, a, b);
        }
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 12345.678) out[0] = s;
}

static inline int grid_for(long long count, int block = 256)
{
    long long g = (count + block - 1) / block;
    if (g < 1) g = 1;
    if (g > 148 * 16) g = 148 * 16;
    return int(g);
}

/* ---- step launch ------------------------------------------------------------------------------ */
/* process-wide tuning knobs from the environment, read once (thread-safe: function-local static initialisation) */
struct EnvKnobs {
    int fast_wpb;              /* UKFB_FAST_WPB: warps per block of the two fast kernels, 1 | 2 | 4 */
    long smem_pad_kb;          /* UKFB_SMEM_PAD_KB: unused dynamic shared memory per block (occupancy experiments) */
    int prefetch_bytes;        /* UKFB_PREFETCH_BYTES: request granularity of the next-wave prefetch (one L2 line) */
    long long prefetch_tiles;  /* UKFB_PREFETCH_TILES: forced prefetch distance, -1 = from the occupancy API, 0 = off */
    bool overlap;              /* UKFB_OVERLAP_LAUNCHES=0: every fast-kernel launch waits for the whole previous one */
    int overlap_max_waves;     /* UKFB_OVERLAP_MAX_WAVES: overlap launches of grids up to this many waves of resident warps (12) */
    int overlap_min_waves_pct; /* UKFB_OVERLAP_MIN_WAVES_PCT: ... and of more than this many hundredths of a wave (100) */
    bool ckpt_elem;            /* UKFB_CKPT_TRANSFORM=elem: checkpoint record transforms per element instead of per tile */
    EnvKnobs()
    {
        const char* e = getenv("UKFB_FAST_WPB");
        const int v = e ? atoi(e) : UKFB_DEFAULT_WPB;
        fast_wpb = (v == 1 || v == 2 || v == 4) ? v : UKFB_DEFAULT_WPB;
        e = getenv("UKFB_SMEM_PAD_KB");
        smem_pad_kb = e ? atol(e) : 0;
        e = getenv("UKFB_PREFETCH_BYTES");
        prefetch_bytes = e && atoi(e) >= 8 ? atoi(e) : UKFB_DEFAULT_PREFETCH_BYTES;
        e = getenv("UKFB_PREFETCH_TILES");
        prefetch_tiles = e ? atoll(e) : -1;
        e = getenv("UKFB_OVERLAP_LAUNCHES");
        overlap = e ? atoi(e) != 0 : true;
        e = getenv("UKFB_OVERLAP_MAX_WAVES");
        overlap_max_waves = e && atoi(e) > 0 ? atoi(e) : 12;
        e = getenv("UKFB_OVERLAP_MIN_WAVES_PCT");
        overlap_min_waves_pct = e ? atoi(e) : 100;
        e = getenv("UKFB_CKPT_TRANSFORM");
        ckpt_elem = e && strcmp(e, "elem") == 0;
    }
};
static const EnvKnobs& knobs()
{
    static const EnvKnobs k;
    return k;
}

/* cudaFuncSetAttribute is per (function, device): remembered under a lock, keyed by the kernel's address (all step
 * kernels share one function-pointer type, so a per-type static would be shared between them) */
static std::mutex g_attr_mu;
template <class K>
static cudaError_t ensure_smem_attr(K kernel, int device, size_t smem)
{
    static std::vector<std::pair<const void*, int>> done;
    const std::pair<const void*, int> key(reinterpret_cast<const void*>(kernel), device);
    std::lock_guard<std::mutex> lock(g_attr_mu);
    for (const auto& d : done)
        if (d == key) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e == cudaSuccess) done.push_back(key);
    return e;
}

template <class F, int G, int WPB, int MINB>
static cudaError_t launch_step_t(const ukfb_handle* h, const StepParams& p)
{
    const size_t smem = sizeof(double) * WPB * Smem<F, G>::TOTAL;
    cudaError_t e = ensure_smem_attr(ukf_step_kernel<F, G, WPB, MINB>, h->device, smem);
    if (e != cudaSuccess) return e;
    const long long per_block = (long long)WPB * G;
    const long long grid = (p.B + per_block - 1) / per_block;
    ukf_step_kernel<F, G, WPB, MINB><<<unsigned(grid), WPB * 32, smem, h->stream>>>(p);
    return cudaGetLastError();
}

/* launch shapes: G filters per warp (32/G lanes per filter in the Cholesky phases), WPB warps per block */
template <class F>
static cudaError_t launch_step_f(const ukfb_handle* h, const StepParams& p)
{
    switch (h->G * 100 + h->WPB * 10 + h->MINB) {
        case 443: return launch_step_t<F, 4, 4, 3>(h, p);
        case 444: return launch_step_t<F, 4, 4, 4>(h, p);
        case 1642: return launch_step_t<F, 16, 4, 2>(h, p);
        case 1652: return launch_step_t<F, 16, 5, 2>(h, p);
        case 842: return launch_step_t<F, 8, 4, 2>(h, p);
        case 844: return launch_step_t<F, 8, 4, 4>(h, p);
        default: return launch_step_t<F, 8, 4, 3>(h, p);
    }
}

template <class F>
static cudaError_t launch_thread_f(const ukfb_handle* h, const StepParams& p)
{
    const size_t smem = sizeof(double) * TSmem<F>::TOTAL;
    cudaError_t e = ensure_smem_attr(ukf_thread_kernel<F>, h->device, smem);
    if (e != cudaSuccess) return e;
    const long long grid = (p.B + TILE - 1) / TILE;
    ukf_thread_kernel<F><<<unsigned(grid), TILE, smem, h->stream>>>(p);
    return cudaGetLastError();
}

/* kernel: the plain instance; kernel_overlap: the one whose launches overlap at their ends (chosen per handle, below) */
template <class K>
static cudaError_t launch_fast(K kernel, K kernel_overlap, int per_lane, ukfb_handle* h, const StepParams& p, ukfb_handle::FastCfg& cfg)
{
    const EnvKnobs& kn = knobs();
    const int wpb = kn.fast_wpb;
    const size_t smem = sizeof(double) * per_lane * TILE * wpb + size_t(kn.smem_pad_kb) * 1024;
    if (!cfg.attr_set) {
        cudaError_t e = ensure_smem_attr(kernel, h->device, smem);
        if (e == cudaSuccess) e = ensure_smem_attr(kernel_overlap, h->device, smem);
        if (e != cudaSuccess) return e;
        cfg.attr_set = true;
    }
    const long long tiles = (p.B + TILE - 1) / TILE;
    const long long grid = (tiles + wpb - 1) / wpb; /* warps past the last tile return at once */
    StepParams q = p;
    /* prefetch distance = a quarter of the resident warps of this kernel on the device (measured on B200, pose C4:
     * flat optimum from 32 to 444 tiles with 1184 resident warps, -2 % at 888, no gain from 1184 on;
     * UKFB_PREFETCH_TILES overrides, 0 = off), request granularity UKFB_PREFETCH_BYTES (one L2 line) */
    if (cfg.prefetch_tiles < 0) {
        int per_sm = 0, sms = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TILE * wpb, smem) != cudaSuccess) per_sm = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device) != cudaSuccess) sms = 0;
        cfg.resident_warps = (long long)per_sm * wpb * sms;
        long long r = kn.prefetch_tiles;
        if (r < 0) {
            r = cfg.resident_warps / 4;
            if (r < 32 && per_sm > 0) r = 32;
        }
        cfg.prefetch_tiles = r > 0 ? r : 0;
    }
    q.prefetch_tiles = cfg.prefetch_tiles;
    q.prefetch_bytes = kn.prefetch_bytes;
    /* Launch number n of this handle's fast kernels waits, tile by tile, for launch n - 1 (tile_done), so the stream need not
     * hold it back until the whole of n - 1 has drained: with programmatic stream serialization its blocks are scheduled as
     * soon as every block of n - 1 has started, i.e. into the slots the last, partial wave of n - 1 leaves empty.
     * The handshake costs every warp an L2 round trip before its first load and a fence after its last store (measured: 3 %
     * of a step), the overlap recovers about half a wave plus the launch gap: it pays for grids of a few waves (a shard of
     * 128 Ki filters: +9 %, 256 Ki: +4 %) and not for many (1 Mi filters, 28 waves: -2 %), and the blocks of a grid of
     * less than one wave would all be resident, waiting.  The batch size of a handle is fixed, so a handle either always
     * or never launches this way.  Whatever else is in the stream (copies, the pack / unpack kernels, another kernel
     * family) keeps full stream order on both sides. */
    const bool overlap = kn.overlap && cfg.resident_warps > 0 && grid * wpb * 100 > kn.overlap_min_waves_pct * cfg.resident_warps &&
                         grid * wpb <= kn.overlap_max_waves * cfg.resident_warps;
    q.tile_done = overlap ? h->tile_done : nullptr;
    q.launch_seq = h->fast_launches + 1;
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3(unsigned(grid));
    lc.blockDim = dim3(TILE * wpb);
    lc.dynamicSmemBytes = smem;
    lc.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at;
    lc.numAttrs = overlap ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&lc, overlap ? kernel_overlap : kernel, q);
    if (e != cudaSuccess) return e;
    if (overlap) h->fast_launches++; /* only a launch that was made adds to the counters */
    return cudaGetLastError();
}

static cudaError_t launch_pose_fast(ukfb_handle* h, const StepParams& p, bool may_have_orientation_meas)
{
    if (may_have_orientation_meas) return launch_fast(ukf_pose_fast_kernel<true, false>, ukf_pose_fast_kernel<true, true>, PF_PER_LANE, h, p, h->fast_cfg[1]);
    return launch_fast(ukf_pose_fast_kernel<false, false>, ukf_pose_fast_kernel<false, true>, PF_PER_LANE, h, p, h->fast_cfg[0]);
}

static cudaError_t launch_ori_fast(ukfb_handle* h, const StepParams& p)
{
    if (p.ori_params) return launch_fast(ukf_ori_fast_kernel<true, false>, ukf_ori_fast_kernel<true, true>, OF_PER_LANE, h, p, h->fast_cfg[1]);
    return launch_fast(ukf_ori_fast_kernel<false, false>, ukf_ori_fast_kernel<false, true>, OF_PER_LANE, h, p, h->fast_cfg[0]);
}

static int launch_step(ukfb_handle* h, const StepParams& p)
{
    cudaError_t e;
    if (h->tiled && h->fast && h->kind == UKFB_POSE) {
        /* can an OrientationMeasurement occur in this launch?  per-filter kinds live on the device: assume yes */
        bool ori_meas = p.do_update && (p.kind == UKFB_MEAS_POSE_ORIENTATION || p.kind == -2 || p.events);
        if (p.do_update && p.tick_kinds) ori_meas = h->tick_kinds_have_orientation;
        e = launch_pose_fast(h, p, ori_meas);
    }
    else if (h->tiled && h->fast)
        e = launch_ori_fast(h, p);
    else if (h->tiled)
        e = h->kind == UKFB_POSE ? launch_thread_f<PoseF>(h, p) : launch_thread_f<OriF>(h, p);
    else
        e = h->kind == UKFB_POSE ? launch_step_f<PoseF>(h, p) : launch_step_f<OriF>(h, p);
    if (e != cudaSuccess) return fail(UKFB_ERR_CUDA, "ukf_step_kernel launch: %s", cudaGetErrorString(e));
    h->launches++;
    return UKFB_OK;
}

static StepParams base_params(const ukfb_handle* h)
{
    StepParams p;
    memset(&p, 0, sizeof(p));
    p.state = h->state;
    p.Q = h->Q;
    p.q_stride = h->q_per_filter ? h->LP : 0;
    p.q_diagonal = h->q_per_filter ? 0 : h->q_diagonal;
    p.B = h->B;
    p.status = h->status;
    p.t_last = h->t_last;
    p.hist = h->hist;
    p.min_dt = h->min_dt;
    p.max_dt = h->max_dt;
    p.acc_mu = h->acc_mu;
    p.acc_cov = h->acc_cov;
    p.gyro_mu = h->gyro_mu;
    p.neg_inv_tau_g = -1.0 / h->tau_g;
    p.neg_inv_tau_a = -1.0 / h->tau_a;
    p.earth[0] = h->earth[0], p.earth[1] = h->earth[1], p.earth[2] = h->earth[2];
    p.kind = -1;
    p.K = 1;
    p.gate_d2 = h->gate_d2;
    p.ori_params = h->ori_params;
    return p;
}

static bool kind_ok(const ukfb_handle* h, int kind)
{
    if (h->kind == UKFB_POSE) return kind >= 0 && kind <= 8;
    return kind == UKFB_MEAS_ORI_VELOCITY;
}

#define NEED_INIT_AS(h, who) \
    if (!(h)->initialized) return fail(UKFB_ERR_NOT_INITIALIZED, "%s: filter not initialized", who)
#define NEED_INIT(h) NEED_INIT_AS(h, __func__)

/* ---- lifecycle ---------------------------------------------------------------------------------- */
extern "C" int ukfb_create(int filter_kind, int64_t batch, int device, ukfb_handle** out)
{
    if (!out) return fail(UKFB_ERR_INVALID, "ukfb_create: out is null");
    *out = nullptr;
    if (filter_kind != UKFB_POSE && filter_kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_create: bad filter kind %d", filter_kind);
    if (batch < 1) return fail(UKFB_ERR_INVALID, "ukfb_create: batch must be >= 1");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(UKFB_ERR_CUDA, "ukfb_create: no CUDA device (%s); this engine has no CPU path", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(UKFB_ERR_INVALID, "ukfb_create: device %d out of range (%d devices)", device, ndev);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(UKFB_ERR_CUDA, "ukfb_create: device %d is sm_%d%d; the kernels are built for sm_100a only", device, prop.major, prop.minor);

    ukfb_handle* h = new (std::nothrow) ukfb_handle;
    if (!h) return fail(UKFB_ERR_NOMEM, "ukfb_create: out of host memory");
    h->kind = filter_kind;
    h->device = device;
    h->B = batch;
    if (filter_kind == UKFB_POSE)
        h->n = PoseF::N, h->MU = PoseF::MU, h->LP = PoseF::LP, h->REC = PoseF::REC;
    else
        h->n = OriF::N, h->MU = OriF::MU, h->LP = OriF::LP, h->REC = OriF::REC;
    if (const char* g = getenv("UKFB_GROUP")) {
        const int G = atoi(g);
        if (G == 4 || G == 8 || G == 16) h->G = G;
    }
    if (const char* g = getenv("UKFB_KERNEL")) { /* fast (default) | thread (literal lane-per-filter) | warp (literal warp-per-group) */
        h->tiled = strcmp(g, "warp") != 0;
        if (strcmp(g, "thread") == 0) h->fast = 0;
    }
    if (const char* g = getenv("UKFB_WARP_WPB")) h->WPB = atoi(g); /* warp-per-group kernel only; the fast kernels: UKFB_FAST_WPB */
    if (const char* g = getenv("UKFB_MINB")) h->MINB = atoi(g);
    Bind bind_(h);
    if (!bind_.ok) {
        delete h;
        return fail(UKFB_ERR_CUDA, "ukfb_create: cudaSetDevice(%d) failed", device);
    }
#define CUH(call)                                                                     \
    do {                                                                              \
        cudaError_t e_ = (call);                                                      \
        if (e_ != cudaSuccess) {                                                      \
            fail(e_ == cudaErrorMemoryAllocation ? UKFB_ERR_NOMEM : UKFB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
            ukfb_destroy(h);                                                          \
            return e_ == cudaErrorMemoryAllocation ? UKFB_ERR_NOMEM : UKFB_ERR_CUDA; \
        }                                                                             \
    } while (0)
    const long long B = batch;
    CUH(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    const long long Bpad = (B + TILE - 1) / TILE * TILE; /* whole tiles: lanes past the end address valid memory */
    CUH(cudaMalloc(&h->state, sizeof(double) * Bpad * h->REC));
    CUH(cudaMalloc(&h->Q, sizeof(double) * h->LP));
    CUH(cudaMalloc(&h->status, sizeof(uint32_t) * B));
    CUH(cudaMalloc(&h->t_last, sizeof(long long) * B));
    CUH(cudaMalloc(&h->hist, sizeof(unsigned long long) * HIST_SLOTS * 8));
    CUH(cudaMalloc(&h->acc_mu, sizeof(double) * B * 3));
    CUH(cudaMalloc(&h->acc_cov, sizeof(double) * B * 9));
    CUH(cudaMalloc(&h->gyro_mu, sizeof(double) * B * 3));
    CUH(cudaMalloc(&h->summary, sizeof(long long) * 2));
    CUH(cudaMalloc(&h->tile_done, sizeof(unsigned long long) * (Bpad / TILE)));
    CUH(cudaMemsetAsync(h->tile_done, 0, sizeof(unsigned long long) * (Bpad / TILE), h->stream));
    CUH(cudaMemsetAsync(h->state, 0, sizeof(double) * Bpad * h->REC, h->stream));
    CUH(cudaMemsetAsync(h->status, 0, sizeof(uint32_t) * B, h->stream));
    CUH(cudaMemsetAsync(h->t_last, 0, sizeof(long long) * B, h->stream));
    CUH(cudaMemsetAsync(h->hist, 0, sizeof(unsigned long long) * HIST_SLOTS * 8, h->stream));
    CUH(cudaMemsetAsync(h->gyro_mu, 0, sizeof(double) * B * 3, h->stream));
    /* Q: zero (base ctor) then the PoseUKF default diagonal (PoseUKF.cpp:103-107) */
    {
        double q[OriF::LP];
        for (int i = 0; i < OriF::LP; ++i) q[i] = 0.0;
        if (filter_kind == UKFB_POSE) {
            const double d[4] = {UKFB_POSE_Q_POSITION, UKFB_POSE_Q_ORIENTATION, UKFB_POSE_Q_VELOCITY, UKFB_POSE_Q_ANGULAR_VELOCITY};
            for (int i = 0; i < 12; ++i) q[tri(i, i)] = d[i / 3];
        }
        CUH(cudaMemcpyAsync(h->Q, q, sizeof(double) * h->LP, cudaMemcpyHostToDevice, h->stream));
        CUH(cudaStreamSynchronize(h->stream));
        h->q_diagonal = 2; /* zero, or the PoseUKF default diagonal (one value per 3 x 3 block) */
    }
    /* stored acceleration: NaN sentinel for PoseUKF (PoseUKF.cpp:109), identity covariance (Measurement.hpp:11) */
    fill_kernel<double><<<grid_for(B * 3), 256, 0, h->stream>>>(h->acc_mu, B * 3, filter_kind == UKFB_POSE ? double(NAN) : 0.0);
    eye3_kernel<<<grid_for(B * 9), 256, 0, h->stream>>>(h->acc_cov, B * 9);
    for (int i = 0; i < 16; ++i) CUH(cudaEventCreate(&h->ev[i]));
    CUH(cudaGetLastError());
    CUH(cudaStreamSynchronize(h->stream));
#undef CUH
    *out = h;
    return UKFB_OK;
}

extern "C" int ukfb_create_sharded(int filter_kind, int64_t batch, const int* devices, int n_devices, ukfb_handle** out)
{
    if (!out) return fail(UKFB_ERR_INVALID, "ukfb_create_sharded: out is null");
    *out = nullptr;
    if (filter_kind != UKFB_POSE && filter_kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_create_sharded: bad filter kind %d", filter_kind);
    if (n_devices < 1 || n_devices > 64) return fail(UKFB_ERR_INVALID, "ukfb_create_sharded: n_devices must be 1..64");
    if (batch < n_devices) return fail(UKFB_ERR_INVALID, "ukfb_create_sharded: batch must be >= n_devices (every shard holds at least one filter)");
    ukfb_handle* h = new (std::nothrow) ukfb_handle;
    if (!h) return fail(UKFB_ERR_NOMEM, "ukfb_create_sharded: out of host memory");
    h->kind = filter_kind;
    h->B = batch;
    if (filter_kind == UKFB_POSE)
        h->n = PoseF::N, h->MU = PoseF::MU, h->LP = PoseF::LP, h->REC = PoseF::REC;
    else
        h->n = OriF::N, h->MU = OriF::MU, h->LP = OriF::LP, h->REC = OriF::REC;
    /* contiguous ranges, the first batch % n shards one filter longer (shard_range of the Python side) */
    const long long base = batch / n_devices, extra = batch % n_devices;
    h->first.assign(size_t(n_devices) + 1, 0);
    for (int i = 0; i < n_devices; ++i) h->first[size_t(i) + 1] = h->first[size_t(i)] + base + (i < extra ? 1 : 0);
    for (int i = 0; i < n_devices; ++i) {
        ukfb_handle* sh = nullptr;
        const int rc = ukfb_create(filter_kind, h->first[size_t(i) + 1] - h->first[size_t(i)], devices ? devices[i] : i, &sh);
        if (rc) {
            for (ukfb_handle* made : h->shards) ukfb_destroy(made);
            delete h;
            return rc; /* the text of ukfb_create stands */
        }
        h->shards.push_back(sh);
    }
    h->device = h->shards[0]->device;
    h->tiled = h->shards[0]->tiled, h->fast = h->shards[0]->fast;
    h->pool = new (std::nothrow) ShardPool(n_devices);
    if (!h->pool) {
        for (ukfb_handle* made : h->shards) ukfb_destroy(made);
        delete h;
        return fail(UKFB_ERR_NOMEM, "ukfb_create_sharded: out of host memory");
    }
    *out = h;
    return UKFB_OK;
}

extern "C" int ukfb_shard_count(const ukfb_handle* h) { return !h ? 0 : (is_sharded(h) ? int(h->shards.size()) : 1); }

extern "C" int ukfb_shard(ukfb_handle* h, int i, ukfb_handle** shard, int64_t* first, int64_t* count)
{
    if (!h) return fail(UKFB_ERR_INVALID, "ukfb_shard: null handle");
    const int n = ukfb_shard_count(h);
    if (i < 0 || i >= n) return fail(UKFB_ERR_INVALID, "ukfb_shard: shard %d out of range (%d shards)", i, n);
    if (shard) *shard = is_sharded(h) ? h->shards[size_t(i)] : h;
    if (first) *first = is_sharded(h) ? h->first[size_t(i)] : 0;
    if (count) *count = is_sharded(h) ? h->first[size_t(i) + 1] - h->first[size_t(i)] : h->B;
    return UKFB_OK;
}

extern "C" int ukfb_host_alloc(void** ptr, uint64_t bytes)
{
    if (!ptr || !bytes) return fail(UKFB_ERR_INVALID, "ukfb_host_alloc: bad argument");
    *ptr = nullptr;
    cudaError_t e = cudaHostAlloc(ptr, size_t(bytes), cudaHostAllocPortable);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? UKFB_ERR_NOMEM : UKFB_ERR_CUDA, "ukfb_host_alloc(%llu bytes): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return UKFB_OK;
}

extern "C" int ukfb_host_free(void* ptr)
{
    if (!ptr) return UKFB_OK;
    CU(cudaFreeHost(ptr));
    return UKFB_OK;
}

extern "C" int ukfb_destroy(ukfb_handle* h)
{
    if (!h) return UKFB_OK;
    if (is_sharded(h)) {
        delete h->pool; /* joins the workers (none is mid-call: the handle is single-caller) */
        for (ukfb_handle* s : h->shards) ukfb_destroy(s);
        delete h;
        return UKFB_OK;
    }
    Bind bind_(h);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->state), cudaFree(h->Q), cudaFree(h->status), cudaFree(h->t_last), cudaFree(h->hist), cudaFree(h->tile_done), cudaFree(h->tick_kinds_dev);
    cudaFree(h->acc_mu), cudaFree(h->acc_cov), cudaFree(h->gyro_mu), cudaFree(h->stage), cudaFree(h->summary), cudaFree(h->ori_params);
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) cudaFree(h->meas_cov[k]);
    for (int i = 0; i < 16; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->pipe.made) {
        cudaStreamSynchronize(h->pipe.s_in), cudaStreamSynchronize(h->pipe.s_out);
        for (int i = 0; i < 2; ++i) {
            cudaFree(h->pipe.in[i]), cudaFree(h->pipe.out[i]);
            cudaEventDestroy(h->pipe.in_ready[i]), cudaEventDestroy(h->pipe.in_consumed[i]);
            cudaEventDestroy(h->pipe.out_ready[i]), cudaEventDestroy(h->pipe.out_drained[i]);
        }
        cudaStreamDestroy(h->pipe.s_in), cudaStreamDestroy(h->pipe.s_out);
    }
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return UKFB_OK;
}

extern "C" int64_t ukfb_batch(const ukfb_handle* h) { return h ? h->B : 0; }
extern "C" int ukfb_dof(const ukfb_handle* h) { return h ? h->n : 0; }
extern "C" int ukfb_mu_size(const ukfb_handle* h) { return h ? h->MU : 0; }
extern "C" int ukfb_device(const ukfb_handle* h) { return h ? h->device : -1; }
extern "C" int ukfb_is_initialized(const ukfb_handle* h) { return h && h->initialized ? 1 : 0; } /* a sharded parent mirrors its shards */

static int initialize_dev(ukfb_handle* h, const double* d_mu, const double* d_sigma)
{
    pack_kernel<<<grid_for(h->B * h->REC), 256, 0, h->stream>>>(h->state, d_mu, d_sigma, h->B, h->n, h->MU, h->LP, h->REC, h->tiled);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(h->t_last, 0, sizeof(long long) * h->B, h->stream)); /* :43 */
    if (h->kind == UKFB_ORIENTATION && h->first_init) {
        ori_default_imu_kernel<<<grid_for(h->B), 256, 0, h->stream>>>(h->state, h->acc_mu, h->gyro_mu, h->B, h->tiled);
        CU(cudaGetLastError());
    }
    h->first_init = false;
    h->initialized = true;
    return UKFB_OK;
}

extern "C" int ukfb_initialize(ukfb_handle* h, const double* mu, const double* sigma)
{
    CHECK_H(h);
    if (!mu || !sigma) return fail(UKFB_ERR_INVALID, "ukfb_initialize: null argument");
    if (is_sharded(h)) {
        const int rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) { return ukfb_initialize(s_, mu + f_ * s_->MU, sigma + f_ * s_->n * s_->n); });
        if (rc == UKFB_OK) h->initialized = true;
        return rc;
    }
    const double *d_mu, *d_sigma;
    Staging st(h, false);
    st.in(&d_mu, mu, sizeof(double) * h->B * h->MU);
    st.in(&d_sigma, sigma, sizeof(double) * h->B * h->n * h->n);
    int rc = st.commit();
    if (!rc) rc = initialize_dev(h, d_mu, d_sigma);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_initialize_from_body_states_dev(ukfb_handle* h, const double* d_rbs)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (h->kind != UKFB_POSE) return fail(UKFB_ERR_INVALID, "ukfb_initialize_from_body_states: BodyStateMeasurement belongs to PoseUKF");
    if (!d_rbs) return fail(UKFB_ERR_INVALID, "ukfb_initialize_from_body_states: null argument");
    pack_rbs_kernel<<<grid_for(h->B * h->REC), 256, 0, h->stream>>>(h->state, d_rbs, h->B, h->tiled);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(h->t_last, 0, sizeof(long long) * h->B, h->stream)); /* initializeFilter, :43 */
    h->first_init = false;
    h->initialized = true;
    return UKFB_OK;
}

extern "C" int ukfb_initialize_from_body_states(ukfb_handle* h, const double* rbs)
{
    CHECK_H(h);
    if (!rbs) return fail(UKFB_ERR_INVALID, "ukfb_initialize_from_body_states: null argument");
    if (is_sharded(h)) {
        if (h->kind != UKFB_POSE) return fail(UKFB_ERR_INVALID, "ukfb_initialize_from_body_states: BodyStateMeasurement belongs to PoseUKF");
        const int rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) { return ukfb_initialize_from_body_states(s_, rbs + f_ * UKFB_RBS_DOUBLES); });
        if (rc == UKFB_OK) h->initialized = true;
        return rc;
    }
    const double* d_rbs;
    Staging st(h, false);
    st.in(&d_rbs, rbs, sizeof(double) * h->B * UKFB_RBS_DOUBLES);
    int rc = st.commit();
    if (!rc) rc = ukfb_initialize_from_body_states_dev(h, d_rbs);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_body_states_dev(ukfb_handle* h, double* d_rbs)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (h->kind != UKFB_POSE) return fail(UKFB_ERR_INVALID, "ukfb_get_body_states: BodyStateMeasurement belongs to PoseUKF");
    NEED_INIT(h);
    if (!d_rbs) return fail(UKFB_ERR_INVALID, "ukfb_get_body_states: null argument");
    unpack_rbs_kernel<<<grid_for(h->B * UKFB_RBS_DOUBLES), 256, 0, h->stream>>>(h->state, d_rbs, h->B, h->tiled);
    CU(cudaGetLastError());
    return UKFB_OK;
}

extern "C" int ukfb_get_body_states(ukfb_handle* h, double* rbs)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (!rbs) return fail(UKFB_ERR_INVALID, "ukfb_get_body_states: null argument");
    UKFB_FAN(h, ukfb_get_body_states(s_, rbs + f_ * UKFB_RBS_DOUBLES));
    double* d_rbs;
    Staging st(h, false);
    st.out(&d_rbs, rbs, sizeof(double) * h->B * UKFB_RBS_DOUBLES);
    int rc = st.commit();
    if (!rc) rc = ukfb_get_body_states_dev(h, d_rbs);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_state_dev(ukfb_handle* h, double* d_mu, double* d_sigma)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (d_mu) unpack_mu_kernel<<<grid_for(h->B * h->MU), 256, 0, h->stream>>>(h->state, d_mu, h->B, h->MU, h->REC, h->tiled);
    if (d_sigma) unpack_sigma_kernel<<<grid_for(h->B * h->n * h->n), 256, 0, h->stream>>>(h->state, d_sigma, h->B, h->n, h->MU, h->REC, h->tiled);
    CU(cudaGetLastError());
    return UKFB_OK;
}

/* ukfb_get_state / ukfb_get_state_async */
static int get_state_host(ukfb_handle* h, double* mu, double* sigma, bool pipelined, const char* who)
{
    CHECK_H_AS(h, who);
    NEED_INIT_AS(h, who);
    /* sharded: every shard lands in its range of the caller's single buffer -- the final gather of the estimates */
    UKFB_FAN(h, get_state_host(s_, mu ? mu + f_ * s_->MU : nullptr, sigma ? sigma + f_ * s_->n * s_->n : nullptr, pipelined, who));
    double *d_mu, *d_sigma;
    Staging st(h, pipelined);
    st.out(&d_mu, mu, sizeof(double) * h->B * h->MU);
    st.out(&d_sigma, sigma, sizeof(double) * h->B * h->n * h->n);
    int rc = st.commit();
    if (!rc) rc = ukfb_get_state_dev(h, d_mu, d_sigma);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_state(ukfb_handle* h, double* mu, double* sigma)
{
    return get_state_host(h, mu, sigma, false, "ukfb_get_state");
}

/* ukfb_get_state without the final synchronisation: the estimates of the steps issued so far are unpacked on the
 * compute stream into one of two staging slots and copied to the host on a copy-out stream, overlapping later
 * steps; mu / sigma are valid after ukfb_synchronize(). */
extern "C" int ukfb_get_state_async(ukfb_handle* h, double* mu, double* sigma)
{
    return get_state_host(h, mu, sigma, true, "ukfb_get_state_async");
}

/* mu entries [first, first + count) of every filter, dense B x count */
__global__ void unpack_mu_range_kernel(const double* __restrict__ state, double* __restrict__ out, long long B, int first, int count, int REC, int tiled)
{
    const long long total = B * count;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / count;
        const int k = int(i - b * count);
        out[i] = state[rec_index(tiled, b, first + k, REC)];
    }
}

static int mu_range_ok(const ukfb_handle* h, int mu_first, int mu_count, const void* out, const char* who)
{
    if (!out) return fail(UKFB_ERR_INVALID, "%s: null argument", who);
    if (mu_first < 0 || mu_count < 1 || mu_first + mu_count > h->MU)
        return fail(UKFB_ERR_INVALID, "%s: entries [%d, %d) are outside the %d-entry state", who, mu_first, mu_first + mu_count, h->MU);
    return UKFB_OK;
}

extern "C" int ukfb_get_mu_range_dev(ukfb_handle* h, int mu_first, int mu_count, double* d_out)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    const int rc = mu_range_ok(h, mu_first, mu_count, d_out, "ukfb_get_mu_range_dev");
    if (rc) return rc;
    unpack_mu_range_kernel<<<grid_for(h->B * mu_count), 256, 0, h->stream>>>(h->state, d_out, h->B, mu_first, mu_count, h->REC, h->tiled);
    CU(cudaGetLastError());
    return UKFB_OK;
}

/* ukfb_get_mu_range / ukfb_get_mu_range_async */
static int get_mu_range_host(ukfb_handle* h, int mu_first, int mu_count, double* out, bool pipelined, const char* who)
{
    CHECK_H_AS(h, who);
    NEED_INIT_AS(h, who);
    int rc = mu_range_ok(h, mu_first, mu_count, out, who);
    if (rc) return rc;
    UKFB_FAN(h, get_mu_range_host(s_, mu_first, mu_count, out + f_ * mu_count, pipelined, who));
    double* d_out;
    Staging st(h, pipelined);
    st.out(&d_out, out, sizeof(double) * h->B * mu_count);
    rc = st.commit();
    if (!rc) rc = ukfb_get_mu_range_dev(h, mu_first, mu_count, d_out);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_mu_range(ukfb_handle* h, int mu_first, int mu_count, double* out)
{
    return get_mu_range_host(h, mu_first, mu_count, out, false, "ukfb_get_mu_range");
}

extern "C" int ukfb_get_mu_range_async(ukfb_handle* h, int mu_first, int mu_count, double* out)
{
    return get_mu_range_host(h, mu_first, mu_count, out, true, "ukfb_get_mu_range_async");
}

/* StepParams::q_diagonal of a broadcast Q, from its packed lower triangle: 1 = no off-diagonal entry, 2 = that and one
 * value on the diagonal of each of the first two 3 x 3 blocks, 0 = neither.  ukfb_set_process_noise and the checkpoint
 * restore both classify with this, so that a restored handle takes the step kernels' path the saved one took. */
static int broadcast_q_class(const double* Qp, int n)
{
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < r; ++c)
            if (Qp[tri(r, c)] != 0.0) return 0;
    const double a = Qp[tri(0, 0)], b = Qp[tri(3, 3)];
    return a == Qp[tri(1, 1)] && a == Qp[tri(2, 2)] && b == Qp[tri(4, 4)] && b == Qp[tri(5, 5)] ? 2 : 1;
}

extern "C" int ukfb_set_process_noise(ukfb_handle* h, const double* Q, int per_filter)
{
    CHECK_H(h);
    if (!Q) return fail(UKFB_ERR_INVALID, "ukfb_set_process_noise: null argument");
    UKFB_FAN(h, ukfb_set_process_noise(s_, Q + (per_filter ? f_ * s_->n * s_->n : 0), per_filter));
    const long long count = per_filter ? h->B : 1;
    const double* d_Q;
    Staging st(h, false);
    st.in(&d_Q, Q, sizeof(double) * count * h->n * h->n);
    int rc = st.commit();
    if (rc) return rc;
    if ((per_filter != 0) != (h->q_per_filter != 0)) {
        CU(cudaStreamSynchronize(h->stream)); /* also completes the copy of Q queued above: a failure below leaves nothing reading Q */
        double* nq = nullptr;
        cudaError_t e = cudaMalloc(&nq, sizeof(double) * count * h->LP);
        if (e != cudaSuccess) return fail(UKFB_ERR_NOMEM, "ukfb_set_process_noise: %s", cudaGetErrorString(e));
        cudaFree(h->Q);
        h->Q = nq;
        h->q_per_filter = per_filter ? 1 : 0;
    }
    h->q_diagonal = 0;
    if (!per_filter) { /* the lower triangle is what pack_q_kernel keeps */
        double qp[OriF::LP];
        for (int r = 0; r < h->n; ++r)
            for (int c = 0; c <= r; ++c) qp[tri(r, c)] = Q[r * h->n + c];
        h->q_diagonal = broadcast_q_class(qp, h->n);
    }
    pack_q_kernel<<<grid_for(count * h->LP), 256, 0, h->stream>>>(h->Q, d_Q, count, h->n, h->LP);
    CU(cudaGetLastError());
    return st.finish();
}

extern "C" int ukfb_get_process_noise(ukfb_handle* h, double* Q, int per_filter)
{
    CHECK_H(h);
    if (!Q) return fail(UKFB_ERR_INVALID, "ukfb_get_process_noise: null argument");
    UKFB_FAN(h, (per_filter || f_ == 0) ? ukfb_get_process_noise(s_, Q + (per_filter ? f_ * s_->n * s_->n : 0), per_filter) : UKFB_OK);
    const long long count = per_filter ? h->B : 1;
    double* d_Q;
    Staging st(h, false);
    st.out(&d_Q, Q, sizeof(double) * count * h->n * h->n);
    int rc = st.commit();
    if (rc) return rc;
    unpack_q_kernel<<<grid_for(count * h->n * h->n), 256, 0, h->stream>>>(h->Q, d_Q, count, h->n, h->LP, h->q_per_filter ? h->LP : 0);
    CU(cudaGetLastError());
    return st.finish();
}

extern "C" int ukfb_set_time_bounds(ukfb_handle* h, double min_dt, double max_dt)
{
    if (!h) return fail(UKFB_ERR_INVALID, "ukfb_set_time_bounds: null handle");
    for (ukfb_handle* s : h->shards) s->min_dt = min_dt, s->max_dt = max_dt; /* host-side fields; the parent keeps a copy */
    h->min_dt = min_dt;
    h->max_dt = max_dt;
    return UKFB_OK;
}

extern "C" int ukfb_get_time_bounds(const ukfb_handle* h, double* min_dt, double* max_dt)
{
    if (!h) return fail(UKFB_ERR_INVALID, "ukfb_get_time_bounds: null handle");
    if (min_dt) *min_dt = h->min_dt;
    if (max_dt) *max_dt = h->max_dt;
    return UKFB_OK;
}

extern "C" int ukfb_set_last_time(ukfb_handle* h, const int64_t* ts_us, int per_filter)
{
    CHECK_H(h);
    if (!ts_us) return fail(UKFB_ERR_INVALID, "ukfb_set_last_time: null argument");
    UKFB_FAN(h, ukfb_set_last_time(s_, ts_us + (per_filter ? f_ : 0), per_filter));
    if (per_filter) {
        CU(cudaMemcpyAsync(h->t_last, ts_us, sizeof(long long) * h->B, cudaMemcpyHostToDevice, h->stream));
    } else {
        fill_kernel<long long><<<grid_for(h->B), 256, 0, h->stream>>>(h->t_last, h->B, (long long)ts_us[0]);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_get_last_time(ukfb_handle* h, int64_t* ts_us)
{
    CHECK_H(h);
    if (!ts_us) return fail(UKFB_ERR_INVALID, "ukfb_get_last_time: null argument");
    UKFB_FAN(h, ukfb_get_last_time(s_, ts_us + f_));
    CU(cudaMemcpyAsync(ts_us, h->t_last, sizeof(long long) * h->B, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_set_mahalanobis_gate(ukfb_handle* h, double max_d2)
{
    CHECK_H(h);
    if (!(max_d2 > 0.0)) return fail(UKFB_ERR_INVALID, "ukfb_set_mahalanobis_gate: the threshold must be positive (+inf accepts everything)");
    for (ukfb_handle* s : h->shards) s->gate_d2 = max_d2;
    h->gate_d2 = max_d2;
    return UKFB_OK;
}

extern "C" int ukfb_get_mahalanobis_gate(const ukfb_handle* h, double* max_d2)
{
    if (!h || !max_d2) return fail(UKFB_ERR_INVALID, "ukfb_get_mahalanobis_gate: null argument");
    *max_d2 = h->gate_d2;
    return UKFB_OK;
}

extern "C" int ukfb_set_orientation_params(ukfb_handle* h, double gyro_bias_tau, double acc_bias_tau, double latitude)
{
    if (!h) return fail(UKFB_ERR_INVALID, "ukfb_set_orientation_params: null handle");
    if (h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_set_orientation_params: not an ORIENTATION handle");
    for (ukfb_handle* s : h->shards) {
        const int rc = ukfb_set_orientation_params(s, gyro_bias_tau, acc_bias_tau, latitude);
        if (rc) return rc;
    }
    h->tau_g = gyro_bias_tau;
    h->tau_a = acc_bias_tau;
    h->latitude = latitude;
    h->earth[0] = UKFB_EARTHW * cos(latitude);
    h->earth[1] = 0.0;
    h->earth[2] = UKFB_EARTHW * sin(latitude);
    if (h->ori_params) { /* back to one parameter set for all filters */
        Bind bind_(h);
        cudaStreamSynchronize(h->stream);
        cudaFree(h->ori_params);
        h->ori_params = nullptr;
    }
    return UKFB_OK;
}

extern "C" int ukfb_set_orientation_params_per_filter(ukfb_handle* h, const double* gyro_bias_tau, const double* acc_bias_tau,
                                                      const double* latitude)
{
    CHECK_H(h);
    if (h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_set_orientation_params_per_filter: not an ORIENTATION handle");
    if (!gyro_bias_tau || !acc_bias_tau || !latitude) return fail(UKFB_ERR_INVALID, "ukfb_set_orientation_params_per_filter: null argument");
    UKFB_FAN(h, ukfb_set_orientation_params_per_filter(s_, gyro_bias_tau + f_, acc_bias_tau + f_, latitude + f_));
    std::vector<double> packed(size_t(h->B) * 5);
    for (long long b = 0; b < h->B; ++b) {
        packed[b * 5] = -1.0 / gyro_bias_tau[b];
        packed[b * 5 + 1] = -1.0 / acc_bias_tau[b];
        packed[b * 5 + 2] = UKFB_EARTHW * cos(latitude[b]);
        packed[b * 5 + 3] = 0.0;
        packed[b * 5 + 4] = UKFB_EARTHW * sin(latitude[b]);
    }
    if (!h->ori_params) {
        cudaError_t e = cudaMalloc(&h->ori_params, sizeof(double) * h->B * 5);
        if (e != cudaSuccess) return fail(UKFB_ERR_NOMEM, "ukfb_set_orientation_params_per_filter: %s", cudaGetErrorString(e));
    }
    CU(cudaMemcpyAsync(h->ori_params, packed.data(), sizeof(double) * h->B * 5, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return UKFB_OK;
}

/* ---- predict --------------------------------------------------------------------------------------- */
extern "C" int ukfb_predict_dt_dev(ukfb_handle* h, const double* d_dt, int per_filter)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (!d_dt) return fail(UKFB_ERR_INVALID, "ukfb_predict_dt: null argument");
    StepParams p = base_params(h);
    p.do_predict = 1;
    p.time_mode = 0;
    p.dt = d_dt;
    p.dt_stride = per_filter ? 1 : 0;
    return launch_step(h, p);
}

extern "C" int ukfb_predict_dt(ukfb_handle* h, const double* dt, int per_filter)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (!dt) return fail(UKFB_ERR_INVALID, "ukfb_predict_dt: null argument");
    UKFB_FAN(h, ukfb_predict_dt(s_, dt + (per_filter ? f_ : 0), per_filter));
    const double* d_dt;
    Staging st(h, false);
    st.in(&d_dt, dt, sizeof(double) * (per_filter ? h->B : 1));
    int rc = st.commit();
    if (!rc) rc = ukfb_predict_dt_dev(h, d_dt, per_filter);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_predict_time_dev(ukfb_handle* h, const int64_t* d_ts_us, int per_filter)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (!d_ts_us) return fail(UKFB_ERR_INVALID, "ukfb_predict_time: null argument");
    StepParams p = base_params(h);
    p.do_predict = 1;
    p.time_mode = 1;
    p.ts = reinterpret_cast<const long long*>(d_ts_us);
    p.ts_stride = per_filter ? 1 : 0;
    return launch_step(h, p);
}

extern "C" int ukfb_predict_time(ukfb_handle* h, const int64_t* ts_us, int per_filter)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (!ts_us) return fail(UKFB_ERR_INVALID, "ukfb_predict_time: null argument");
    UKFB_FAN(h, ukfb_predict_time(s_, ts_us + (per_filter ? f_ : 0), per_filter));
    const int64_t* d_ts;
    Staging st(h, false);
    st.in(&d_ts, ts_us, sizeof(int64_t) * (per_filter ? h->B : 1));
    int rc = st.commit();
    if (!rc) rc = ukfb_predict_time_dev(h, d_ts, per_filter);
    return rc ? rc : st.finish();
}

/* ---- measurements ------------------------------------------------------------------------------------ */
extern "C" int ukfb_meas_dim(int meas_kind)
{
    if (meas_kind < 0 || meas_kind >= UKFB_MEAS_KIND_COUNT) return 0;
    return meas_dim(meas_kind);
}

static void set_update(StepParams& p, int kind, const double* d_mu, const double* d_cov, int cov_per_filter, const uint8_t* d_mask)
{
    const int m = meas_dim(kind);
    p.do_update = 1;
    p.kind = kind;
    p.z = d_mu;
    p.z_stride = m;
    p.R = d_cov;
    p.r_stride = cov_per_filter ? m * m : 0;
    p.r_ld = m;
    p.mask = d_mask;
}

extern "C" int ukfb_update_dev(ukfb_handle* h, int meas_kind, const double* d_mu, const double* d_cov, int cov_per_filter,
                               const uint8_t* d_mask)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (!kind_ok(h, meas_kind)) return fail(UKFB_ERR_INVALID, "ukfb_update: measurement kind %d does not belong to this filter kind", meas_kind);
    if (!d_mu || !d_cov) return fail(UKFB_ERR_INVALID, "ukfb_update: null argument");
    StepParams p = base_params(h);
    set_update(p, meas_kind, d_mu, d_cov, cov_per_filter, d_mask);
    return launch_step(h, p);
}

extern "C" int ukfb_update(ukfb_handle* h, int meas_kind, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (!kind_ok(h, meas_kind)) return fail(UKFB_ERR_INVALID, "ukfb_update: measurement kind %d does not belong to this filter kind", meas_kind);
    if (!mu) return fail(UKFB_ERR_INVALID, "ukfb_update: null argument");
    if (!cov && !h->meas_cov_per_filter[meas_kind]) return fail(UKFB_ERR_INVALID, "ukfb_update: null covariance and none kept by ukfb_set_measurement_cov for kind %d", meas_kind);
    const int m = meas_dim(meas_kind);
    UKFB_FAN(h, ukfb_update(s_, meas_kind, mu + f_ * m, cov ? cov + (cov_per_filter ? f_ * m * m : 0) : nullptr, cov_per_filter, mask ? mask + f_ : nullptr));
    const double *d_mu, *d_cov;
    const uint8_t* d_mask;
    Staging st(h, false);
    st.in(&d_mu, mu, sizeof(double) * h->B * m);
    st.in(&d_cov, cov, sizeof(double) * (cov_per_filter ? h->B : 1) * m * m);
    st.in(&d_mask, mask, size_t(h->B));
    int rc = st.commit();
    if (rc) return rc;
    if (!cov) d_cov = h->meas_cov[meas_kind], cov_per_filter = h->meas_cov_per_filter[meas_kind] == 2;
    rc = ukfb_update_dev(h, meas_kind, d_mu, d_cov, cov_per_filter, d_mask);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_set_measurement_cov(ukfb_handle* h, int meas_kind, const double* cov, int per_filter)
{
    CHECK_H(h);
    if (!kind_ok(h, meas_kind)) return fail(UKFB_ERR_INVALID, "ukfb_set_measurement_cov: measurement kind %d does not belong to this filter kind", meas_kind);
    if (!cov) return fail(UKFB_ERR_INVALID, "ukfb_set_measurement_cov: null argument");
    const int m = meas_dim(meas_kind);
    if (is_sharded(h)) {
        const int rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) { return ukfb_set_measurement_cov(s_, meas_kind, cov + (per_filter ? f_ * m * m : 0), per_filter); });
        if (rc == UKFB_OK) h->meas_cov_per_filter[meas_kind] = per_filter ? 2 : 1; /* the parent only remembers that one is kept */
        return rc;
    }
    const size_t bytes = sizeof(double) * size_t(per_filter ? h->B : 1) * m * m;
    CU(cudaStreamSynchronize(h->stream));
    if (h->meas_cov[meas_kind]) CU(cudaFree(h->meas_cov[meas_kind]));
    h->meas_cov[meas_kind] = nullptr;
    cudaError_t e = cudaMalloc(&h->meas_cov[meas_kind], bytes);
    if (e != cudaSuccess) return fail(UKFB_ERR_NOMEM, "ukfb_set_measurement_cov: %s", cudaGetErrorString(e));
    h->meas_cov_per_filter[meas_kind] = per_filter ? 2 : 1;
    CU(cudaMemcpyAsync(h->meas_cov[meas_kind], cov, bytes, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_update_mixed_dev(ukfb_handle* h, const int8_t* d_kinds, const double* d_mu3, const double* d_cov33)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (!d_kinds || !d_mu3 || !d_cov33) return fail(UKFB_ERR_INVALID, "ukfb_update_mixed: null argument");
    StepParams p = base_params(h);
    p.do_update = 1;
    p.kind = -2;
    p.kinds = d_kinds;
    p.z = d_mu3;
    p.z_stride = 3;
    p.R = d_cov33;
    p.r_stride = 9;
    p.r_ld = 3;
    return launch_step(h, p);
}

extern "C" int ukfb_update_mixed(ukfb_handle* h, const int8_t* kinds, const double* mu3, const double* cov33)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (!kinds || !mu3 || !cov33) return fail(UKFB_ERR_INVALID, "ukfb_update_mixed: null argument");
    /* a kind of the other filter family is an API error, as calling a non-existent overload would be */
    for (long long b = 0; b < h->B; ++b)
        if (kinds[b] != UKFB_MEAS_NONE && !kind_ok(h, kinds[b]))
            return fail(UKFB_ERR_INVALID, "ukfb_update_mixed: kinds[%lld] = %d does not belong to this filter kind", b, int(kinds[b]));
    UKFB_FAN(h, ukfb_update_mixed(s_, kinds + f_, mu3 + f_ * 3, cov33 + f_ * 9));
    const int8_t* d_kinds;
    const double *d_mu3, *d_cov33;
    Staging st(h, false);
    st.in(&d_kinds, kinds, size_t(h->B));
    st.in(&d_mu3, mu3, sizeof(double) * h->B * 3);
    st.in(&d_cov33, cov33, sizeof(double) * h->B * 9);
    int rc = st.commit();
    if (!rc) rc = ukfb_update_mixed_dev(h, d_kinds, d_mu3, d_cov33);
    return rc ? rc : st.finish();
}

static int store_vec3_dev(ukfb_handle* h, double* dst_mu, double* dst_cov, const double* d_mu, const double* d_cov, int cov_per_filter,
                          const uint8_t* d_mask, int check)
{
    store_vec3_kernel<<<grid_for(h->B), 256, 0, h->stream>>>(dst_mu, dst_cov, d_mu, d_cov, cov_per_filter ? 9 : 0, d_mask, h->status, check, h->B);
    CU(cudaGetLastError());
    return UKFB_OK;
}

extern "C" int ukfb_set_acceleration_dev(ukfb_handle* h, const double* d_mu, const double* d_cov, int cov_per_filter, const uint8_t* d_mask)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (!d_mu) return fail(UKFB_ERR_INVALID, "ukfb_set_acceleration: null argument");
    /* PoseUKF stores unchecked (PoseUKF.cpp:175-178); OrientationUKF checks (OrientationUKF.cpp:61) */
    return store_vec3_dev(h, h->acc_mu, h->acc_cov, d_mu, d_cov, cov_per_filter, d_mask, h->kind == UKFB_ORIENTATION);
}

extern "C" int ukfb_set_acceleration(ukfb_handle* h, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    CHECK_H(h);
    if (!mu) return fail(UKFB_ERR_INVALID, "ukfb_set_acceleration: null argument");
    UKFB_FAN(h, ukfb_set_acceleration(s_, mu + f_ * 3, cov ? cov + (cov_per_filter ? f_ * 9 : 0) : nullptr, cov_per_filter, mask ? mask + f_ : nullptr));
    const double *d_mu, *d_cov;
    const uint8_t* d_mask;
    Staging st(h, false);
    st.in(&d_mu, mu, sizeof(double) * h->B * 3);
    st.in(&d_cov, cov, sizeof(double) * (cov_per_filter ? h->B : 1) * 9);
    st.in(&d_mask, mask, size_t(h->B));
    int rc = st.commit();
    if (!rc) rc = ukfb_set_acceleration_dev(h, d_mu, d_cov, cov_per_filter, d_mask);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_set_rotation_rate_dev(ukfb_handle* h, const double* d_mu, const double* d_cov, int cov_per_filter, const uint8_t* d_mask)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_set_rotation_rate: not an ORIENTATION handle");
    if (!d_mu) return fail(UKFB_ERR_INVALID, "ukfb_set_rotation_rate: null argument");
    /* the rotation-rate covariance is never read by the reference (OrientationUKF.cpp:88 passes .mu only) but
     * checkMeasurment still inspects it */
    return store_vec3_dev(h, h->gyro_mu, nullptr, d_mu, d_cov, cov_per_filter, d_mask, 1);
}

extern "C" int ukfb_set_rotation_rate(ukfb_handle* h, const double* mu, const double* cov, int cov_per_filter, const uint8_t* mask)
{
    CHECK_H(h);
    if (h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_set_rotation_rate: not an ORIENTATION handle");
    if (!mu) return fail(UKFB_ERR_INVALID, "ukfb_set_rotation_rate: null argument");
    UKFB_FAN(h, ukfb_set_rotation_rate(s_, mu + f_ * 3, cov ? cov + (cov_per_filter ? f_ * 9 : 0) : nullptr, cov_per_filter, mask ? mask + f_ : nullptr));
    const double *d_mu, *d_cov;
    const uint8_t* d_mask;
    Staging st(h, false);
    st.in(&d_mu, mu, sizeof(double) * h->B * 3);
    st.in(&d_cov, cov, sizeof(double) * (cov_per_filter ? h->B : 1) * 9);
    st.in(&d_mask, mask, size_t(h->B));
    int rc = st.commit();
    if (!rc) rc = ukfb_set_rotation_rate_dev(h, d_mu, d_cov, cov_per_filter, d_mask);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_rotation_rate(ukfb_handle* h, double* out)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_get_rotation_rate: not an ORIENTATION handle");
    if (!out) return fail(UKFB_ERR_INVALID, "ukfb_get_rotation_rate: null argument");
    UKFB_FAN(h, ukfb_get_rotation_rate(s_, out + f_ * 3));
    double* d_out;
    Staging st(h, false);
    st.out(&d_out, out, sizeof(double) * h->B * 3);
    int rc = st.commit();
    if (rc) return rc;
    rotation_rate_kernel<<<grid_for(h->B), 256, 0, h->stream>>>(h->state, h->gyro_mu, h->earth[0], h->earth[1], h->earth[2], h->ori_params,
                                                               d_out, h->B, h->tiled);
    CU(cudaGetLastError());
    return st.finish();
}

/* ---- fused step ------------------------------------------------------------------------------------------ */
extern "C" int ukfb_step_dev(ukfb_handle* h, const double* d_dt, int dt_per_filter, int meas_kind, const double* d_mu, const double* d_cov,
                             int cov_per_filter, const uint8_t* d_mask)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (!d_dt) return fail(UKFB_ERR_INVALID, "ukfb_step: null dt");
    StepParams p = base_params(h);
    p.do_predict = 1;
    p.dt = d_dt;
    p.dt_stride = dt_per_filter ? 1 : 0;
    if (meas_kind != UKFB_MEAS_NONE) {
        if (!kind_ok(h, meas_kind)) return fail(UKFB_ERR_INVALID, "ukfb_step: measurement kind %d does not belong to this filter kind", meas_kind);
        if (!d_mu || !d_cov) return fail(UKFB_ERR_INVALID, "ukfb_step: null measurement");
        set_update(p, meas_kind, d_mu, d_cov, cov_per_filter, d_mask);
    }
    return launch_step(h, p);
}

/* ukfb_step / ukfb_step_async */
static int step_host(ukfb_handle* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu, const double* cov,
                     int cov_per_filter, const uint8_t* mask, bool pipelined, const char* who)
{
    CHECK_H_AS(h, who);
    NEED_INIT_AS(h, who);
    if (!dt) return fail(UKFB_ERR_INVALID, "%s: null dt", who);
    const bool upd = meas_kind != UKFB_MEAS_NONE;
    if (upd && !kind_ok(h, meas_kind)) return fail(UKFB_ERR_INVALID, "%s: measurement kind %d does not belong to this filter kind", who, meas_kind);
    if (upd && !mu) return fail(UKFB_ERR_INVALID, "%s: null measurement", who);
    if (upd && !cov && !h->meas_cov_per_filter[meas_kind])
        return fail(UKFB_ERR_INVALID, "%s: null covariance and none kept by ukfb_set_measurement_cov for kind %d", who, meas_kind);
    const int m = upd ? meas_dim(meas_kind) : 0;
    UKFB_FAN(h, step_host(s_, dt + (dt_per_filter ? f_ : 0), dt_per_filter, meas_kind, mu ? mu + f_ * m : nullptr,
                          cov ? cov + (cov_per_filter ? f_ * m * m : 0) : nullptr, cov_per_filter, mask ? mask + f_ : nullptr, pipelined, who));
    const double *d_dt, *d_mu = nullptr, *d_cov = nullptr;
    const uint8_t* d_mask = nullptr;
    Staging st(h, pipelined);
    st.in(&d_dt, dt, sizeof(double) * (dt_per_filter ? h->B : 1));
    if (upd) {
        st.in(&d_mu, mu, sizeof(double) * h->B * m);
        st.in(&d_cov, cov, sizeof(double) * (cov_per_filter ? h->B : 1) * m * m);
        st.in(&d_mask, mask, size_t(h->B));
    }
    int rc = st.commit();
    if (rc) return rc;
    if (upd && !cov) d_cov = h->meas_cov[meas_kind], cov_per_filter = h->meas_cov_per_filter[meas_kind] == 2;
    rc = ukfb_step_dev(h, d_dt, dt_per_filter, meas_kind, d_mu, d_cov, cov_per_filter, d_mask);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_step(ukfb_handle* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu, const double* cov,
                         int cov_per_filter, const uint8_t* mask)
{
    return step_host(h, dt, dt_per_filter, meas_kind, mu, cov, cov_per_filter, mask, false, "ukfb_step");
}

/* ukfb_step without the final synchronisation: the inputs are copied on a copy-in stream into one of two staging
 * slots while the previous step's kernel runs; the host arrays must stay valid and unchanged until
 * ukfb_synchronize() (or until two further ukfb_step_async calls have been issued and the first has been waited
 * for); pinned host memory makes the copies truly asynchronous. */
extern "C" int ukfb_step_async(ukfb_handle* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu, const double* cov,
                               int cov_per_filter, const uint8_t* mask)
{
    return step_host(h, dt, dt_per_filter, meas_kind, mu, cov, cov_per_filter, mask, true, "ukfb_step_async");
}

extern "C" int ukfb_run_dev(ukfb_handle* h, int K, const double* d_dt, int dt_per_filter, const int8_t* kinds_host, const double* d_mu3,
                            const double* d_cov33, int cov_per_filter, const double* d_imu)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (K < 1) return fail(UKFB_ERR_INVALID, "ukfb_run: K must be >= 1");
    if (!d_dt) return fail(UKFB_ERR_INVALID, "ukfb_run: null dt");
    bool any = false, has_ori = false;
    if (kinds_host)
        for (int k = 0; k < K; ++k) {
            if (kinds_host[k] == UKFB_MEAS_NONE) continue;
            if (!kind_ok(h, kinds_host[k])) return fail(UKFB_ERR_INVALID, "ukfb_run: kinds[%d] = %d does not belong to this filter kind", k, int(kinds_host[k]));
            any = true;
            if (h->kind == UKFB_POSE && kinds_host[k] == UKFB_MEAS_POSE_ORIENTATION) has_ori = true;
        }
    h->tick_kinds_have_orientation = has_ori;
    if (any && (!d_mu3 || !d_cov33)) return fail(UKFB_ERR_INVALID, "ukfb_run: null measurement stream");
    if (d_imu && h->kind != UKFB_ORIENTATION) return fail(UKFB_ERR_INVALID, "ukfb_run: imu stream on a POSE handle");
    StepParams p = base_params(h);
    p.K = K;
    p.do_predict = 1;
    p.dt = d_dt;
    p.dt_stride = dt_per_filter ? 1 : 0;
    p.dt_kstride = dt_per_filter ? h->B : 1;
    if (any) {
        /* the K tick kinds ride in a small device array of the handle, rewritten only when the schedule changes */
        if (h->tick_kinds_cap < size_t(K)) {
            CU(cudaStreamSynchronize(h->stream));
            if (h->tick_kinds_dev) CU(cudaFree(h->tick_kinds_dev));
            h->tick_kinds_dev = nullptr, h->tick_kinds_cap = 0;
            h->tick_kinds_last.clear();
            const size_t want = align256(size_t(K));
            cudaError_t e = cudaMalloc(&h->tick_kinds_dev, want);
            if (e != cudaSuccess) return fail(UKFB_ERR_NOMEM, "tick kinds of %zu bytes: %s", want, cudaGetErrorString(e));
            h->tick_kinds_cap = want;
        }
        if (h->tick_kinds_last.size() != size_t(K) || memcmp(h->tick_kinds_last.data(), kinds_host, size_t(K)) != 0) {
            h->tick_kinds_last.assign(kinds_host, kinds_host + K);
            /* from the handle's own copy: it stays unchanged until the next call replaces it, after this copy in stream order */
            CU(cudaMemcpyAsync(h->tick_kinds_dev, h->tick_kinds_last.data(), size_t(K), cudaMemcpyHostToDevice, h->stream));
        }
        p.do_update = 1;
        p.tick_kinds = h->tick_kinds_dev;
        p.z = d_mu3;
        p.z_stride = 3;
        p.z_kstride = h->B * 3;
        p.R = d_cov33;
        p.r_stride = cov_per_filter ? 9 : 0;
        p.r_kstride = cov_per_filter ? h->B * 9 : 9;
        p.r_ld = 3;
    }
    p.imu = d_imu;
    p.imu_kstride = h->B * 6;
    return launch_step(h, p);
}

/* ---- event streams --------------------------------------------------------------------------------------- */
extern "C" int ukfb_run_events_dev(ukfb_handle* h, int K, const int64_t* d_ts_us, const int8_t* d_kinds, const double* d_mu3,
                                   const double* d_cov, int cov_mode)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    if (K < 1) return fail(UKFB_ERR_INVALID, "ukfb_run_events: K must be >= 1");
    if (!d_ts_us || !d_kinds || !d_mu3 || !d_cov) return fail(UKFB_ERR_INVALID, "ukfb_run_events: null argument");
    if (cov_mode != 0 && cov_mode != 1) return fail(UKFB_ERR_INVALID, "ukfb_run_events: cov_mode must be 0 (per-kind table) or 1 (per event)");
    StepParams p = base_params(h);
    p.K = K;
    p.events = 1;
    p.do_predict = 1;
    p.time_mode = 1;
    p.ts = reinterpret_cast<const long long*>(d_ts_us);
    p.ts_stride = 1;
    p.ts_kstride = h->B;
    p.do_update = 1;
    p.kind = -2;
    p.kinds = d_kinds;
    p.kinds_kstride = h->B;
    p.z = d_mu3;
    p.z_stride = 3;
    p.z_kstride = h->B * 3;
    p.R = d_cov;
    p.r_ld = 3;
    p.r_stride = cov_mode ? 9 : 0;
    p.r_kstride = cov_mode ? h->B * 9 : 0;
    p.r_kind_stride = cov_mode ? 0 : 9;
    return launch_step(h, p);
}

/* ukfb_run_events / ukfb_run_events_async on one device.  The arrays point at this handle's first filter in slot 0 and
 * their slots are src_B filters apart (src_B = h->B for a one-device handle, the parent's batch for a shard). */
static int run_events_host(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3, const double* cov,
                           int cov_mode, long long src_B, bool async)
{
    CHECK_H(h);
    NEED_INIT(h);
    const size_t B = size_t(h->B), pitch = size_t(src_B), rows = size_t(K);
    const int64_t* d_ts;
    const int8_t* d_kinds;
    const double *d_mu3, *d_cov;
    Staging st(h, async);
    st.in_rows(&d_ts, ts_us, sizeof(int64_t) * B, rows, sizeof(int64_t) * pitch);
    st.in_rows(&d_kinds, kinds, B, rows, pitch);
    st.in_rows(&d_mu3, mu3, sizeof(double) * 3 * B, rows, sizeof(double) * 3 * pitch);
    if (cov_mode)
        st.in_rows(&d_cov, cov, sizeof(double) * 9 * B, rows, sizeof(double) * 9 * pitch);
    else
        st.in(&d_cov, cov, sizeof(double) * UKFB_EVENT_KIND_COUNT * 9);
    int rc = st.commit();
    if (!rc) rc = ukfb_run_events_dev(h, K, d_ts, d_kinds, d_mu3, d_cov, cov_mode);
    return rc ? rc : st.finish();
}

static int run_events_any(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3, const double* cov,
                          int cov_mode, bool async, const char* who)
{
    CHECK_H(h);
    NEED_INIT(h);
    if (K < 1) return fail(UKFB_ERR_INVALID, "%s: K must be >= 1", who);
    if (!ts_us || !kinds || !mu3 || !cov) return fail(UKFB_ERR_INVALID, "%s: null argument", who);
    if (cov_mode != 0 && cov_mode != 1) return fail(UKFB_ERR_INVALID, "%s: cov_mode must be 0 (per-kind table) or 1 (per event)", who);
    const long long B = h->B;
    UKFB_FAN(h, run_events_host(s_, K, ts_us + f_, kinds + f_, mu3 + f_ * 3, cov_mode ? cov + f_ * 9 : cov, cov_mode, B, async));
    return run_events_host(h, K, ts_us, kinds, mu3, cov, cov_mode, B, async);
}

extern "C" int ukfb_run_events(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3, const double* cov,
                               int cov_mode)
{
    return run_events_any(h, K, ts_us, kinds, mu3, cov, cov_mode, false, "ukfb_run_events");
}

/* ukfb_run_events without the final synchronisation: the queues travel on the copy-in stream into one of the two
 * staging slots while the previous launch runs (same slots and rules as ukfb_step_async) */
extern "C" int ukfb_run_events_async(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3,
                                     const double* cov, int cov_mode)
{
    return run_events_any(h, K, ts_us, kinds, mu3, cov, cov_mode, true, "ukfb_run_events_async");
}

/* ---- status ------------------------------------------------------------------------------------------------ */
extern "C" int ukfb_get_status(ukfb_handle* h, uint32_t* flags)
{
    CHECK_H(h);
    if (!flags) return fail(UKFB_ERR_INVALID, "ukfb_get_status: null argument");
    UKFB_FAN(h, ukfb_get_status(s_, flags + f_));
    CU(cudaMemcpyAsync(flags, h->status, sizeof(uint32_t) * h->B, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_clear_status(ukfb_handle* h)
{
    CHECK_H(h);
    UKFB_FAN(h, ukfb_clear_status(s_));
    CU(cudaMemsetAsync(h->status, 0, sizeof(uint32_t) * h->B, h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_status_summary(ukfb_handle* h, int64_t* n_flagged, uint32_t* any_bits)
{
    CHECK_H(h);
    if (is_sharded(h)) {
        std::vector<int64_t> n(h->shards.size(), 0);
        std::vector<uint32_t> bits(h->shards.size(), 0u);
        const int rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) {
            size_t i = 0;
            while (h->first[i] != f_) ++i; /* the shard whose range starts at f_ (every shard holds >= 1 filter) */
            return ukfb_status_summary(s_, &n[i], &bits[i]);
        });
        if (rc) return rc;
        int64_t nt = 0;
        uint32_t bt = 0;
        for (size_t i = 0; i < n.size(); ++i) nt += n[i], bt |= bits[i];
        if (n_flagged) *n_flagged = nt;
        if (any_bits) *any_bits = bt;
        return UKFB_OK;
    }
    CU(cudaMemsetAsync(h->summary, 0, sizeof(long long) * 2, h->stream));
    status_summary_kernel<<<grid_for(h->B), 256, 0, h->stream>>>(h->status, h->B, h->summary);
    CU(cudaGetLastError());
    long long out[2] = {0, 0};
    CU(cudaMemcpyAsync(out, h->summary, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (n_flagged) *n_flagged = out[0];
    if (any_bits) *any_bits = uint32_t(out[1]);
    return UKFB_OK;
}

extern "C" int ukfb_get_mean_iter_hist(ukfb_handle* h, uint64_t hist[8])
{
    CHECK_H(h);
    if (!hist) return fail(UKFB_ERR_INVALID, "ukfb_get_mean_iter_hist: null argument");
    if (is_sharded(h)) {
        for (int k = 0; k < 8; ++k) hist[k] = 0;
        for (ukfb_handle* s : h->shards) {
            uint64_t one[8];
            const int rc = ukfb_get_mean_iter_hist(s, one);
            if (rc) return rc;
            for (int k = 0; k < 8; ++k) hist[k] += one[k];
        }
        return UKFB_OK;
    }
    unsigned long long tmp[HIST_SLOTS * 8];
    CU(cudaMemcpyAsync(tmp, h->hist, sizeof(tmp), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < 8; ++k) hist[k] = 0;
    for (int s = 0; s < HIST_SLOTS; ++s)
        for (int k = 0; k < 8; ++k) hist[k] += tmp[s * 8 + k];
    return UKFB_OK;
}

extern "C" int ukfb_clear_mean_iter_hist(ukfb_handle* h)
{
    CHECK_H(h);
    UKFB_FAN(h, ukfb_clear_mean_iter_hist(s_));
    CU(cudaMemsetAsync(h->hist, 0, sizeof(unsigned long long) * HIST_SLOTS * 8, h->stream));
    return UKFB_OK;
}

/* ---- per-filter access (kernels: ukf_index.cuh) ------------------------------------------------------------------ */
static IndexParams index_params(const ukfb_handle* h, long long n_rows, const long long* d_idx)
{
    IndexParams p{};
    p.state = h->state;
    p.B = h->B;
    p.MU = h->MU, p.n = h->n, p.REC = h->REC, p.tiled = h->tiled;
    p.idx = d_idx;
    p.n_rows = n_rows;
    p.t_last = h->t_last;
    p.status = h->status;
    return p;
}

/* the checks of every host-pointer call, before anything is enqueued: indices in [0, B), unique when asked */
static int check_indices(const ukfb_handle* h, int64_t n, const int64_t* idx, bool unique, const char* who)
{
    for (int64_t k = 0; k < n; ++k)
        if (idx[k] < 0 || idx[k] >= h->B)
            return fail(UKFB_ERR_INVALID, "%s: idx[%lld] = %lld is outside [0, %lld)", who, (long long)k, (long long)idx[k], h->B);
    if (unique && n > 1) {
        try {
            std::vector<int64_t> s(idx, idx + n);
            std::sort(s.begin(), s.end());
            const auto d = std::adjacent_find(s.begin(), s.end());
            if (d != s.end()) return fail(UKFB_ERR_INVALID, "%s: filter %lld is listed twice", who, (long long)*d);
        } catch (const std::bad_alloc&) {
            return fail(UKFB_ERR_NOMEM, "%s: out of host memory", who);
        }
    }
    return UKFB_OK;
}

/* a sharded parent's index list split by shard: local indices and the caller's row of each, in the caller's order.
 * Throws std::bad_alloc. */
struct ShardRows {
    std::vector<std::vector<int64_t>> local, pos;
    ShardRows(const ukfb_handle* h, int64_t n, const int64_t* idx) : local(h->shards.size()), pos(h->shards.size())
    {
        for (int64_t k = 0; k < n; ++k) {
            const size_t s = size_t(std::upper_bound(h->first.begin(), h->first.end(), (long long)idx[k]) - h->first.begin()) - 1;
            local[s].push_back(idx[k] - h->first[s]);
            pos[s].push_back(k);
        }
    }
};

/* the shard whose range starts at filter f (every shard holds at least one filter) */
static size_t shard_at(const ukfb_handle* h, long long f)
{
    size_t i = 0;
    while (h->first[i] != f) ++i;
    return i;
}

static int get_state_indexed_launch(ukfb_handle* h, long long n, const long long* d_idx, double* d_mu, double* d_sigma)
{
    IndexParams p = index_params(h, n, d_idx);
    p.mu = d_mu, p.sigma = d_sigma;
    get_state_indexed_kernel<<<grid_for(n * (d_sigma ? h->n * h->n : h->MU)), 256, 0, h->stream>>>(p);
    CU(cudaGetLastError());
    return UKFB_OK;
}

extern "C" int ukfb_get_state_indexed_dev(ukfb_handle* h, int64_t n, const int64_t* d_idx, double* d_mu, double* d_sigma)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (n < 0) return fail(UKFB_ERR_INVALID, "ukfb_get_state_indexed_dev: n is negative");
    if (n == 0) return UKFB_OK;
    if (!d_idx || !d_mu) return fail(UKFB_ERR_INVALID, "ukfb_get_state_indexed_dev: null argument");
    NEED_INIT(h);
    return get_state_indexed_launch(h, n, reinterpret_cast<const long long*>(d_idx), d_mu, d_sigma);
}

/* one device, checked indices: stages n rows only */
static int get_state_indexed_one(ukfb_handle* h, int64_t n, const int64_t* idx, double* mu, double* sigma)
{
    CHECK_H(h); /* a shard runs this on its worker thread: select its device there */
    if (n == 0) return UKFB_OK;
    const long long* d_idx;
    double *d_mu, *d_sigma;
    Staging st(h, false);
    st.in(&d_idx, idx, sizeof(int64_t) * n);
    st.out(&d_mu, mu, sizeof(double) * n * h->MU);
    st.out(&d_sigma, sigma, sizeof(double) * n * h->n * h->n);
    int rc = st.commit();
    if (!rc) rc = get_state_indexed_launch(h, n, d_idx, d_mu, d_sigma);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_get_state_indexed(ukfb_handle* h, int64_t n, const int64_t* idx, double* mu, double* sigma)
{
    CHECK_H(h);
    if (n < 0) return fail(UKFB_ERR_INVALID, "ukfb_get_state_indexed: n is negative");
    if (n == 0) return UKFB_OK;
    if (!idx || !mu) return fail(UKFB_ERR_INVALID, "ukfb_get_state_indexed: null argument");
    NEED_INIT(h);
    int rc = check_indices(h, n, idx, false, "ukfb_get_state_indexed");
    if (rc || !is_sharded(h)) return rc ? rc : get_state_indexed_one(h, n, idx, mu, sigma);
    /* sharded: each shard gathers its rows into a buffer of its own, then puts them at the caller's rows */
    const size_t nn = size_t(h->n) * size_t(h->n);
    try {
        const ShardRows rows(h, n, idx);
        std::vector<std::vector<double>> m(h->shards.size()), sg(h->shards.size());
        for (size_t i = 0; i < h->shards.size(); ++i) {
            m[i].resize(rows.local[i].size() * size_t(h->MU));
            if (sigma) sg[i].resize(rows.local[i].size() * nn);
        }
        return fan_out(h, [&](ukfb_handle* s_, long long f_, long long) -> int {
            const size_t i = shard_at(h, f_);
            const int64_t c = int64_t(rows.local[i].size());
            const int r = get_state_indexed_one(s_, c, rows.local[i].data(), m[i].data(), sigma ? sg[i].data() : nullptr);
            if (r) return r;
            for (int64_t j = 0; j < c; ++j) {
                const size_t k = size_t(rows.pos[i][size_t(j)]);
                std::memcpy(mu + k * h->MU, m[i].data() + size_t(j) * h->MU, sizeof(double) * h->MU);
                if (sigma) std::memcpy(sigma + k * nn, sg[i].data() + size_t(j) * nn, sizeof(double) * nn);
            }
            return UKFB_OK;
        });
    } catch (const std::bad_alloc&) {
        return fail(UKFB_ERR_NOMEM, "ukfb_get_state_indexed: out of host memory");
    }
}

static int initialize_indexed_launch(ukfb_handle* h, long long n, const long long* d_idx, const double* d_mu, const double* d_sigma)
{
    IndexParams p = index_params(h, n, d_idx);
    p.mu = const_cast<double*>(d_mu), p.sigma = const_cast<double*>(d_sigma); /* read only by this kernel */
    initialize_indexed_kernel<<<grid_for(n * h->REC), 256, 0, h->stream>>>(p);
    CU(cudaGetLastError());
    return UKFB_OK;
}

extern "C" int ukfb_initialize_indexed_dev(ukfb_handle* h, int64_t n, const int64_t* d_idx, const double* d_mu, const double* d_sigma)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (n < 0) return fail(UKFB_ERR_INVALID, "ukfb_initialize_indexed_dev: n is negative");
    if (n == 0) return UKFB_OK;
    if (!d_idx || !d_mu || !d_sigma) return fail(UKFB_ERR_INVALID, "ukfb_initialize_indexed_dev: null argument");
    NEED_INIT(h);
    return initialize_indexed_launch(h, n, reinterpret_cast<const long long*>(d_idx), d_mu, d_sigma);
}

static int initialize_indexed_one(ukfb_handle* h, int64_t n, const int64_t* idx, const double* mu, const double* sigma)
{
    CHECK_H(h); /* a shard runs this on its worker thread: select its device there */
    if (n == 0) return UKFB_OK;
    const long long* d_idx;
    const double *d_mu, *d_sigma;
    Staging st(h, false);
    st.in(&d_idx, idx, sizeof(int64_t) * n);
    st.in(&d_mu, mu, sizeof(double) * n * h->MU);
    st.in(&d_sigma, sigma, sizeof(double) * n * h->n * h->n);
    int rc = st.commit();
    if (!rc) rc = initialize_indexed_launch(h, n, d_idx, d_mu, d_sigma);
    return rc ? rc : st.finish();
}

extern "C" int ukfb_initialize_indexed(ukfb_handle* h, int64_t n, const int64_t* idx, const double* mu, const double* sigma)
{
    CHECK_H(h);
    if (n < 0) return fail(UKFB_ERR_INVALID, "ukfb_initialize_indexed: n is negative");
    if (n == 0) return UKFB_OK;
    if (!idx || !mu || !sigma) return fail(UKFB_ERR_INVALID, "ukfb_initialize_indexed: null argument");
    NEED_INIT(h);
    int rc = check_indices(h, n, idx, true, "ukfb_initialize_indexed");
    if (rc || !is_sharded(h)) return rc ? rc : initialize_indexed_one(h, n, idx, mu, sigma);
    /* sharded: each shard gets contiguous copies of its rows */
    const size_t nn = size_t(h->n) * size_t(h->n);
    try {
        const ShardRows rows(h, n, idx);
        std::vector<std::vector<double>> m(h->shards.size()), sg(h->shards.size());
        for (size_t i = 0; i < h->shards.size(); ++i) {
            const size_t c = rows.local[i].size();
            m[i].resize(c * size_t(h->MU));
            sg[i].resize(c * nn);
            for (size_t j = 0; j < c; ++j) {
                const size_t k = size_t(rows.pos[i][j]);
                std::memcpy(m[i].data() + j * h->MU, mu + k * h->MU, sizeof(double) * h->MU);
                std::memcpy(sg[i].data() + j * nn, sigma + k * nn, sizeof(double) * nn);
            }
        }
        return fan_out(h, [&](ukfb_handle* s_, long long f_, long long) -> int {
            const size_t i = shard_at(h, f_);
            return initialize_indexed_one(s_, int64_t(rows.local[i].size()), rows.local[i].data(), m[i].data(), sg[i].data());
        });
    } catch (const std::bad_alloc&) {
        return fail(UKFB_ERR_NOMEM, "ukfb_initialize_indexed: out of host memory");
    }
}

/* one device: every match counted, the first min(max_n, count) written to idx */
static int find_status_one(ukfb_handle* h, uint32_t bits, int64_t max_n, int64_t* idx, int64_t* n_found)
{
    CHECK_H(h); /* a shard runs this on its worker thread: select its device there */
    const long long chunks = (h->B + FS_CHUNK - 1) / FS_CHUNK;
    const long long cap = max_n < h->B ? (long long)max_n : h->B;
    const size_t bc = align256(sizeof(long long) * (chunks + 1));
    int rc = stage_grow(h, h->stage, h->stage_bytes, bc + sizeof(long long) * (cap > 0 ? cap : 1), false);
    if (rc) return rc;
    IndexParams p = index_params(h, chunks, nullptr);
    p.bits = bits;
    p.max_n = cap;
    p.counts = reinterpret_cast<long long*>(h->stage);
    p.out_idx = reinterpret_cast<long long*>(h->stage + bc);
    const size_t smem = sizeof(long long) * TILE;
    find_status_count_kernel<<<unsigned(chunks), TILE, smem, h->stream>>>(p);
    find_status_scan_kernel<<<1, TILE, smem, h->stream>>>(p);
    if (cap > 0) find_status_write_kernel<<<unsigned(chunks), TILE, smem, h->stream>>>(p);
    CU(cudaGetLastError());
    long long total = 0;
    CU(cudaMemcpyAsync(&total, p.counts + chunks, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const long long got = total < cap ? total : cap;
    if (got > 0) {
        CU(cudaMemcpyAsync(idx, p.out_idx, sizeof(long long) * got, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    *n_found = total;
    return UKFB_OK;
}

extern "C" int ukfb_find_status(ukfb_handle* h, uint32_t bits, int64_t max_n, int64_t* idx, int64_t* n_found)
{
    CHECK_H(h);
    if (max_n < 0 || !n_found || (max_n > 0 && !idx)) return fail(UKFB_ERR_INVALID, "ukfb_find_status: bad argument");
    if (!is_sharded(h)) return find_status_one(h, bits, max_n, idx, n_found);
    /* sharded: up to max_n from every shard, concatenated in shard order (ascending), truncated; counts summed */
    try {
        const size_t S = h->shards.size();
        std::vector<std::vector<int64_t>> part(S);
        std::vector<int64_t> cnt(S, 0);
        for (size_t i = 0; i < S; ++i) part[i].resize(size_t(std::min<long long>(max_n, h->first[i + 1] - h->first[i])));
        const int rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) -> int {
            const size_t i = shard_at(h, f_);
            return find_status_one(s_, bits, int64_t(part[i].size()), part[i].data(), &cnt[i]);
        });
        if (rc) return rc;
        int64_t total = 0, w = 0;
        for (size_t i = 0; i < S; ++i) {
            const int64_t got = std::min<int64_t>(cnt[i], int64_t(part[i].size()));
            for (int64_t j = 0; j < got && w < max_n; ++j) idx[w++] = part[i][size_t(j)] + h->first[i];
            total += cnt[i];
        }
        *n_found = total;
        return UKFB_OK;
    } catch (const std::bad_alloc&) {
        return fail(UKFB_ERR_NOMEM, "ukfb_find_status: out of host memory");
    }
}

static int clear_status_indexed_one(ukfb_handle* h, int64_t n, const int64_t* idx)
{
    CHECK_H(h); /* a shard runs this on its worker thread: select its device there */
    if (n == 0) return UKFB_OK;
    const long long* d_idx;
    Staging st(h, false);
    st.in(&d_idx, idx, sizeof(int64_t) * n);
    int rc = st.commit();
    if (rc) return rc;
    clear_status_indexed_kernel<<<grid_for(n), 256, 0, h->stream>>>(index_params(h, n, d_idx));
    CU(cudaGetLastError());
    return st.finish();
}

extern "C" int ukfb_clear_status_indexed(ukfb_handle* h, int64_t n, const int64_t* idx)
{
    CHECK_H(h);
    if (n < 0) return fail(UKFB_ERR_INVALID, "ukfb_clear_status_indexed: n is negative");
    if (n == 0) return UKFB_OK;
    if (!idx) return fail(UKFB_ERR_INVALID, "ukfb_clear_status_indexed: null argument");
    int rc = check_indices(h, n, idx, false, "ukfb_clear_status_indexed");
    if (rc || !is_sharded(h)) return rc ? rc : clear_status_indexed_one(h, n, idx);
    try {
        const ShardRows rows(h, n, idx);
        return fan_out(h, [&](ukfb_handle* s_, long long f_, long long) -> int {
            const size_t i = shard_at(h, f_);
            return clear_status_indexed_one(s_, int64_t(rows.local[i].size()), rows.local[i].data());
        });
    } catch (const std::bad_alloc&) {
        return fail(UKFB_ERR_NOMEM, "ukfb_clear_status_indexed: out of host memory");
    }
}

/* ---- checkpoint / restore (format: include/ukf_batch.h; record transforms: ukf_checkpoint.cuh) ----------------------- */
enum { CK_RECORDS, CK_T_LAST, CK_STATUS, CK_ACC_MU, CK_ACC_COV, CK_GYRO_MU, CK_Q, CK_ORI, CK_MEAS0 };
static_assert(CK_MEAS0 + UKFB_MEAS_KIND_COUNT == UKFB_CKPT_SECTIONS, "one section per measurement kind");

struct CkptSection {
    uint32_t id, zero;
    uint64_t offset, bytes;
};
struct CkptHeader {
    char magic[8];
    uint32_t version, header_bytes;
    uint64_t total_bytes;
    int32_t kind, MU, n;
    uint32_t n_sections;
    int64_t B;
    uint32_t initialized, first_init;
    double min_dt, max_dt, gate_d2, tau_g, tau_a, latitude, earth[3];
    uint64_t hist[8];
    uint32_t q_per_filter, has_ori_params;
    uint32_t meas_cov_mode[UKFB_MEAS_KIND_COUNT]; /* 0 none, 1 broadcast, 2 per filter: ukfb_handle::meas_cov_per_filter */
    uint8_t zero[16];
    CkptSection section[UKFB_CKPT_SECTIONS];
    uint8_t pad[UKFB_CKPT_HEADER_BYTES - 256 - UKFB_CKPT_SECTIONS * sizeof(CkptSection)];
};
static_assert(sizeof(CkptHeader) == UKFB_CKPT_HEADER_BYTES && offsetof(CkptHeader, B) == 40 && offsetof(CkptHeader, min_dt) == 56 &&
                  offsetof(CkptHeader, hist) == 128 && offsetof(CkptHeader, q_per_filter) == 192 &&
                  offsetof(CkptHeader, meas_cov_mode) == 200 && offsetof(CkptHeader, section) == 256,
              "the header layout of include/ukf_batch.h");
static const char CKPT_MAGIC[8] = {'U', 'K', 'F', 'B', 'C', 'K', 'P', 'T'};

/* what decides the sections an image has */
struct CkptModes {
    uint32_t q_per_filter = 0, has_ori_params = 0;
    uint32_t meas[UKFB_MEAS_KIND_COUNT] = {};
};

static CkptModes ckpt_modes(const ukfb_handle* h) /* a one-device handle: its own; a sharded parent: shard 0's (the setters fan out) */
{
    const ukfb_handle* s = is_sharded(h) ? h->shards[0] : h;
    CkptModes m;
    m.q_per_filter = s->q_per_filter ? 1 : 0;
    m.has_ori_params = s->ori_params ? 1 : 0;
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) m.meas[k] = uint32_t(s->meas_cov_per_filter[k]);
    return m;
}

/* where the sections of an image of B filters lie */
struct CkptLayout {
    uint64_t off[UKFB_CKPT_SECTIONS] = {}, bytes[UKFB_CKPT_SECTIONS] = {};
    uint64_t row[UKFB_CKPT_SECTIONS] = {}; /* bytes per filter; 0 = one block for all filters (or absent) */
    uint64_t total = 0;
};

static CkptLayout ckpt_layout(int kind, long long B, const CkptModes& m)
{
    const int LP = kind == UKFB_POSE ? PoseF::LP : OriF::LP, REC = kind == UKFB_POSE ? PoseF::REC : OriF::REC;
    uint64_t block[UKFB_CKPT_SECTIONS] = {};
    bool per[UKFB_CKPT_SECTIONS] = {};
    block[CK_RECORDS] = sizeof(double) * REC, block[CK_T_LAST] = sizeof(int64_t), block[CK_STATUS] = sizeof(uint32_t);
    block[CK_ACC_MU] = block[CK_GYRO_MU] = sizeof(double) * 3, block[CK_ACC_COV] = sizeof(double) * 9;
    for (int s = CK_RECORDS; s <= CK_GYRO_MU; ++s) per[s] = true;
    block[CK_Q] = sizeof(double) * LP, per[CK_Q] = m.q_per_filter != 0;
    block[CK_ORI] = m.has_ori_params ? sizeof(double) * 5 : 0, per[CK_ORI] = true;
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) {
        const int d = meas_dim(k);
        block[CK_MEAS0 + k] = m.meas[k] ? sizeof(double) * d * d : 0;
        per[CK_MEAS0 + k] = m.meas[k] == 2;
    }
    CkptLayout L;
    uint64_t at = UKFB_CKPT_HEADER_BYTES;
    for (int s = 0; s < UKFB_CKPT_SECTIONS; ++s) {
        if (!block[s]) continue;
        at = align256(at);
        L.off[s] = at;
        L.row[s] = per[s] ? block[s] : 0;
        L.bytes[s] = per[s] ? block[s] * uint64_t(B) : block[s];
        at += L.bytes[s];
    }
    L.total = at;
    return L;
}

/* the header of an image of B filters with the handle-wide values of the one-device handle s; hist is left zero */
static CkptHeader ckpt_header(const ukfb_handle* s, long long B, const CkptModes& m, const CkptLayout& L)
{
    CkptHeader hd;
    memset(&hd, 0, sizeof(hd));
    memcpy(hd.magic, CKPT_MAGIC, 8);
    hd.version = UKFB_CHECKPOINT_VERSION, hd.header_bytes = UKFB_CKPT_HEADER_BYTES, hd.total_bytes = L.total;
    hd.kind = s->kind, hd.MU = s->MU, hd.n = s->n, hd.n_sections = UKFB_CKPT_SECTIONS, hd.B = B;
    hd.initialized = s->initialized ? 1 : 0, hd.first_init = s->first_init ? 1 : 0;
    hd.min_dt = s->min_dt, hd.max_dt = s->max_dt, hd.gate_d2 = s->gate_d2;
    hd.tau_g = s->tau_g, hd.tau_a = s->tau_a, hd.latitude = s->latitude;
    for (int i = 0; i < 3; ++i) hd.earth[i] = s->earth[i];
    hd.q_per_filter = m.q_per_filter, hd.has_ori_params = m.has_ori_params;
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) hd.meas_cov_mode[k] = m.meas[k];
    for (int i = 0; i < UKFB_CKPT_SECTIONS; ++i) hd.section[i] = CkptSection{uint32_t(i), 0u, L.off[i], L.bytes[i]};
    return hd;
}

/* every check of a restore, on the host, before anything is enqueued; h: the handle restored into (a parent for a
 * sharded one).  On success *L is the image's layout. */
static int ckpt_check(const ukfb_handle* h, const CkptHeader& hd, uint64_t bytes, CkptLayout* L, const char* who)
{
    if (memcmp(hd.magic, CKPT_MAGIC, 8) != 0) return fail(UKFB_ERR_INVALID, "%s: not a checkpoint image (bad magic)", who);
    if (hd.version != UKFB_CHECKPOINT_VERSION || hd.header_bytes != UKFB_CKPT_HEADER_BYTES || hd.n_sections != UKFB_CKPT_SECTIONS)
        return fail(UKFB_ERR_INVALID, "%s: image version %u (header %u bytes, %u sections); this library reads version %d", who,
                    hd.version, hd.header_bytes, hd.n_sections, UKFB_CHECKPOINT_VERSION);
    if (hd.kind != h->kind || hd.B != h->B || hd.MU != h->MU || hd.n != h->n)
        return fail(UKFB_ERR_INVALID, "%s: the image holds %lld filters of kind %d (MU %d, n %d); this handle %lld of kind %d", who,
                    (long long)hd.B, hd.kind, hd.MU, hd.n, h->B, h->kind);
    if (hd.initialized > 1 || hd.first_init > 1 || hd.q_per_filter > 1 || hd.has_ori_params > 1 ||
        (hd.has_ori_params && h->kind != UKFB_ORIENTATION))
        return fail(UKFB_ERR_INVALID, "%s: bad flags in the image header", who);
    CkptModes m;
    m.q_per_filter = hd.q_per_filter, m.has_ori_params = hd.has_ori_params;
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) {
        if (hd.meas_cov_mode[k] > 2 || (hd.meas_cov_mode[k] && !kind_ok(h, k)))
            return fail(UKFB_ERR_INVALID, "%s: bad kept-covariance mode %u for measurement kind %d", who, hd.meas_cov_mode[k], k);
        m.meas[k] = hd.meas_cov_mode[k];
    }
    *L = ckpt_layout(h->kind, h->B, m);
    for (int s = 0; s < UKFB_CKPT_SECTIONS; ++s) {
        const CkptSection& e = hd.section[s];
        if (e.id != uint32_t(s) || e.zero || e.offset != L->off[s] || e.bytes != L->bytes[s])
            return fail(UKFB_ERR_INVALID, "%s: section %d is %llu bytes at %llu; the header's modes make it %llu bytes at %llu", who, s,
                        (unsigned long long)e.bytes, (unsigned long long)e.offset, (unsigned long long)L->bytes[s],
                        (unsigned long long)L->off[s]);
    }
    if (hd.total_bytes != L->total || L->total > bytes)
        return fail(UKFB_ERR_INVALID, "%s: the image needs %llu bytes (header: %llu), %llu given", who, (unsigned long long)L->total,
                    (unsigned long long)hd.total_bytes, (unsigned long long)bytes);
    return UKFB_OK;
}

/* the alignment gaps of an image before each present section: fn(offset, bytes) -- zeroed, so that an image's bytes
 * depend on the filters' state alone */
UKFB_HD int ckpt_gaps(const CkptSection* sec, uint64_t at[UKFB_CKPT_SECTIONS], uint64_t len[UKFB_CKPT_SECTIONS])
{
    uint64_t end = UKFB_CKPT_HEADER_BYTES;
    int n = 0;
    for (int s = 0; s < UKFB_CKPT_SECTIONS; ++s)
        if (sec[s].bytes) {
            if (sec[s].offset > end) at[n] = end, len[n++] = sec[s].offset - end;
            end = sec[s].offset + sec[s].bytes;
        }
    return n;
}

/* the header, its histogram summed over the handle's slots on the device (the header travels as the kernel's argument),
 * and the zero gaps between sections */
__global__ void ckpt_header_kernel(const CkptHeader hd, const unsigned long long* __restrict__ hist, unsigned long long* __restrict__ out)
{
    const unsigned long long* w = reinterpret_cast<const unsigned long long*>(&hd);
    for (int i = threadIdx.x; i < UKFB_CKPT_HEADER_BYTES / 8; i += blockDim.x) {
        const int k = i - int(offsetof(CkptHeader, hist) / 8);
        unsigned long long v = w[i];
        if (k >= 0 && k < 8) {
            v = 0;
            for (int s = 0; s < HIST_SLOTS; ++s) v += hist[s * 8 + k];
        }
        out[i] = v;
    }
    char* img = reinterpret_cast<char*>(out);
    uint64_t at[UKFB_CKPT_SECTIONS], len[UKFB_CKPT_SECTIONS];
    const int gaps = ckpt_gaps(hd.section, at, len);
    for (int g = 0; g < gaps; ++g)
        for (uint64_t j = threadIdx.x; j < len[g]; j += blockDim.x) img[at[g] + j] = 0;
}

struct CkptHist {
    unsigned long long w[8];
};
/* a restored histogram: all of it in slot 0, the other slots zero */
__global__ void ckpt_hist_kernel(const CkptHist v, unsigned long long* __restrict__ hist)
{
    for (int i = threadIdx.x; i < HIST_SLOTS * 8; i += blockDim.x) hist[i] = i < 8 ? v.w[i] : 0ull;
}

template <int REC>
static void ckpt_tile_launch(const ukfb_handle* h, bool save, const CkptParams& p)
{
    const long long tiles = (p.B + TILE - 1) / TILE;
    const unsigned grid = unsigned(std::min<long long>(tiles, 148 * 16));
    const size_t smem = sizeof(ckpt_word) * ckpt_tile_words(REC); /* one warp per block: 24 / 28 KB, no opt-in needed */
    if (save)
        ckpt_save_tile_kernel<REC><<<grid, TILE, smem, h->stream>>>(p);
    else
        ckpt_restore_tile_kernel<REC><<<grid, TILE, smem, h->stream>>>(p);
}

/* records of filters [f0, f0 + n) (f0 a multiple of TILE: whole tiles in either layout start at f0 * REC) <-> n rows.
 * Per tile through shared memory; UKFB_CKPT_TRANSFORM=elem selects the per-element kernels (DESIGN.md 7.6 compares them) */
static int ckpt_transform(ukfb_handle* h, bool save, ckpt_word* rows, long long f0, long long n)
{
    const CkptParams p{reinterpret_cast<ckpt_word*>(h->state) + f0 * h->REC, rows, n, h->REC, h->tiled};
    if (knobs().ckpt_elem) {
        if (save)
            ckpt_save_elem_kernel<<<grid_for(n * h->REC), 256, 0, h->stream>>>(p);
        else
            ckpt_restore_elem_kernel<<<grid_for(n * h->REC), 256, 0, h->stream>>>(p);
    } else if (h->REC == PoseF::REC)
        ckpt_tile_launch<PoseF::REC>(h, save, p);
    else
        ckpt_tile_launch<OriF::REC>(h, save, p);
    CU(cudaGetLastError());
    return UKFB_OK;
}

/* host-pointer calls move the record section through a device buffer of at most this many bytes, a whole number of tiles
 * at a time; every other section is dense on the device and goes straight between the caller's buffer and its array */
constexpr long long CKPT_STAGE_BYTES = 64ll << 20;
static long long ckpt_chunk(const ukfb_handle* h)
{
    const long long per = CKPT_STAGE_BYTES / (long long)(sizeof(double) * h->REC) / TILE * TILE;
    return std::min<long long>(per, (h->B + TILE - 1) / TILE * TILE);
}

/* the device arrays behind the sections other than the records, on a one-device handle */
static void* ckpt_array(ukfb_handle* h, int s)
{
    switch (s) {
        case CK_T_LAST: return h->t_last;
        case CK_STATUS: return h->status;
        case CK_ACC_MU: return h->acc_mu;
        case CK_ACC_COV: return h->acc_cov;
        case CK_GYRO_MU: return h->gyro_mu;
        case CK_Q: return h->Q;
        case CK_ORI: return h->ori_params;
        default: return h->meas_cov[s - CK_MEAS0];
    }
}

/* bytes of section s that a one-device handle of h->B filters holds (its rows of a per-filter section, or the block) */
static uint64_t ckpt_local_bytes(const ukfb_handle* h, const CkptLayout& G, int s)
{
    return G.row[s] ? G.row[s] * uint64_t(h->B) : G.bytes[s];
}

/* save_dev: the whole image of a one-device handle into d_img, enqueue only */
static int ckpt_save_enqueue(ukfb_handle* h, char* d_img, const CkptLayout& L, const CkptHeader& hd)
{
    ckpt_header_kernel<<<1, 256, 0, h->stream>>>(hd, h->hist, reinterpret_cast<unsigned long long*>(d_img));
    CU(cudaGetLastError());
    if (int rc = ckpt_transform(h, true, reinterpret_cast<ckpt_word*>(d_img + L.off[CK_RECORDS]), 0, h->B)) return rc;
    for (int s = CK_T_LAST; s < UKFB_CKPT_SECTIONS; ++s)
        if (L.bytes[s]) CU(cudaMemcpyAsync(d_img + L.off[s], ckpt_array(h, s), L.bytes[s], cudaMemcpyDeviceToDevice, h->stream));
    return UKFB_OK;
}

/* host save of one device holding filters [first, first + B) of an image of layout G: its rows of every per-filter
 * section into their places in `buf`, the blocks stored once when first = 0, and its histogram summed into hist[8] */
static int ckpt_save_part(ukfb_handle* h, long long first, const CkptLayout& G, char* buf, uint64_t hist[8])
{
    CHECK_H_AS(h, "ukfb_checkpoint_save"); /* a shard runs this on its worker thread: select its device there */
    const long long chunk = ckpt_chunk(h);
    const uint64_t rb = G.row[CK_RECORDS];
    ckpt_word* d_rows;
    Staging st(h, false);
    st.scratch(&d_rows, size_t(chunk * rb));
    int rc = st.commit();
    if (rc) return rc;
    for (long long f0 = 0; f0 < h->B; f0 += chunk) { /* the next chunk's transform waits for this chunk's copy: one stream */
        const long long n = std::min(chunk, h->B - f0);
        if ((rc = ckpt_transform(h, true, d_rows, f0, n))) return rc;
        CU(cudaMemcpyAsync(buf + G.off[CK_RECORDS] + uint64_t(first + f0) * rb, d_rows, size_t(n * rb), cudaMemcpyDeviceToHost, h->stream));
    }
    for (int s = CK_T_LAST; s < UKFB_CKPT_SECTIONS; ++s)
        if (G.bytes[s] && (G.row[s] || first == 0))
            CU(cudaMemcpyAsync(buf + G.off[s] + uint64_t(first) * G.row[s], ckpt_array(h, s), ckpt_local_bytes(h, G, s), cudaMemcpyDeviceToHost,
                               h->stream));
    unsigned long long slots[HIST_SLOTS * 8];
    CU(cudaMemcpyAsync(slots, h->hist, sizeof(slots), cudaMemcpyDeviceToHost, h->stream));
    if ((rc = st.finish())) return rc;
    for (int k = 0; k < 8; ++k) {
        hist[k] = 0;
        for (int j = 0; j < HIST_SLOTS; ++j) hist[k] += slots[j * 8 + k];
    }
    return UKFB_OK;
}

/* restore of one device holding filters [first, first + B) from an image of layout G with the checked header hd:
 * src is the image in host memory (host-pointer call: records staged by chunks, blocking) or in this device's memory
 * (restore_dev: enqueue only).  hist_here: the image's histogram goes to this device, else its histogram is cleared.
 * q_host: the image's broadcast Q (LP doubles, host), or null when per filter.  Buffers whose mode changes are all
 * allocated before any old one is freed, so a failed allocation leaves this device's handle as it was. */
static int ckpt_restore_part(ukfb_handle* h, long long first, const CkptLayout& G, const char* src, bool src_dev, const CkptHeader& hd,
                             bool hist_here, const double* q_host, const char* who)
{
    CHECK_H_AS(h, who);
    const long long chunk = ckpt_chunk(h);
    const uint64_t rb = G.row[CK_RECORDS];
    ckpt_word* d_rows = nullptr;
    Staging st(h, false);
    if (!src_dev) {
        st.scratch(&d_rows, size_t(chunk * rb));
        if (int rc = st.commit()) return rc;
    }
    /* the arrays whose size changes with the image's modes: new ones first */
    double** slot[2 + UKFB_MEAS_KIND_COUNT];
    double* fresh[2 + UKFB_MEAS_KIND_COUNT];
    int sec[2 + UKFB_MEAS_KIND_COUNT], nr = 0;
    if (int(hd.q_per_filter) != h->q_per_filter) slot[nr] = &h->Q, sec[nr++] = CK_Q;
    if (bool(hd.has_ori_params) != (h->ori_params != nullptr)) slot[nr] = &h->ori_params, sec[nr++] = CK_ORI;
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k)
        if (int(hd.meas_cov_mode[k]) != h->meas_cov_per_filter[k]) slot[nr] = &h->meas_cov[k], sec[nr++] = CK_MEAS0 + k;
    for (int i = 0; i < nr; ++i) {
        fresh[i] = nullptr;
        const uint64_t bytes = ckpt_local_bytes(h, G, sec[i]);
        const cudaError_t e = bytes ? cudaMalloc(&fresh[i], bytes) : cudaSuccess;
        if (e != cudaSuccess) {
            for (int j = 0; j < i; ++j) cudaFree(fresh[j]);
            return fail(UKFB_ERR_NOMEM, "%s: %s", who, cudaGetErrorString(e));
        }
    }
    if (nr) {
        CU(cudaStreamSynchronize(h->stream)); /* nothing may still read the old arrays */
        for (int i = 0; i < nr; ++i) {
            cudaFree(*slot[i]);
            *slot[i] = fresh[i];
        }
    }
    h->q_per_filter = int(hd.q_per_filter);
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) h->meas_cov_per_filter[k] = int(hd.meas_cov_mode[k]);
    const cudaMemcpyKind kind = src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    int rc = UKFB_OK;
    if (src_dev)
        rc = ckpt_transform(h, false, reinterpret_cast<ckpt_word*>(const_cast<char*>(src) + G.off[CK_RECORDS]), 0, h->B);
    else
        for (long long f0 = 0; f0 < h->B && !rc; f0 += chunk) { /* this chunk's copy waits for the last chunk's transform */
            const long long n = std::min(chunk, h->B - f0);
            CU(cudaMemcpyAsync(d_rows, src + G.off[CK_RECORDS] + uint64_t(first + f0) * rb, size_t(n * rb), cudaMemcpyHostToDevice, h->stream));
            rc = ckpt_transform(h, false, d_rows, f0, n);
        }
    if (rc) return rc;
    for (int s = CK_T_LAST; s < UKFB_CKPT_SECTIONS; ++s)
        if (G.bytes[s]) CU(cudaMemcpyAsync(ckpt_array(h, s), src + G.off[s] + uint64_t(first) * G.row[s], ckpt_local_bytes(h, G, s), kind, h->stream));
    CkptHist hv;
    for (int k = 0; k < 8; ++k) hv.w[k] = hist_here ? hd.hist[k] : 0ull;
    ckpt_hist_kernel<<<1, 256, 0, h->stream>>>(hv, h->hist);
    CU(cudaGetLastError());
    h->q_diagonal = hd.q_per_filter ? 0 : broadcast_q_class(q_host, h->n);
    h->min_dt = hd.min_dt, h->max_dt = hd.max_dt, h->gate_d2 = hd.gate_d2;
    h->tau_g = hd.tau_g, h->tau_a = hd.tau_a, h->latitude = hd.latitude;
    for (int i = 0; i < 3; ++i) h->earth[i] = hd.earth[i];
    h->initialized = hd.initialized != 0, h->first_init = hd.first_init != 0;
    return src_dev ? UKFB_OK : st.finish();
}

/* restore_dev's one read-back: the header and, where the header's Q section is one block that lies inside the image,
 * that block behind it (checked on the host afterwards like every other field) */
__global__ void ckpt_probe_kernel(const unsigned char* __restrict__ img, uint64_t bytes, unsigned char* __restrict__ out)
{
    const CkptSection* q = reinterpret_cast<const CkptSection*>(img + offsetof(CkptHeader, section)) + CK_Q;
    for (int i = threadIdx.x; i < UKFB_CKPT_HEADER_BYTES; i += blockDim.x) out[i] = img[i];
    const uint64_t off = q->offset, n = q->bytes;
    if (n && n <= sizeof(double) * OriF::LP && off >= UKFB_CKPT_HEADER_BYTES && off <= bytes && n <= bytes - off)
        for (uint64_t i = threadIdx.x; i < n; i += blockDim.x) out[UKFB_CKPT_HEADER_BYTES + i] = img[off + i];
}

extern "C" int ukfb_checkpoint_size(ukfb_handle* h, uint64_t* bytes)
{
    if (!h || !bytes) return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_size: null argument");
    *bytes = ckpt_layout(h->kind, h->B, ckpt_modes(h)).total;
    return UKFB_OK;
}

extern "C" int ukfb_checkpoint_save(ukfb_handle* h, void* buf, uint64_t bytes)
{
    CHECK_H(h);
    NEED_INIT(h);
    const CkptModes m = ckpt_modes(h);
    const CkptLayout G = ckpt_layout(h->kind, h->B, m);
    if (!buf) return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_save: null buffer");
    if (bytes < G.total)
        return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_save: the image needs %llu bytes, the buffer has %llu", (unsigned long long)G.total,
                    (unsigned long long)bytes);
    char* out = static_cast<char*>(buf);
    CkptHeader hd = ckpt_header(is_sharded(h) ? h->shards[0] : h, h->B, m, G);
    uint64_t at[UKFB_CKPT_SECTIONS], len[UKFB_CKPT_SECTIONS];
    for (int g = ckpt_gaps(hd.section, at, len) - 1; g >= 0; --g) memset(out + at[g], 0, len[g]); /* the sections go in concurrently */
    std::vector<std::array<uint64_t, 8>> part(h->shards.empty() ? 1 : h->shards.size());
    const int rc = is_sharded(h) ? fan_out(h, [&](ukfb_handle* s_, long long f_, long long) { return ckpt_save_part(s_, f_, G, out, part[shard_at(h, f_)].data()); })
                                 : ckpt_save_part(h, 0, G, out, part[0].data());
    if (rc) return rc;
    /* handle-wide values of shard 0 (every setter fans out: the shards agree), the histogram summed over the shards */
    for (const auto& p : part)
        for (int k = 0; k < 8; ++k) hd.hist[k] += p[size_t(k)];
    memcpy(out, &hd, sizeof(hd));
    return UKFB_OK;
}

extern "C" int ukfb_checkpoint_restore(ukfb_handle* h, const void* buf, uint64_t bytes)
{
    CHECK_H(h);
    if (!buf) return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_restore: null buffer");
    if (bytes < sizeof(CkptHeader))
        return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_restore: %llu bytes cannot hold an image", (unsigned long long)bytes);
    const char* in = static_cast<const char*>(buf);
    CkptHeader hd;
    memcpy(&hd, in, sizeof(hd));
    CkptLayout G;
    int rc = ckpt_check(h, hd, bytes, &G, "ukfb_checkpoint_restore");
    if (rc) return rc;
    double q[OriF::LP]; /* the broadcast Q, copied out: the caller's buffer need not be aligned */
    if (!hd.q_per_filter) memcpy(q, in + G.off[CK_Q], G.bytes[CK_Q]);
    const double* qp = hd.q_per_filter ? nullptr : q;
    if (!is_sharded(h)) return ckpt_restore_part(h, 0, G, in, false, hd, true, qp, "ukfb_checkpoint_restore");
    /* a shard that cannot allocate fails alone: the others are restored (UKFB_ERR_NOMEM names the shard) */
    rc = fan_out(h, [&](ukfb_handle* s_, long long f_, long long) { return ckpt_restore_part(s_, f_, G, in, false, hd, f_ == 0, qp, "ukfb_checkpoint_restore"); });
    if (rc) return rc;
    /* the parent's own copies of handle-wide values (the setters keep them too) */
    h->min_dt = hd.min_dt, h->max_dt = hd.max_dt, h->gate_d2 = hd.gate_d2;
    h->tau_g = hd.tau_g, h->tau_a = hd.tau_a, h->latitude = hd.latitude;
    for (int i = 0; i < 3; ++i) h->earth[i] = hd.earth[i];
    for (int k = 0; k < UKFB_MEAS_KIND_COUNT; ++k) h->meas_cov_per_filter[k] = int(hd.meas_cov_mode[k]);
    h->initialized = hd.initialized != 0, h->first_init = hd.first_init != 0;
    return UKFB_OK;
}

extern "C" int ukfb_checkpoint_save_dev(ukfb_handle* h, void* d_buf, uint64_t bytes)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    NEED_INIT(h);
    const CkptModes m = ckpt_modes(h);
    const CkptLayout L = ckpt_layout(h->kind, h->B, m);
    if (!d_buf) return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_save_dev: null buffer");
    if (bytes < L.total)
        return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_save_dev: the image needs %llu bytes, the buffer has %llu",
                    (unsigned long long)L.total, (unsigned long long)bytes);
    return ckpt_save_enqueue(h, static_cast<char*>(d_buf), L, ckpt_header(h, h->B, m, L));
}

extern "C" int ukfb_checkpoint_restore_dev(ukfb_handle* h, const void* d_buf, uint64_t bytes)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    if (!d_buf) return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_restore_dev: null buffer");
    if (bytes < sizeof(CkptHeader))
        return fail(UKFB_ERR_INVALID, "ukfb_checkpoint_restore_dev: %llu bytes cannot hold an image", (unsigned long long)bytes);
    const char* in = static_cast<const char*>(d_buf);
    const size_t probe = UKFB_CKPT_HEADER_BYTES + sizeof(double) * OriF::LP;
    int rc = stage_grow(h, h->stage, h->stage_bytes, probe, false);
    if (rc) return rc;
    ckpt_probe_kernel<<<1, 256, 0, h->stream>>>(reinterpret_cast<const unsigned char*>(in), bytes, reinterpret_cast<unsigned char*>(h->stage));
    CU(cudaGetLastError());
    unsigned char back[UKFB_CKPT_HEADER_BYTES + sizeof(double) * OriF::LP];
    CU(cudaMemcpyAsync(back, h->stage, probe, cudaMemcpyDeviceToHost, h->stream)); /* after whatever wrote the image on this stream */
    CU(cudaStreamSynchronize(h->stream));
    CkptHeader hd;
    memcpy(&hd, back, sizeof(hd));
    CkptLayout L;
    rc = ckpt_check(h, hd, bytes, &L, "ukfb_checkpoint_restore_dev");
    if (rc) return rc;
    double q[OriF::LP]; /* checked: a broadcast Q section is one block inside the image, so the probe copied it */
    if (!hd.q_per_filter) memcpy(q, back + UKFB_CKPT_HEADER_BYTES, L.bytes[CK_Q]);
    return ckpt_restore_part(h, 0, L, in, true, hd, true, hd.q_per_filter ? nullptr : q, "ukfb_checkpoint_restore_dev");
}

/* ---- stream plumbing ------------------------------------------------------------------------------------------ */
extern "C" int ukfb_synchronize(ukfb_handle* h)
{
    CHECK_H(h);
    UKFB_FAN(h, ukfb_synchronize(s_));
    CU(cudaStreamSynchronize(h->stream));
    if (h->pipe.made) {
        CU(cudaStreamSynchronize(h->pipe.s_in));
        CU(cudaStreamSynchronize(h->pipe.s_out));
    }
    return UKFB_OK;
}

extern "C" void* ukfb_stream(ukfb_handle* h) { return h ? reinterpret_cast<void*>(h->stream) : nullptr; } /* sharded parent: null */

extern "C" int ukfb_wait_for_stream(ukfb_handle* h, void* cuda_stream)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    cudaEvent_t e;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaError_t rc = cudaEventRecord(e, reinterpret_cast<cudaStream_t>(cuda_stream));
    if (rc == cudaSuccess) rc = cudaStreamWaitEvent(h->stream, e, 0);
    cudaEventDestroy(e); /* released once the recorded work has completed */
    if (rc != cudaSuccess) return fail(UKFB_ERR_CUDA, "ukfb_wait_for_stream: %s", cudaGetErrorString(rc));
    return UKFB_OK;
}

extern "C" int ukfb_stream_wait(ukfb_handle* h, void* cuda_stream)
{
    CHECK_H(h);
    UKFB_NOT_SHARDED(h);
    cudaEvent_t e;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaError_t rc = cudaEventRecord(e, h->stream);
    if (rc == cudaSuccess) rc = cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(cuda_stream), e, 0);
    cudaEventDestroy(e);
    if (rc != cudaSuccess) return fail(UKFB_ERR_CUDA, "ukfb_stream_wait: %s", cudaGetErrorString(rc));
    return UKFB_OK;
}

extern "C" int ukfb_event_record(ukfb_handle* h, int slot)
{
    CHECK_H(h);
    if (slot < 0 || slot >= 16) return fail(UKFB_ERR_INVALID, "ukfb_event_record: slot out of range");
    UKFB_FAN(h, ukfb_event_record(s_, slot)); /* every shard records on its own stream */
    CU(cudaEventRecord(h->ev[slot], h->stream));
    return UKFB_OK;
}

extern "C" int ukfb_event_elapsed_ms(ukfb_handle* h, int slot_begin, int slot_end, float* ms)
{
    CHECK_H(h);
    if (slot_begin < 0 || slot_begin >= 16 || slot_end < 0 || slot_end >= 16 || !ms) return fail(UKFB_ERR_INVALID, "ukfb_event_elapsed_ms: bad argument");
    if (is_sharded(h)) { /* the slowest shard: device-timed, max over devices */
        *ms = 0.f;
        for (ukfb_handle* s : h->shards) {
            float one = 0.f;
            const int rc = ukfb_event_elapsed_ms(s, slot_begin, slot_end, &one);
            if (rc) return rc;
            if (one > *ms) *ms = one;
        }
        return UKFB_OK;
    }
    CU(cudaEventSynchronize(h->ev[slot_end]));
    CU(cudaEventElapsedTime(ms, h->ev[slot_begin], h->ev[slot_end]));
    return UKFB_OK;
}

extern "C" int64_t ukfb_launch_count(const ukfb_handle* h)
{
    if (!h) return 0;
    long long n = h->launches;
    for (const ukfb_handle* s : h->shards) n += s->launches;
    return n;
}

extern "C" int64_t ukfb_overlapped_launch_count(const ukfb_handle* h)
{
    if (!h) return 0;
    long long n = (long long)h->fast_launches;
    for (const ukfb_handle* s : h->shards) n += (long long)s->fast_launches;
    return n;
}

/* self-test of the device SO(3) kernels (so3.cuh): q = exp(v), w = log(q), rc = 1 / x, (sq, rs) = sqrt / rsqrt of x */
__global__ void so3_selftest_kernel(const double* __restrict__ v, const double* __restrict__ x, double* __restrict__ out, long long n)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double q[4], w[3], sq, rs;
        so3_exp(v + 3 * i, 1.0, q);
        so3_log(q, w);
        fast_sqrt_rsqrt(x[i], sq, rs);
        double* o = out + UKFB_SELFTEST_STRIDE * i;
        o[0] = q[0], o[1] = q[1], o[2] = q[2], o[3] = q[3], o[4] = w[0], o[5] = w[1], o[6] = w[2];
        o[7] = fast_rcp(x[i]), o[8] = sq, o[9] = rs;
        /* the branch-free pair of the fast kernels (ukf_pose_fast.cuh): polynomial exp, reciprocal-free log */
        double qf[4], wf[3];
        bool slow = false;
        pf_exp(v + 3 * i, 1.0, qf, slow);
        pf_log(qf, wf, slow);
        o[10] = wf[0], o[11] = wf[1], o[12] = wf[2], o[13] = slow ? 1.0 : 0.0;
        /* their any-angle pair: eighth-angle polynomial + three squarings, three square roots + asin form; run as the pair
         * type the kernels use (second slot: the opposite rotation) */
        D2 v2[3] = {D2(v[3 * i], -v[3 * i]), D2(v[3 * i + 1], -v[3 * i + 1]), D2(v[3 * i + 2], -v[3 * i + 2])}, q2[4], w2[3];
        bool hard = false;
        pf_exp_wide<D2>(v2, 1.0, q2, hard);
        pf_log_wide<D2>(q2, w2);
        o[14] = q2[0].a, o[15] = q2[1].a, o[16] = q2[2].a, o[17] = q2[3].a;
        o[18] = w2[0].a, o[19] = w2[1].a, o[20] = hard ? 1.0 : w2[2].a;
        if (!hard && !(w2[0].b == -w2[0].a && w2[1].b == -w2[1].a && w2[2].b == -w2[2].a)) o[20] = 1.0 / 0.0; /* the two slots must mirror */
    }
}

extern "C" int ukfb_selftest_so3(ukfb_handle* h, int64_t n, const double* v, const double* x, double* out)
{
    CHECK_H(h);
    if (n < 1 || !v || !x || !out) return fail(UKFB_ERR_INVALID, "ukfb_selftest_so3: bad argument");
    if (is_sharded(h)) return ukfb_selftest_so3(h->shards[0], n, v, x, out);
    const double *d_v, *d_x;
    double* d_out;
    Staging st(h, false);
    st.in(&d_v, v, sizeof(double) * n * 3);
    st.in(&d_x, x, sizeof(double) * n);
    st.out(&d_out, out, sizeof(double) * n * UKFB_SELFTEST_STRIDE);
    int rc = st.commit();
    if (rc) return rc;
    so3_selftest_kernel<<<grid_for(n), 256, 0, h->stream>>>(d_v, d_x, d_out, n);
    CU(cudaGetLastError());
    return st.finish();
}

extern "C" int ukfb_measure_fp64_peak(ukfb_handle* h, double* flops_per_s)
{
    CHECK_H(h);
    if (!flops_per_s) return fail(UKFB_ERR_INVALID, "ukfb_measure_fp64_peak: null argument");
    if (is_sharded(h)) return ukfb_measure_fp64_peak(h->shards[0], flops_per_s);
    int rc = stage_grow(h, h->stage, h->stage_bytes, 256, false);
    if (rc) return rc;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, h->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(a, h->stream));
        dfma_peak_kernel<<<blocks, threads, 0, h->stream>>>(reinterpret_cast<double*>(h->stage), iters, 0.999999, 1e-9);
        CU(cudaEventRecord(b, h->stream));
        CU(cudaEventSynchronize(b));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, a, b));
        const double flops = 2.0 * 64.0 * double(iters) * double(blocks) * double(threads);
        if (rep > 0 && ms > 0.f && flops / (ms * 1e-3) > best) best = flops / (ms * 1e-3);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *flops_per_s = best;
    return UKFB_OK;
}
