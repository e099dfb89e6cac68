/*
 * emu_index.cpp -- runs the per-filter access kernels (ukf_index.cuh) on host threads, launched as ukf_batch.cu launches
 * them.  TEST INFRASTRUCTURE ONLY (tests/test_emu_indexed.py): exercises their indexing -- both record layouts, ragged
 * tiles, skipped indices, the compaction's offsets -- in the GPU-less build container, optionally under ASan / UBSan.
 * Nothing in the product links or loads this.
 */
#define UKFB_SIMT_EMU 1
#include "../../slam_pose_estimation_b200/csrc/ukf_index.cuh"

using namespace ukfb;

static IndexParams params(double* state, long long B, int kind, int tiled, const long long* idx, long long n)
{
    IndexParams p{};
    p.state = state;
    p.B = B;
    p.n = kind == 0 ? 12 : 13;
    p.MU = kind == 0 ? 13 : 14;
    p.REC = p.MU + p.n * (p.n + 1) / 2;
    p.tiled = tiled;
    p.idx = idx;
    p.n_rows = n;
    return p;
}

/* state: the device image of the records (tiled: [tile][entry][lane], AoS: [filter][entry]) */
extern "C" void emu_get_state_indexed(double* state, long long B, int kind, int tiled, const long long* idx, long long n, double* mu,
                                      double* sigma)
{
    IndexParams p = params(state, B, kind, tiled, idx, n);
    p.mu = mu, p.sigma = sigma;
    if (n > 0) simt_emu::launch(get_state_indexed_kernel, 3, 96, 0, p); /* a grid smaller than the rows: the stride loop */
}

extern "C" void emu_initialize_indexed(double* state, long long B, int kind, int tiled, const long long* idx, long long n,
                                       const double* mu, const double* sigma, long long* t_last)
{
    IndexParams p = params(state, B, kind, tiled, idx, n);
    p.mu = const_cast<double*>(mu), p.sigma = const_cast<double*>(sigma), p.t_last = t_last;
    if (n > 0) simt_emu::launch(initialize_indexed_kernel, 3, 96, 0, p);
}

extern "C" void emu_clear_status_indexed(uint32_t* status, long long B, const long long* idx, long long n)
{
    IndexParams p = params(nullptr, B, 0, 1, idx, n);
    p.status = status;
    if (n > 0) simt_emu::launch(clear_status_indexed_kernel, 4, 64, 0, p); /* a grid smaller than n: the stride loop */
}

/* counts: chunks + 1 words of scratch; returns the count, the first min(max_n, count) matches in out */
extern "C" long long emu_find_status(const uint32_t* status, long long B, uint32_t bits, long long max_n, long long* counts,
                                     long long* out)
{
    const long long chunks = (B + FS_CHUNK - 1) / FS_CHUNK;
    IndexParams p = params(nullptr, B, 0, 1, nullptr, chunks);
    p.status = const_cast<uint32_t*>(status), p.bits = bits, p.max_n = max_n < B ? max_n : B, p.counts = counts, p.out_idx = out;
    const size_t smem = sizeof(long long) * TILE;
    simt_emu::launch(find_status_count_kernel, unsigned(chunks), TILE, smem, p);
    simt_emu::launch(find_status_scan_kernel, 1, TILE, smem, p);
    if (p.max_n > 0) simt_emu::launch(find_status_write_kernel, unsigned(chunks), TILE, smem, p);
    return counts[chunks];
}
