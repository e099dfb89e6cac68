/*
 * ukf_index.cuh -- per-filter access to the records of a batch: gather the states of listed filters, re-initialise
 * listed filters, list the filters whose status word has given bits, clear the status of listed filters.
 *
 * What the reference does on ONE of its N filter objects (UnscentedKalmanFilter.hpp:40-44 initializeFilter, :51-75
 * getCurrentState), here for the filters idx[0..n) of a batch, touching only their records.  Every kernel works on both
 * record layouts (rec_index): 32-filter entry-major tiles (fast and thread kernels) and AoS (warp kernel).
 *
 * Gather / scatter: one thread per element of the dense rows (gather) or of the records (scatter), grid-stride, in
 * the element order of the whole-batch unpack / pack kernels of ukf_batch.cu.  Rows in index order therefore make the
 * same accesses as ukfb_get_state_dev / ukfb_initialize; random indices cost one sector per record entry.
 *
 * Status compaction: one 32-thread block per FS_CHUNK filters; lane l scans FS_PER_LANE consecutive filters of the
 * chunk.  Pass 1 counts per chunk, one single-block pass turns the counts into exclusive offsets (and the total),
 * pass 2 writes the matching indices at their offsets.  The order is ascending whatever order the blocks run in.
 *
 * Every kernel takes one IndexParams and synchronises with __syncwarp only, so the same source runs in the host
 * emulation of tests/simt_emu.  The compaction kernels keep all 32 lanes up to every __syncwarp.
 */
#ifndef UKFB_INDEX_CUH
#define UKFB_INDEX_CUH

#include "ukf_thread.cuh"

namespace ukfb {

/* element index of record entry e of filter b: AoS records (warp kernel) or 32-filter entry-major tiles (thread kernel) */
UKFB_HD long long rec_index(int tiled, long long b, int e, int REC) { return tiled ? tile_index(b, e, REC) : b * REC + e; }

constexpr int FS_PER_LANE = 32;     /* status compaction: consecutive filters per lane */
constexpr int FS_CHUNK = TILE * FS_PER_LANE;

struct IndexParams {
    double* state;          /* records of the handle */
    long long B;            /* filters of the handle */
    int MU, n, REC, tiled;
    const long long* idx;   /* n_rows filter indices */
    long long n_rows;
    double* mu;             /* n_rows x MU (gather: out, scatter: in) */
    double* sigma;          /* n_rows x n x n, or null (gather: full symmetric out; scatter: lower triangle read) */
    long long* t_last;      /* scatter: zeroed at idx */
    uint32_t* status;       /* clear: zeroed at idx; compaction: read */
    uint32_t bits;          /* compaction: any of these bits */
    long long max_n;        /* compaction: indices written at most */
    long long* counts;      /* compaction: per chunk, then exclusive offsets; counts[n_chunks] = total */
    long long* out_idx;     /* compaction: ascending matches */
};

/* the filter of row k, or -1 for a row past the end or an index outside [0, B) (skipped: never read or written) */
UKFB_D long long ix_row_filter(const IndexParams& p, long long k)
{
    if (k >= p.n_rows) return -1;
    const long long b = p.idx[k];
    return (b >= 0 && b < p.B) ? b : -1;
}

/* getCurrentState (:51-75) of the listed filters: rows k of mu / sigma = filter idx[k].  One thread per output element,
 * in the order of ukfb_get_state_dev's unpack kernels: for rows in index order the same accesses as the whole-batch read */
UKFB_GLOBAL void get_state_indexed_kernel(const IndexParams p)
{
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    for (long long i = t0; i < p.n_rows * p.MU; i += stride) {
        const long long k = i / p.MU;
        const long long b = ix_row_filter(p, k);
        if (b >= 0) p.mu[i] = p.state[rec_index(p.tiled, b, int(i - k * p.MU), p.REC)];
    }
    if (!p.sigma) return;
    const int nn = p.n * p.n;
    for (long long i = t0; i < p.n_rows * nn; i += stride) {
        const long long k = i / nn;
        const int e = int(i - k * nn);
        int r = e / p.n, c = e - (e / p.n) * p.n;
        if (c > r) {
            const int t = r;
            r = c;
            c = t;
        }
        const long long b = ix_row_filter(p, k);
        if (b >= 0) p.sigma[i] = p.state[rec_index(p.tiled, b, p.MU + tri(r, c), p.REC)];
    }
}

/* initializeFilter (:40-44) of the listed filters: record = (mu, lower triangle of sigma), t_last = 0 (:43).  One thread
 * per record element, as ukfb_initialize's pack kernel */
UKFB_GLOBAL void initialize_indexed_kernel(const IndexParams p)
{
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    for (long long i = t0; i < p.n_rows * p.REC; i += stride) {
        const long long k = i / p.REC;
        const int e = int(i - k * p.REC);
        const long long b = ix_row_filter(p, k);
        if (b < 0) continue;
        double v;
        if (e < p.MU)
            v = p.mu[k * p.MU + e];
        else {
            const int el = e - p.MU;
            int r = 0;
            while ((r + 1) * (r + 2) / 2 <= el) ++r;
            v = p.sigma[(k * p.n + r) * p.n + (el - r * (r + 1) / 2)];
        }
        p.state[rec_index(p.tiled, b, e, p.REC)] = v;
        if (e == 0) p.t_last[b] = 0;
    }
}

/* ukfb_clear_status for the listed filters */
UKFB_GLOBAL void clear_status_indexed_kernel(const IndexParams p)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < p.n_rows; k += (long long)gridDim.x * blockDim.x) {
        const long long b = ix_row_filter(p, k);
        if (b >= 0) p.status[b] = 0u;
    }
}

/* matches among the FS_PER_LANE filters of this lane in chunk `chunk` */
UKFB_D long long fs_lane_count(const IndexParams& p, long long chunk, int lane)
{
    const long long first = chunk * FS_CHUNK + (long long)lane * FS_PER_LANE;
    long long c = 0;
    for (int j = 0; j < FS_PER_LANE; ++j)
        if (first + j < p.B && (p.status[first + j] & p.bits)) ++c;
    return c;
}

/* pass 1: counts[chunk] = matches in the chunk */
UKFB_GLOBAL void find_status_count_kernel(const IndexParams p)
{
    UKFB_SMEM_DECL
    long long* lc = reinterpret_cast<long long*>(ukfb_smem);
    const int lane = int(threadIdx.x) & 31;
    lc[lane] = fs_lane_count(p, blockIdx.x, lane);
    __syncwarp();
    if (lane == 0) {
        long long s = 0;
        for (int l = 0; l < TILE; ++l) s += lc[l];
        p.counts[blockIdx.x] = s;
    }
    __syncwarp();
}

/* pass 1b, one block: counts[0..n_chunks) -> exclusive offsets, counts[n_chunks] = total.  n_chunks = p.n_rows */
UKFB_GLOBAL void find_status_scan_kernel(const IndexParams p)
{
    UKFB_SMEM_DECL
    long long* ls = reinterpret_cast<long long*>(ukfb_smem);
    const int lane = int(threadIdx.x) & 31;
    const long long nc = p.n_rows, per = (nc + TILE - 1) / TILE;
    const long long a = (long long)lane * per, z = a + per < nc ? a + per : nc;
    long long s = 0;
    for (long long c = a; c < z; ++c) s += p.counts[c];
    ls[lane] = s;
    __syncwarp();
    long long off = 0;
    for (int l = 0; l < lane; ++l) off += ls[l];
    __syncwarp();
    for (long long c = a; c < z; ++c) {
        const long long v = p.counts[c];
        p.counts[c] = off;
        off += v;
    }
    if (lane == TILE - 1) p.counts[nc] = off;
    __syncwarp();
}

/* pass 2: the matches of each lane at counts[chunk] + (matches of the lanes before it), the first max_n only */
UKFB_GLOBAL void find_status_write_kernel(const IndexParams p)
{
    UKFB_SMEM_DECL
    long long* lc = reinterpret_cast<long long*>(ukfb_smem);
    const int lane = int(threadIdx.x) & 31;
    const long long chunk = blockIdx.x;
    lc[lane] = fs_lane_count(p, chunk, lane);
    __syncwarp();
    long long off = p.counts[chunk];
    for (int l = 0; l < lane; ++l) off += lc[l];
    const long long first = chunk * FS_CHUNK + (long long)lane * FS_PER_LANE;
    for (int j = 0; j < FS_PER_LANE && off < p.max_n; ++j)
        if (first + j < p.B && (p.status[first + j] & p.bits)) p.out_idx[off++] = first + j;
    __syncwarp();
}

} /* namespace ukfb */

#endif
