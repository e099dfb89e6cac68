/*
 * ukf_checkpoint.cuh -- the two layout transforms of a checkpoint image (include/ukf_batch.h, "checkpoint / restore"):
 * the handle's filter records <-> the image's record section, one row of REC entries per filter in filter order (mu,
 * then the packed lower triangle of sigma in tri(r, c) order: the record's own entry order).
 *
 * The records are kept in one of two layouts (rec_index): 32-filter entry-major tiles (fast and thread kernels) or AoS
 * (warp kernel).  AoS records already are rows, so both transforms copy straight through there.  For tiles, a tile of
 * 32 filters is one contiguous block of 32 x REC doubles in the records AND in the rows (23 KB for PoseUKF, 26 KB for
 * OrientationUKF), and the transform is a transpose of that block.  Two versions:
 *   - per element (ckpt_*_elem_kernel): one thread per element of the destination, grid-stride, in the element order of
 *     the whole-batch unpack / pack kernels of ukf_batch.cu: the save reads 8 bytes from each 256-byte line it touches;
 *   - per tile (ckpt_*_tile_kernel): one warp per tile, staged through shared memory, so that both the read and the write
 *     of a tile are whole 256-byte lines.  Each warp owns its own piece of shared memory and synchronises with __syncwarp
 *     only, which is what the host emulation of tests/simt_emu runs.
 * Both copy 64-bit words and do no arithmetic on them: NaN payloads and -0.0 come through bit for bit.  Rows past B in
 * a ragged last tile are neither read nor written, nor are the padding lanes of the records.
 */
#ifndef UKFB_CHECKPOINT_CUH
#define UKFB_CHECKPOINT_CUH

#include "ukf_index.cuh"

namespace ukfb {

typedef unsigned long long ckpt_word;

struct CkptParams {
    ckpt_word* rec;  /* records of the handle (Bpad x REC words in the handle's layout) */
    ckpt_word* rows; /* B x REC words, filter-major */
    long long B;
    int REC, tiled;
};

/* shared memory of one warp of the tile kernels: REC rows of 33 words (the 33rd keeps the transposed accesses of a warp
 * on different banks) */
UKFB_HD constexpr int ckpt_tile_words(int REC) { return REC * (TILE + 1); }

/* AoS records: a straight copy, grid-stride over the whole grid */
UKFB_D void ckpt_copy_words(ckpt_word* dst, const ckpt_word* src, long long count)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) dst[i] = src[i];
}

/* save, per element: rows[b][e] = record entry e of filter b */
UKFB_GLOBAL void ckpt_save_elem_kernel(const CkptParams p)
{
    const long long total = p.B * p.REC;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / p.REC;
        p.rows[i] = p.rec[rec_index(p.tiled, b, int(i - b * p.REC), p.REC)];
    }
}

/* restore, per element: record entry e of filter b = rows[b][e] */
UKFB_GLOBAL void ckpt_restore_elem_kernel(const CkptParams p)
{
    const long long total = p.B * p.REC;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / p.REC;
        p.rec[rec_index(p.tiled, b, int(i - b * p.REC), p.REC)] = p.rows[i];
    }
}

/* save, per tile.  blockDim.x = 32 x warps; dynamic shared memory = warps x ckpt_tile_words(REC) words */
template <int REC>
UKFB_GLOBAL void ckpt_save_tile_kernel(const CkptParams p)
{
    if (!p.tiled) {
        ckpt_copy_words(p.rows, p.rec, p.B * REC);
        return;
    }
    UKFB_SMEM_DECL
    const int lane = int(threadIdx.x) & 31, warp = int(threadIdx.x) >> 5, wpb = int(blockDim.x) >> 5;
    ckpt_word* s = reinterpret_cast<ckpt_word*>(ukfb_smem) + (long long)warp * ckpt_tile_words(REC);
    const long long tiles = (p.B + TILE - 1) / TILE;
    /* t is the same for the 32 lanes of a warp: the warp stays whole up to every __syncwarp */
    for (long long t = (long long)blockIdx.x * wpb + warp; t < tiles; t += (long long)gridDim.x * wpb) {
        const ckpt_word* src = p.rec + t * (TILE * REC);
        ckpt_word v[REC]; /* loads first, shared-memory stores after: ptxas interleaves them as its 32 registers allow */
#pragma unroll
        for (int e = 0; e < REC; ++e) v[e] = src[e * TILE + lane]; /* whole lines: entry e of 32 filters */
#pragma unroll
        for (int e = 0; e < REC; ++e) s[e * (TILE + 1) + lane] = v[e];
        __syncwarp();
        const long long left = p.B - t * TILE;
        const int nb = left < TILE ? int(left) : TILE;
        ckpt_word* dst = p.rows + t * (TILE * REC);
        for (int k = lane; k < nb * REC; k += TILE) { /* whole lines: the rows of the tile's filters, one after the other */
            const int f = k / REC;
            dst[k] = s[(k - f * REC) * (TILE + 1) + f];
        }
        __syncwarp();
    }
}

/* restore, per tile: the inverse.  The padding lanes of a ragged last tile keep what they hold. */
template <int REC>
UKFB_GLOBAL void ckpt_restore_tile_kernel(const CkptParams p)
{
    if (!p.tiled) {
        ckpt_copy_words(p.rec, p.rows, p.B * REC);
        return;
    }
    UKFB_SMEM_DECL
    const int lane = int(threadIdx.x) & 31, warp = int(threadIdx.x) >> 5, wpb = int(blockDim.x) >> 5;
    ckpt_word* s = reinterpret_cast<ckpt_word*>(ukfb_smem) + (long long)warp * ckpt_tile_words(REC);
    const long long tiles = (p.B + TILE - 1) / TILE;
    for (long long t = (long long)blockIdx.x * wpb + warp; t < tiles; t += (long long)gridDim.x * wpb) {
        const long long left = p.B - t * TILE;
        const int nb = left < TILE ? int(left) : TILE;
        const ckpt_word* src = p.rows + t * (TILE * REC);
        if (nb == TILE) { /* a whole tile: unrolled, loads ahead of the stores as far as ptxas schedules them */
            ckpt_word v[REC];
#pragma unroll
            for (int j = 0; j < REC; ++j) v[j] = src[j * TILE + lane];
#pragma unroll
            for (int j = 0; j < REC; ++j) {
                const int k = j * TILE + lane, f = k / REC;
                s[(k - f * REC) * (TILE + 1) + f] = v[j];
            }
        } else
            for (int k = lane; k < nb * REC; k += TILE) {
                const int f = k / REC;
                s[(k - f * REC) * (TILE + 1) + f] = src[k];
            }
        __syncwarp();
        ckpt_word* dst = p.rec + t * (TILE * REC);
        if (lane < nb) {
#pragma unroll
            for (int e = 0; e < REC; ++e) dst[e * TILE + lane] = s[e * (TILE + 1) + lane];
        }
        __syncwarp();
    }
}

} /* namespace ukfb */

#endif
