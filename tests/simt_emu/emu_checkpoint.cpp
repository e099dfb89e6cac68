/*
 * emu_checkpoint.cpp -- runs the checkpoint record transforms (ukf_checkpoint.cuh) on host threads.  TEST INFRASTRUCTURE
 * ONLY (tests/test_emu_checkpoint.py): exercises their indexing -- both record layouts, ragged last tiles, grids smaller
 * than the work, several warps per block -- in the GPU-less build container, optionally under ASan / UBSan.  Nothing in
 * the product links or loads this.
 */
#define UKFB_SIMT_EMU 1
#include "../../slam_pose_estimation_b200/csrc/ukf_checkpoint.cuh"

using namespace ukfb;

template <int REC>
static void tile(int save, const CkptParams& p, unsigned grid, unsigned warps)
{
    const size_t smem = sizeof(ckpt_word) * warps * ckpt_tile_words(REC);
    if (save)
        simt_emu::launch(ckpt_save_tile_kernel<REC>, grid, 32 * warps, smem, p);
    else
        simt_emu::launch(ckpt_restore_tile_kernel<REC>, grid, 32 * warps, smem, p);
}

/* rec: the device image of the records (tiled: [tile][entry][lane], AoS: [filter][entry]); rows: B x REC.
 * variant 0: per element (grid x 96 threads), 1: per tile (grid blocks of `warps` warps) */
extern "C" void emu_checkpoint_transform(int save, int variant, unsigned long long* rec, unsigned long long* rows, long long B, int kind,
                                         int tiled, unsigned grid, unsigned warps)
{
    const int REC = kind == 0 ? 91 : 105;
    const CkptParams p{rec, rows, B, REC, tiled};
    if (variant == 0) {
        if (save)
            simt_emu::launch(ckpt_save_elem_kernel, grid, 96, 0, p);
        else
            simt_emu::launch(ckpt_restore_elem_kernel, grid, 96, 0, p);
    } else if (REC == 91)
        tile<91>(save, p, grid, warps);
    else
        tile<105>(save, p, grid, warps);
}
