/* nvbio_b200_debug.h -- test / tuning hooks exported by libnvbio_b200.so.  NOT part of the drop-in ABI (include/nvbio_b200.h):
 * they switch between the library's own GPU code paths so that the tests can exercise each of them and the microbenchmarks can
 * compare them; none of them changes a result.  Process-wide, not thread-safe. */
#ifndef NVBIO_B200_DEBUG_H
#define NVBIO_B200_DEBUG_H
#ifdef __cplusplus
extern "C" {
#endif

/* banded / full-matrix Gotoh: 0 = automatic, 1 = the int32 one-alignment-per-thread kernels for everything */
void nvb_debug_force_gotoh_path(int path);
/* full-matrix pair kernel occupancy variant: 0 = per-type default, 2 / 3 / 4 = minimum CTAs per SM */
void nvb_debug_full_minb(int minb);
/* full-matrix dispatch: 0 = by batch size, 1 = always the warp-per-pair kernel, 2 = never */
void nvb_debug_full_warp(int mode);
/* 0: always the run-time-format pair kernel (PFMT 0); 1 (default): the compile-time 2- / 4-bit big-endian kernels where they apply */
void nvb_debug_pair_format(int on);
/* 1 (default): the banded pair kernels keep two pattern rows in flight per thread; 0: one row per loop iteration */
void nvb_debug_pair_rows2(int on);
/* 1 (default): nvb_banded_gotoh_traceback resolves gap-free alignments from the score kernels' sink (gapless fast path) and runs the
   direction-matrix traceback only for the others; 0: the direction-matrix traceback for every alignment */
void nvb_debug_traceback_fast(int on);
/* bytes of unused dynamic shared memory added to every banded pair-kernel CTA: measures what a landing buffer (e.g. for bulk
   copies of the text windows) would cost in resident CTAs per SM */
void nvb_debug_pair_extra_smem(int bytes);

/* seed + extend composition: 0 = automatic (the per-read path when no per-hit output is requested), 1 = always the per-hit path.
   This and the two switches below are process-wide; a call reads each of them once */
void nvb_debug_pipeline_path(int path);

/* seed-match stage of the per-read path with a k-mer table: 1 (default) = seeds on k-mers with three or more occurrences are finished
   by a second kernel, 0 = one pass.  Same results; for A/B timing and tests */
void nvb_debug_seed_split(int on);

/* extension stage of the per-read path (LOCAL, constant scheme, 2-bit reads): 1 (default) = a read that equals its window on a band
   diagonal gets score = match * len and its sink without running the DP (exact: nothing can score more), 0 = every job through the
   DP kernels.  Same results; for A/B timing and tests */
void nvb_debug_perfect_shortcut(int on);

#ifdef __cplusplus
}
#endif
#endif
