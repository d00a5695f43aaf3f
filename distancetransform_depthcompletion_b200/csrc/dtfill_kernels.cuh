// dtfill_kernels.cuh -- sm_100a kernels of the DT + nearest-neighbour fill path.
//
// Pipeline for a batch of frames [B,H,W] float32 (all device resident):
//   K1  k1_mask_rows      in -> source bit rows, per-word source prefix, row counts, validity mask (u8), row-local
//                         lists of the valid depths
//                         (reference: value_mask tools.py:8 / eval_NYU.py:115, with_value tools.py:22, net.py:131)
//   K1b k1b_scan_compact  per frame: exclusive row bases (= raster ranks, OpenCV's label initialisation),
//                         depth_list = in[valid] in raster order (tools.py:24), task list for K2
//   K2  k2_chamfer<PPL>   one warp per task: OpenCV's forward/backward 5x5 chamfer scan with label
//                         propagation (the cv2 call at tools.py:9) restructured as row-sequential,
//                         lane-parallel (min,+) scans on packed keys kept in registers, fused with the gather
//                         depth_list[lbl-1] (tools.py:25-27) and the dt / lbl outputs
//   K3  k3_sky            rows above the first source row in closed form from two rows of the scan (pipelined mode)
//   K2w k2_chamfer_wide   same scan with 64-bit keys and rows in shared memory, for frames the packed 32-bit
//                         key cannot hold (width > 1216, 2H+W too large, or >= 2^17 sources)
//   K4  k4_metrics_*      masked RMSE/MAE/iRMSE/iMAE(/REL/delta) reductions of evaluation.py:82-123, 196-239
//   K5  k5_dt_pool_*      one level of the CNN input stage's DT pooling (net.py:71-123)
//   K6  k6_outlier_removal  KITTI outlier filter (data_read.py:103-128)
//   K7  k7_edt_*          exact Euclidean feature transform (extension, SURVEY.md 8 f-4): column pass + parabola row pass
//   K8  k8_png_*          16-bit grayscale PNG files -> uint16 samples (inflate, then row unfilter), the step before K1
//                         of the uint16 entry (data_read.py:215 reads the files with PIL)
//   K9  k9_png_*          uint16 samples or float32 depth -> 16-bit grayscale PNG files (row filter, deflate per segment,
//                         offsets, pack), so that filled maps leave the device compressed
//   K10 k10_sample_bits   NYU sample coordinates -> a bitmap of 1 bit per pixel, read by K1's sampled input kind, which
//                         forms `gt * Mask` from the dense ground truth in registers (dtfill_eval_sampled)
// One header per kernel (dtfill_k*.cuh); dtfill_common.cuh holds the key format, the structs and the helpers.
//
// Key format of the fast path (SURVEY.md section 7 H1): dist:11 | order:4 | label:17.  "order" is the position
// of a candidate in OpenCV's comparison sequence, so that OpenCV's "first candidate that is strictly smaller
// wins" is a plain unsigned minimum (one VIADDMNMX per candidate); label is the 1-based raster rank of the
// source, which is also what cv2 returns with DIST_LABEL_PIXEL.  Stencil candidates use even order values:
// a stored key may then keep the 0/1 order bit left by the carry application (which is not cleared) without
// changing the outcome of any later comparison.
#pragma once
#include "dtfill_common.cuh"
#include "dtfill_k1_mask.cuh"
#include "dtfill_k1b_plan.cuh"
#include "dtfill_k2_chamfer.cuh"
#include "dtfill_k3_sky.cuh"
#include "dtfill_k2_wide.cuh"
#include "dtfill_k4_metrics.cuh"
#include "dtfill_k4_exact.cuh"
#include "dtfill_k5_pool.cuh"
#include "dtfill_k6_outlier.cuh"
#include "dtfill_k7_edt.cuh"
#include "dtfill_k8_png.cuh"
#include "dtfill_k9_png_encode.cuh"
#include "dtfill_k10_sample.cuh"
