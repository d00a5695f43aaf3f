/*
 * dtfill.h -- C ABI of libdtfill.so: the B200 (sm_100a) implementation of the reference's
 * "distance transform + nearest-neighbour fill" preprocessing path and of its evaluation metrics.
 *
 * The reference (placeforyiming/DistanceTransform-DepthCompletion) has no FFI layer: the boundary is the
 * Python function signature (numpy in, numpy out).  Each entry point below names the reference interface it
 * stands behind (file:line relative to the reference checkout); the ctypes binding a maintainer adds to the
 * reference is shown in INTEGRATION.md and shipped as distancetransform_depthcompletion_b200/_lib.py.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative DTFILL_E_*
 * code, with a human-readable message available from dtfill_last_error() (thread local).  No C++ exception
 * crosses the ABI.  A handle owns one CUDA device, one stream (its own, or one lent by the caller) and a
 * workspace that grows on demand; a handle is used from one host thread at a time.  Buffers named in/out
 * are owned by the caller.  "is_device" flags say whether a pointer is a device pointer on the handle's
 * device (used as is) or a host pointer (copied with cudaMemcpyAsync on the handle's stream; pinned host
 * memory makes that copy fast, see dtfill_host_alloc).  There is no CPU fallback: without a usable CUDA
 * device dtfill_create fails.
 */
#ifndef DTFILL_H_
#define DTFILL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTFILL_ABI_VERSION 9      /* 9: dtfill_eval_sampled; 8: dtfill_eval_png; 7: PNG encode (dtfill_png_encode, dtfill_png_encode_depth, dtfill_run_png_to_png); 6: PNG decode (dtfill_png_decode, dtfill_run_png, DTFILL_E_DATA); 5: sparse upload (dtfill_set_sparse_upload, dtfill_transfer_bytes); 4: dtfill_run_eval_async + dtfill_eval_totals, dtfill_edt; 3: metrics_ex, allreduce, status ring */

enum {
    DTFILL_OK = 0,
    DTFILL_E_ARG = -1,        /* bad argument (NULL pointer, non-positive size, unsupported size)            */
    DTFILL_E_CUDA = -2,       /* a CUDA runtime call failed; message has the CUDA error string               */
    DTFILL_E_INDEX = -3,      /* numpy's IndexError: a frame's labels index outside its list of valid depths */
    DTFILL_E_NOMEM = -4,
    DTFILL_E_DATA = -5        /* a file is not a supported or intact 16-bit grayscale PNG                     */
};

enum { DTFILL_METRICS_KITTI = 0, DTFILL_METRICS_NYU = 1 };

/* Number of doubles per frame written by dtfill_metrics (and length of the `sums` vector minus one). */
#define DTFILL_METRIC_COLS 9   /* mse, rmse, mae, irmse, imae, delta1, delta2, delta3, valid_count */

typedef struct dtfill_ctx dtfill_t;

/* Create / destroy a handle bound to CUDA device `device`. */
int  dtfill_create(int device, dtfill_t** out_handle);
void dtfill_destroy(dtfill_t* h);

/* Run all device work of this handle on `cuda_stream` (a cudaStream_t) instead of the handle's own
 * stream; NULL restores the handle's stream.  Used to interoperate with torch.cuda streams. */
int  dtfill_set_stream(dtfill_t* h, void* cuda_stream);

/* Block until everything queued on the handle's stream has finished. */
int  dtfill_synchronize(dtfill_t* h);

/*
 * The hot path.  For every frame b of `in` (float32 [B,H,W], dense, channel 0 already selected):
 *
 *   source(p)   = !( (float)(1.0f - in[p]) > src_thr )      value_mask of nearest_point,
 *                                                            solution_DeepNet/tools.py:8 (src_thr 0.1),
 *                                                            solution_DeepNet/eval_NYU.py:115 (src_thr 0.001)
 *   (dt, lbl)   = cv2.distanceTransformWithLabels(mask, DIST_L1, 5, DIST_LABEL_PIXEL)
 *                                                            tools.py:9, eval_NYU.py:116, demo.py:80 --
 *                 bit-exact, including which of several equidistant sources wins (OpenCV scan order)
 *   valid(p)    = in[p] > val_thr                            tools.py:22, eval_NYU.py:124, net.py:131-132
 *   depth_list  = in[valid] in raster order                  tools.py:24, eval_NYU.py:126
 *   out_depth   = depth_list[lbl - 1]  (numpy indexing, -1 = last element)   tools.py:25-27, eval_NYU.py:128-131
 *
 * Outputs (each may be NULL to skip it, except out_depth):
 *   out_depth float32 [B,H,W]   the filled depth  (return value of DT_complete_batch tools.py:13-35 and of
 *                               Distance_Transform eval_NYU.py:120-133)
 *   out_dt    float32 [B,H,W]   the distance channel (first return value of nearest_point tools.py:10);
 *                               65533.0 where no source is reachable, like OpenCV
 *   out_lbl   int32   [B,H,W]   the label map (second return value of nearest_point)
 *   out_mask  uint8   [B,H,W]   validity ("DT-pooling") mask in[p] > val_thr (net.py:131-132), 0/1
 *   out_counts int32  [B,2]     per frame: number of sources, number of valid pixels (host pointer when
 *                               out_is_device == 0, device pointer otherwise; may be NULL)
 *
 * dtfill_run waits for completion.  If some frame's labels index outside its depth_list (no valid pixel at
 * all, or more sources than valid pixels) the reference raises IndexError: the call returns DTFILL_E_INDEX and
 * stores the first such frame in *first_bad_frame (other frames' outputs are still written).
 * dtfill_run_async only enqueues on the handle's stream (device pointers only); call dtfill_status afterwards.
 */
int dtfill_run(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W,
               float src_thr, float val_thr,
               float* out_depth, float* out_dt, int32_t* out_lbl, uint8_t* out_mask, int32_t* out_counts,
               int out_is_device, int* first_bad_frame);

int dtfill_run_async(dtfill_t* h, const float* in_dev, int B, int H, int W, float src_thr, float val_thr,
                     float* out_depth_dev, float* out_dt_dev, int32_t* out_lbl_dev, uint8_t* out_mask_dev,
                     int32_t* out_counts_dev);

/* The same path fed with the frames as the KITTI depth PNGs hold them (SURVEY.md 8(f-3)): uint16 samples,
 * depth = sample / 256 (data_read.py:215 `depth_png.astype(np.float32) / 256.`, exact in float32), laid out
 * [B, H_in, W]; rows [crop_top, H_in) of every frame are the frame that is processed (train.py:211, eval.py:156
 * `lidar[:, 96:, :, :]`), so H = H_in - crop_top in every output.  The decode and the crop happen inside the first
 * kernel: the input costs 2 bytes per pixel of HBM traffic instead of 4, and no float32 copy of the input exists
 * unless out_lidar (nullable, float32 [B,H,W]: the decoded, cropped frames the reference hands to its CNN next to
 * the filled depth) asks for it.  All other arguments, outputs and errors as dtfill_run / dtfill_run_async. */
int dtfill_run_u16(dtfill_t* h, const uint16_t* in, int in_is_device, int B, int H_in, int W, int crop_top,
                   float src_thr, float val_thr,
                   float* out_lidar, float* out_depth, float* out_dt, int32_t* out_lbl, uint8_t* out_mask,
                   int32_t* out_counts, int out_is_device, int* first_bad_frame);

int dtfill_run_u16_async(dtfill_t* h, const uint16_t* in_dev, int B, int H_in, int W, int crop_top,
                         float src_thr, float val_thr,
                         float* out_lidar_dev, float* out_depth_dev, float* out_dt_dev, int32_t* out_lbl_dev,
                         uint8_t* out_mask_dev, int32_t* out_counts_dev);

/*
 * The step in front of dtfill_run_u16: KITTI depth PNG files (data_read.py:215 `Image.open(f)`) decoded on the device
 * (kernels k8_png_inflate, k8_png_unfilter; dtfill_k8_png.cuh).  Only non-interlaced 16-bit grayscale PNGs are supported
 * (any row filters, any DEFLATE content, the zlib stream split over any IDAT chunks, ancillary chunks skipped); chunk
 * CRC-32s are not checked, the zlib stream's Adler-32 is.  Per-frame status codes (int32):
 *   0 ok, 1 bad signature, 2 unsupported IHDR, 3 size differs from (H, W), 4 broken or truncated chunk structure or no
 *   IDAT, 5 bad zlib header, 6 invalid DEFLATE data (including running out of input), 7 decompressed size != H*(1+2W),
 *   8 filter type > 4, 9 Adler-32 mismatch.
 * A failed frame's samples are zero.  H * (1 + 2 W) < 2^28.
 *
 * dtfill_png_decode: B files packed back to back in `data`; file b is data[offsets[b], offsets[b+1]) (offsets int64
 * [B+1], on the same side as data).  Writes uint16 [B,H,W] native-endian samples and out_status int32 [B] (nullable when
 * the outputs are host pointers).  Enqueue-only when input and outputs are all device pointers; otherwise the call
 * waits and returns DTFILL_E_DATA with *first_bad_frame when a frame failed (the other frames are still written).
 */
int dtfill_png_decode(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H, int W,
                      uint16_t* out, int32_t* out_status, int out_is_device, int* first_bad_frame);

/* Decode into the handle's workspace, then exactly the dtfill_run_u16 path (crop_top, thresholds, outputs, IndexError):
 * the decoded samples never leave the device.  Synchronous.  A decode failure (DTFILL_E_DATA, first failed frame) wins
 * over IndexError. */
int dtfill_run_png(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H_in, int W,
                   int crop_top, float src_thr, float val_thr, float* out_lidar, float* out_depth, float* out_dt,
                   int32_t* out_lbl, uint8_t* out_mask, int32_t* out_counts, int out_is_device, int* first_bad_frame);

/* Host-only test hook (no handle, no GPU), like dtfill_debug_compact: the same decode of one file of nbytes, run serially
 * on the CPU.  Returns the status code above (samples of a failed file are zero), or -1 for bad arguments. */
int dtfill_debug_png_decode_host(const uint8_t* png, long nbytes, int H, int W, uint16_t* out);

/*
 * The way out, the mirror of dtfill_png_decode: frames encoded on the device as 16-bit grayscale PNG files (kernels
 * k9_png_filter, k9_png_deflate, k9_png_offsets, k9_png_pack; dtfill_k9_png_encode.cuh), so that only compressed bytes
 * cross the link.  Every file is colour type 0, bit depth 16, non-interlaced: signature, IHDR, an IDAT holding the zlib
 * header, one IDAT per 16 rows (fixed-Huffman DEFLATE blocks, or stored blocks where those would be larger, ending
 * byte-aligned), an IDAT holding the Adler-32, IEND.  Rows are filtered with libpng's heuristic (least sum of absolute
 * signed differences, ties to the lowest filter type).  The bytes are a pure function of the samples: the host hook
 * below writes identical files.  H * (1 + 2 W) < 2^28.
 *
 * dtfill_png_encode_bound: worst-case bytes of one file (every segment stored, plus all chunk overhead); DTFILL_E_ARG
 * for an unsupported size.
 * dtfill_png_encode: uint16 samples [B,H,W] -> B files back to back in out; out_offsets int64 [B+1] (file b =
 * out[off[b], off[b+1])), the layout dtfill_png_decode takes.  out_capacity must be >= B * dtfill_png_encode_bound(H, W)
 * (else DTFILL_E_ARG and nothing is written).  Enqueue-only when input and outputs are all device pointers; otherwise
 * the call waits and copies only offsets[B] bytes device -> host.
 * dtfill_png_encode_depth: float32 depth in metres [B,H,W]; each sample is
 *     sample = clip(nan_to_num(fl32(d * 256), nan=0, posinf=65535), 0, 65535) truncated toward zero,
 * applied inside k9_png_filter (no uint16 copy exists).  For d in [0, 65535/256] this is (d * 256).astype(np.uint16),
 * the usual way KITTI depth is written; on d = k/256 (a frame decoded from a PNG) it is the identity.
 */
int64_t dtfill_png_encode_bound(int H, int W);
int dtfill_png_encode(dtfill_t* h, const uint16_t* in, int in_is_device, int B, int H, int W,
                      uint8_t* out, int64_t out_capacity, int64_t* out_offsets, int out_is_device);
int dtfill_png_encode_depth(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W,
                            uint8_t* out, int64_t out_capacity, int64_t* out_offsets, int out_is_device);

/* dtfill_run_png, then the filled depth encoded as by dtfill_png_encode_depth: PNG files in, PNG files of
 * H = H_in - crop_top rows out.  The decoded samples and the float32 depth never leave the device.  Synchronous.
 * DTFILL_E_DATA (first failed frame) wins over DTFILL_E_INDEX; with either, the files of all frames are still written. */
int dtfill_run_png_to_png(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H_in,
                          int W, int crop_top, float src_thr, float val_thr, uint8_t* out, int64_t out_capacity,
                          int64_t* out_offsets, int out_is_device, int* first_bad_frame);

/* Host-only test hook (no handle, no GPU): the same encoder run serially on the CPU.  capacity >= the bound.  Returns the
 * file size, or -1 for bad arguments. */
long dtfill_debug_png_encode_host(const uint16_t* samples, int H, int W, uint8_t* out, long capacity);
/* Host-only test hook: the depth -> sample rule of dtfill_png_encode_depth (the function k9_png_filter runs) on n floats.
 * Returns 0, or -1 for bad arguments. */
int dtfill_debug_depth_samples_host(const float* depth, long n, uint16_t* out);

/* Synchronise and report the outcome of EVERY dtfill_run_async / dtfill_run_u16_async since the previous dtfill_status:
 * DTFILL_OK, or DTFILL_E_INDEX with *first_bad_frame = the smallest frame index (within its call) that any of those
 * calls flagged.  Each call owns a slot of a status ring, so no call's verdict is lost however many calls are in
 * flight or how deep the pipeline is.  *kernel_launches receives the number of kernels launched by the last call. */
int dtfill_status(dtfill_t* h, int* first_bad_frame, int* kernel_launches);

/*
 * Evaluation metrics of evaluation.py for B frame pairs:
 *   mode DTFILL_METRICS_KITTI  Result.evaluate      evaluation.py:82-123  (metres -> mm, 1/km)
 *   mode DTFILL_METRICS_NYU    Result_NYU.evaluate  evaluation.py:196-239 (no scaling, REL, delta1..3)
 * pred float32 [B,H,W]; gt float64 (gt_is_f64 != 0, data_read.py:223) or float32 [B,H,W].
 * per_frame (nullable) double [B][DTFILL_METRIC_COLS] = mse, rmse, mae, irmse, imae, delta1, delta2, delta3,
 * valid_count (delta* are 0 in KITTI mode).  sums (nullable) double [DTFILL_METRIC_COLS + 1] = column sums of
 * per_frame over the B frames followed by B -- the running totals eval.py:212-232 / eval_NYU.py:207-229 keep
 * (mean of per-frame metrics).  Both are host pointers unless out_is_device; the call waits for completion
 * when they are host pointers.
 */
int dtfill_metrics(dtfill_t* h, const float* pred, const void* gt, int gt_is_f64, int in_is_device,
                   int B, int H, int W, int mode, double* per_frame, double* sums, int out_is_device);

/* Summation order of dtfill_metrics / dtfill_metrics_ex.  1 (default; DTFILL_METRICS_EXACT=0 for the other): the per-pixel
 * terms of the valid pixels are compacted in raster order and summed in the order of numpy's pairwise add.reduce, in the
 * dtype numpy uses (float32 for a float32 ground truth, float64 for a float64 one), so every metric equals the
 * reference's bit for bit.  0: fixed-order float64 sums straight from the frames (one pass, ~5x faster): 1e-9 relative
 * for a float64 ground truth, ~1e-5 for a float32 one (numpy's own float32 rounding).  The fused sweep entry
 * dtfill_run_eval_async always uses the one-pass sums. */
int dtfill_set_metrics_exact(dtfill_t* h, int enabled);

/* dtfill_metrics with running totals: accumulate != 0 adds this batch's column sums and frame count to the device
 * vector `sums` (out_is_device required) instead of overwriting it -- the `+=` of eval.py:212-232 /
 * eval_NYU.py:207-229, one batch per call, no host synchronisation. */
int dtfill_metrics_ex(dtfill_t* h, const float* pred, const void* gt, int gt_is_f64, int in_is_device,
                      int B, int H, int W, int mode, double* per_frame, double* sums, int out_is_device,
                      int accumulate);

/*
 * The evaluation loop of the reference's KITTI ablation notebook, from the files (SURVEY.md section 3 C):
 *     lidar = png.astype(float32) / 256        data_read.py:215
 *     gt    = png / 256.  (float64)            data_read.py:223
 *     Result().evaluate(Distance_Transform(lidar, src_thr), gt)
 * for B pairs of 16-bit grayscale PNG files of H x W (no crop), host files laid out as for dtfill_png_decode.  The 2B
 * files are decoded in one launch, the LiDAR frames filled as by dtfill_run_u16, and the metrics computed against the
 * ground-truth samples in KITTI mode and numpy's summation order (whatever dtfill_set_metrics_exact says), so that
 * per_frame [B][DTFILL_METRIC_COLS] and sums [DTFILL_METRIC_COLS + 1] (host, nullable; layout of dtfill_metrics) equal
 * the reference's bit for bit.  No per-pixel data crosses the link.  Synchronous.
 * Errors, frame by frame as the loop meets them: DTFILL_E_DATA for the first frame with a file that fails to decode
 * (LiDAR before ground truth at the same frame), which wins over DTFILL_E_INDEX for the first LiDAR frame
 * Distance_Transform rejects (no valid depth, exactly one valid depth, labels outside the list of valid depths);
 * *first_bad_frame receives the frame.  On an error the contents of per_frame and sums are unspecified.
 */
int dtfill_eval_png(dtfill_t* h, const uint8_t* lidar, const int64_t* lidar_offsets, const uint8_t* gt,
                    const int64_t* gt_offsets, int B, int H, int W, float src_thr, float val_thr, double* per_frame,
                    double* sums, int* first_bad_frame);

/*
 * The evaluation loop of the reference's NYU script (eval_NYU.py:138-254, data_read.py:337-371) from dense ground truth:
 *     Mask = zeros(H, W);  Mask[rows_b, cols_b] = 1                 data_read.py:360-364 (duplicates collapse)
 *     pred = Distance_Transform(gt_b * Mask, src_thr)               eval_NYU.py:120-133
 *     Result_NYU().evaluate(pred[r0:r1, c0:c1], gt_b[r0:r1, c0:c1]) eval_NYU.py:202-207
 * for the B frames of gt (float32 [B,H,W]; a device pointer when gt_is_device, used in place and never copied, else host).
 * Frame b's sample coordinates are rows[k], cols[k] for k in [sample_offsets[b], sample_offsets[b+1]) (int32, int64
 * offsets [B+1]; device pointers when coords_are_device, in which case every index from the smallest to the largest
 * offset must lie within rows and cols: the device can check the coordinates' values, not the arrays' length).  The
 * coordinates become a bitmap of 1 bit per pixel
 * (k10_sample_bits), K1 forms `gt * Mask` from the ground truth and the bitmap in registers (out_lidar, host, nullable:
 * that sparse frame [B,H,W]), the fill keeps the filled depth on the device, and the NYU-mode metrics of the window are
 * computed against the same ground-truth buffer in numpy's summation order (whatever dtfill_set_metrics_exact says), so
 * that per_frame [B][DTFILL_METRIC_COLS] and sums [DTFILL_METRIC_COLS + 1] (host, nullable; layout of dtfill_metrics) equal
 * the reference's bit for bit.  With a resident ground truth only the coordinates and offsets go up and only the counts and
 * the metrics come back (dtfill_transfer_bytes).  Synchronous; strict order on the handle's stream.
 * Errors: DTFILL_E_ARG for a window that is empty or leaves the frame, decreasing offsets (a negative count) and
 * coordinates outside [0,H) x [0,W) (host coordinates are checked on the host, device ones on the device; *first_bad_frame
 * receives the frame); then DTFILL_E_INDEX for the first frame Distance_Transform rejects (no valid depth, exactly one
 * valid depth, labels outside the list of valid depths).  On an error the contents of the outputs are unspecified.
 */
int dtfill_eval_sampled(dtfill_t* h, const float* gt, int gt_is_device, int B, int H, int W, const int32_t* rows,
                        const int32_t* cols, const int64_t* sample_offsets, int coords_are_device, int r0, int r1, int c0,
                        int c1, float src_thr, float val_thr, float* out_lidar, double* per_frame, double* sums,
                        int* first_bad_frame);

/*
 * One step of an evaluation sweep, fused (BASELINE.json configs[4]; the loop body of eval.py:212-232: DT_complete_batch,
 * Result.evaluate per frame, running `+=` of the per-frame metrics): dtfill_run_async followed, on the same internal
 * stream, by the metric kernels on the filled depth against gt_dev (float64 when gt_is_f64, else float32, [B,H,W]).  The
 * column sums of the per-frame metrics and the frame count are added to running totals the handle keeps per pipeline
 * lane, so in pipelined mode consecutive steps overlap like plain fills and nothing synchronises with the host.
 * dtfill_eval_totals collects them: it joins the calls in flight (dtfill_flush) and writes (accumulate == 0) or adds
 * (accumulate != 0) the totals [DTFILL_METRIC_COLS + 1] to the device vector sums_dev on the handle's stream, in a fixed
 * order, and clears the handle's running totals -- ready for dtfill_allreduce_sums.  Bad frames (IndexError) are
 * reported by dtfill_status as for dtfill_run_async; their metrics are undefined.
 */
int dtfill_run_eval_async(dtfill_t* h, const float* in_dev, const void* gt_dev, int gt_is_f64, int B, int H, int W,
                          float src_thr, float val_thr, int mode,
                          float* out_depth_dev, float* out_dt_dev, int32_t* out_lbl_dev, uint8_t* out_mask_dev,
                          int32_t* out_counts_dev);
int dtfill_eval_totals(dtfill_t* h, double* sums_dev, int accumulate);

/*
 * Multi-GPU (SURVEY.md 8(e)): frames shard contiguously over one process per GPU with no data-path exchange; the only
 * collective is a sum all-reduce of the metric totals {sum rmse_f, sum mae_f, ..., n_frames} (mean-of-per-frame-metrics
 * rule of eval.py:212-232, 252-259).  dtfill_allreduce_sums issues ncclAllReduce(sum, float64, in place) over `n`
 * doubles at the device pointer `sums_dev` on the handle's stream, i.e. right behind the kernels of dtfill_metrics(_ex)
 * that produced them; nothing is synchronised on the host.  `nccl_comm` is an ncclComm_t: one the caller already owns,
 * or one made by dtfill_comm_create from the 128-byte ncclUniqueId that rank 0 obtained with dtfill_nccl_unique_id and
 * sent to the other ranks by any means (torch.distributed broadcast in sharding.py).  libnccl.so.2 is resolved with
 * dlopen at the first of these calls (DTFILL_NCCL_LIB overrides the name); without it they return DTFILL_E_CUDA.
 */
#define DTFILL_NCCL_ID_BYTES 128
int dtfill_nccl_unique_id(void* out_id /* DTFILL_NCCL_ID_BYTES */);
int dtfill_comm_create(dtfill_t* h, const void* id, int nranks, int rank, void** out_nccl_comm);
int dtfill_comm_destroy(void* nccl_comm);
int dtfill_allreduce_sums(dtfill_t* h, void* nccl_comm, double* sums_dev, int n);

/*
 * DT pooling of the CNN input stage: generate_multi_channel (solution_DeepNet/net.py:83-123, identical in all
 * model classes) with the weights of create_weight_matrix (net.py:71-81).  data, mask: float32 [B,H,W] (the
 * reference's [B,H,W,1]); data is the sparse depth already divided by scale_range and multiplied by the mask
 * (net.py:467-486), mask the validity mask (net.py:464-465).  Writes levels 2..scale_num (1 <= scale_num <= 4)
 * into out [scale_num-1][B,H,W]: level k is pooled from level k-1 with mask = level k-1 > 0.001 (net.py:95-96).
 * table_size odd, <= 15.  Waits for completion when out is a host pointer.
 */
int dtfill_dt_pool(dtfill_t* h, const float* data, const float* mask, int in_is_device, int B, int H, int W,
                   int table_size, int scale_num, float* out, int out_is_device);
/* Same, and the masks the levels are pooled with (SURVEY.md 8 a-5): out_masks (nullable) uint8 [scale_num-1][B,H,W],
 * out_masks[k] = out[k] > 0.001 (net.py:95-96, :105-106) = the "DT-pooling mask" of level k+2, a Chebyshev
 * dilation of the validity mask by (table_size / 2) pixels per level. */
int dtfill_dt_pool_ex(dtfill_t* h, const float* data, const float* mask, int in_is_device, int B, int H, int W,
                      int table_size, int scale_num, float* out, uint8_t* out_masks, int out_is_device);

/* The older variant of the pooling in demo.py:65-149 (no mask; weights 10 ** (T - |dy| - |dx|), demo.py:65-76; the selected
 * pixels are those whose value times weight equals the window's maximum, demo.py:120-121; denominator
 * 1e-6 + count_nonzero of the selected values, :122).  data float32 [B,H,W]; out float32 [scale_num - 1][B,H,W] = levels
 * 2..scale_num before the division by scale_range (the Python mirror divides).  table_size odd, <= 15 (demo.py uses 11). */
int dtfill_dt_pool_demo(dtfill_t* h, const float* data, int in_is_device, int B, int H, int W, int table_size,
                        int scale_num, float* out, int out_is_device);

/* KITTI outlier filter outlier_removal (data_read.py:103-128), the step just before the path: in, out float32
 * [B,H,W]; a depth more than 1.0 m farther than the average of the valid depths in its 7 x 7 diamond is zeroed. */
int dtfill_outlier_removal(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, float* out,
                           int out_is_device);

/*
 * EXTENSION (SURVEY.md 8 f-4; no reference function stands behind it: every call site of the reference computes the
 * 5x5 chamfer transform above, tools.py:9): the exact Euclidean feature transform of the same source mask,
 * source(p) = !((float)(1.0f - in[p]) > src_thr).  Separable: a row pass (one warp per row: ballots of the predicate,
 * nearest source column per pixel from bit scans), then down every column the lower envelope of the parabolas
 * (y - y')^2 + h(y',x)^2, one thread per column so that a warp's accesses are coalesced.  in float32 [B,H,W]; out_d2 int32
 * [B,H,W] = squared distance to the nearest source (2^31 - 1 for a frame without sources); out_idx (nullable) int32
 * [B,H,W] = y' * W + x' of a source at that distance (-1 if none): among several sources at the minimal distance the first
 * in raster order.  H <= 4096, W <= 25600.
 * Oracle: scipy.ndimage.distance_transform_edt (squared distances identical; an index is checked by the distance it
 * attains).  Waits for completion when the outputs are host pointers.
 */
int dtfill_edt(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, float src_thr,
               int32_t* out_d2, int32_t* out_idx, int out_is_device);

/* Pipelined mode.  depth 1 (default): strict stream order -- when a call's work completes, in stream order, its
 * outputs are final.  depth 2..4: consecutive dtfill_run_async calls may overlap: a call runs on one of `depth` internal
 * streams, behind whatever was queued on the handle's stream before it and behind the call `depth` back (which used the
 * same workspace), so the HBM-bound first stage of one batch overlaps the ALU-bound scan of the previous one.
 * The handle's stream sees the outputs only after dtfill_flush (or dtfill_status / dtfill_synchronize, which
 * flush).  Callers must not reuse a call's output buffers for the next call. */
int dtfill_set_pipeline_depth(dtfill_t* h, int depth);
int dtfill_flush(dtfill_t* h);

/* Frames are split into bands of rows that one warp each processes independently (exact: every band is
 * extended by a halo derived from a guaranteed upper bound of the distances inside it).  cap > 0: target cost of
 * one band in row steps; 0: never split; -1 (default): chosen from the batch size and the SM count. */
int dtfill_set_band_cap(dtfill_t* h, int cap);

/* Rows above a frame's first source row are not scanned: their distances and labels follow in closed form from two
 * rows of the scan (kernel k3_sky; exact, see the kernel's header).  rows = least number of such rows for which
 * this is done; 0: never, every row goes through the scan; -1 (default): 8 (the tallest tiles of a KITTI frame lose
 * a third of their row steps: a single frame takes 0.137 instead of 0.209 ms on a B200). */
int dtfill_set_sky_min(dtfill_t* h, int rows);

/* A batch is processed as n sub-batches on forked streams so that the ALU-bound scan of one overlaps the
 * HBM-bound predicate pass of the next (joined back into the handle's stream before the call returns / the
 * async call's work is complete).  n <= 0: automatic (4 for batches of 64 frames or more). */
int dtfill_set_subbatches(dtfill_t* h, int n);

/* Introspection for tests and tuning: copies the task list (tiles) the planner produced for the last run.
 * Each task is 12 int32: frame, lo, hi, r0, r1, kind, scratch_off, fstart, clo, c0, c1, reserved (see
 * dtfill_kernels.cuh struct Task; kind 3 = unused slot).  Returns the number of tasks written (<= max_tasks),
 * or a negative error code. */
int dtfill_debug_get_tasks(dtfill_t* h, int32_t* out, int max_tasks);
/* Raw status words of the last call (n <= 64): [0] first bad frame, [1] wide tasks, [4..] planner phase clocks when
 * the library is built with -DDTFILL_PLANNER_CLOCKS. */
int dtfill_debug_read_status(dtfill_t* h, int32_t* out, int n);

/* Tuning only: the stages whose bit is set are not launched by the following runs (bit 0 k1_mask_rows, 1 k1b_scan_compact,
 * 2 k2_chamfer*, 3 k3_sky), so that one stage can be timed against the workspace a complete run left behind.  Outputs
 * of such runs are meaningless. */
int dtfill_debug_set_skip(dtfill_t* h, int mask);

/* Per-kernel timing of the hot path with CUDA events recorded on the handle's stream between the launches of
 * dtfill_run / dtfill_run_async (off by default).  dtfill_kernel_times waits for the last run and writes the
 * milliseconds of k1_mask_rows, k1b_scan_compact, k2_chamfer, k2_chamfer_wide, k3_sky into ms[0..4]. */
#define DTFILL_NUM_KERNELS 5
int dtfill_set_profiling(dtfill_t* h, int enabled);
int dtfill_kernel_times(dtfill_t* h, float* ms);

/* Pageable host buffers handed to dtfill_run / dtfill_run_u16 (what numpy allocates: the reference's contract,
 * tools.py:13-35) are staged through pinned mirrors owned by the handle: `threads` host threads per direction copy a
 * slice into / out of the mirror while the DMA engines move the previous slices and the kernels run, so a pageable
 * caller gets close to the PCIe limit.  -1 (default): three quarters of the usable CPUs, clamped to 2..12; 0: no staging (the
 * driver stages the copies on the calling thread).  Buffers that are already pinned (dtfill_host_alloc,
 * cudaHostRegister) are copied directly in either case. */
int dtfill_set_stage_threads(dtfill_t* h, int threads);

/* Sparse upload (on by default; DTFILL_SPARSE_UPLOAD=0).  dtfill_run with a PAGEABLE float32 host input: the host threads
 * that would copy a slice into a page-locked mirror compact it instead into (pixel index, value) pairs of the pixels that
 * are a source (tools.py:8) or valid (tools.py:22) -- the only pixels whose value the path ever reads -- and the device
 * rebuilds the dense slice from zeros + pairs in front of the first kernel.  Results are bit-identical; it applies when
 * 0.0f is neither a source nor valid (true for the reference's thresholds 0.1 / 0.001 and 0.1) and falls back to the
 * dense copy for a slice with more than 25 % such pixels.  dtfill_transfer_bytes reports what the last synchronous call
 * with host buffers moved over the link in each direction. */
int dtfill_set_sparse_upload(dtfill_t* h, int enabled);
int dtfill_transfer_bytes(dtfill_t* h, unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);
/* Host-only test hook (needs neither a handle nor a GPU): the compaction of the sparse upload on src[0..n): indices and
 * value bits of the pixels that are a source or valid for the given thresholds, in order; returns their number, or -1 on
 * bad arguments (cap >= n + 16 entries are needed in idx and val: the packed stores write whole vectors). */
long dtfill_debug_compact(const float* src, long n, float src_thr, float val_thr, uint32_t* idx, uint32_t* val, long cap);

/* Pinned host memory for fast host<->device copies (cudaHostAlloc / cudaFreeHost). */
int  dtfill_host_alloc(void** out_ptr, size_t bytes);
void dtfill_host_free(void* ptr);

/* Message describing the last error on this thread ("" if none). */
const char* dtfill_last_error(void);

/* DTFILL_ABI_VERSION the library was built with. */
int dtfill_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DTFILL_H_ */
