/*
 * pmp_b200.h -- C ABI of the B200-native partition-map prediction library (libpmp_b200.so).
 *
 * The reference (AolinFeng/PMP-VVC-TIP2023) has no FFI of its own: its boundary is four
 * nn.Module classes, four Python functions and the PartitionMat text format (SURVEY.md
 * section 8(b)).  Every entry point below names the reference interface it replaces
 * (paths relative to /root/reference).  The Python package pmp_vvc_tip2023_b200 binds these
 * with ctypes and re-exposes the reference's own names (INTEGRATION.md shows the stubs).
 *
 * Conventions: plain pointers and sizes only; all data pointers are DEVICE pointers unless
 * the name ends in _host; every call is asynchronous on `stream` (a cudaStream_t passed as
 * void*; NULL = legacy default stream) unless documented otherwise; return 0 on success, a
 * negative pmp_status on failure with a message available from pmp_last_error() (thread
 * local).  A handle is bound to one device and must not be shared between host threads.
 * There is no CPU fallback: without a CUDA device pmp_create fails.
 */
#ifndef PMP_B200_H
#define PMP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMP_B200_VERSION 200 /* 0.2.0 */

typedef struct pmp_handle pmp_handle;

enum pmp_status {
    PMP_OK = 0,
    PMP_ERR_ARG = -1,      /* bad argument */
    PMP_ERR_CUDA = -2,     /* CUDA runtime/driver error (message has the detail) */
    PMP_ERR_NO_DEVICE = -3,
    PMP_ERR_STATE = -4,    /* unknown weight set, wrong net kind ... */
    PMP_ERR_UNSUPPORTED = -5,
    PMP_ERR_ABORTED = -6   /* a callback of pmp_predict_stream(_multi) returned non-zero (message names it and its value) */
};

/* Net kinds: Model_QBD.py:59 Luma_Q_Net, :100 Luma_MSBD_Net, :157 Chroma_Q_Net, :198 Chroma_MSBD_Net */
enum pmp_net { PMP_NET_LUMA_Q = 0, PMP_NET_LUMA_MSBD = 1, PMP_NET_CHROMA_Q = 2, PMP_NET_CHROMA_MSBD = 3 };

/* Conv engines.  TC: tcgen05/TMEM implicit-GEMM with TMA-fed halo tiles and split-precision
 * (hi+lo 16-bit) operands, fp32 accumulate; SIMT: exact fp32 CUDA-core direct convolution. */
enum pmp_engine { PMP_ENGINE_SIMT = 0, PMP_ENGINE_TC = 1 };
/* 16-bit operand format of the TC engine */
enum pmp_tc_dtype { PMP_TC_FP16 = 0, PMP_TC_BF16 = 1 };
/* block input dtype */
enum pmp_in_dtype { PMP_IN_U8 = 0, PMP_IN_F32 = 1 };

int pmp_version(void);
const char *pmp_last_error(void);

/* Lifetime.  pmp_create binds to `device` and creates no streams; pmp_predict_host / pmp_predict_stream create two
 * streams and pinned staging buffers on their first call, which pmp_destroy frees.  A new handle runs PMP_ENGINE_TC / PMP_TC_FP16. */
int pmp_create(int device, pmp_handle **out);
void pmp_destroy(pmp_handle *h);
int pmp_set_engine(pmp_handle *h, int engine, int tc_dtype);
int pmp_get_engine(pmp_handle *h);
/* Tolerance of the near-threshold report in pmp_run_component / pmp_map2partition flags bits 1..3 (default 1e-2, the
 * north-star parity bar on map values). */
int pmp_set_near_tol(pmp_handle *h, float near_tol);
/* Sticky fp16 range guard of the TC engine: number of epilogue threads that produced an activation beyond +-65504 with
 * fp16 operands since creation / the last reset (the hi/lo split clamps there, so a non-zero count means wrong results:
 * switch the handle to PMP_TC_BF16).  Synchronises the device. */
int pmp_saturation_count(pmp_handle *h, long long *count_host, int reset);
/* Number of kernels launched by this handle since creation (bench.py's gpu_launches). */
long long pmp_launch_count(pmp_handle *h);
/* Name/elapsed-ms of per-kernel-class CUDA-event timers (enabled with pmp_profile(h,1)); see bench.py. */
int pmp_profile(pmp_handle *h, int enable);
int pmp_profile_read(pmp_handle *h, int idx, char *name, int name_len, double *ms, long long *launches,
                     double *flops, double *bytes);

/* ---- weights ---------------------------------------------------------------------------
 * Replaces torch.load + load_state_dict + .cuda() of Inference_QBD.py:33-46,:221-224.
 * tensors_host[i] points at HOST fp32 data of the i-th parameter in the reference's
 * state_dict order for `net` (pmp_vvc_tip2023_b200/netspec.py lists names and shapes);
 * numel[i] is checked against the expected size.  Packs once into device operand layouts for
 * both engines (synchronous).  Returns the weight-set id in *wset. */
int pmp_weights_create(pmp_handle *h, int net, const float *const *tensors_host, const int64_t *numel,
                       int n_tensors, int *wset);
int pmp_weights_destroy(pmp_handle *h, int wset);
/* Same from an exported weight file (.pmpw, python -m pmp_vvc_tip2023_b200.export_weights), read on the host: a 64-byte
 * header ("PMPW0001", int32 net kind, int32 tensor count, int64 total floats, uint64 FNV-1a-64 of everything after the
 * header), one record per tensor (int32 name length, name, int32 ndim, int32 dims[ndim]), zero padding to a multiple of
 * 64 bytes, then the fp32 data in record order, all little-endian.  Every field is checked against the library's own
 * parameter table; any mismatch returns PMP_ERR_ARG, creates no weight set and names the path and the first field that
 * failed.  *net_out (may be NULL) receives the net kind, *wset the weight-set id. */
int pmp_weights_load(pmp_handle *h, const char *path, int *net_out, int *wset);

/* ---- nets ------------------------------------------------------------------------------
 * pmp_forward_q      == Luma_Q_Net.forward / Chroma_Q_Net.forward      (Model_QBD.py:78-98,:176-196)
 * pmp_forward_msbd   == Luma_MSBD_Net.forward / Chroma_MSBD_Net.forward (Model_QBD.py:127-155,:225-253)
 * blocks: [B,1,68,68] (luma) or [B,3,34,34] (chroma), u8 or f32 (values 0..255, no normalisation).
 * qt_out / qt: [B,1,8,8] f32 (raw, un-rounded).  out0..2: [B,2,16,16] f32 (ch0 cumulative MTT depth,
 * ch1 direction). */
int pmp_forward_q(pmp_handle *h, int wset, const void *blocks, int in_dtype, int B, float *qt_out, void *stream);
int pmp_forward_msbd(pmp_handle *h, int wset, const void *blocks, int in_dtype, const float *qt, int B,
                     float *out0, float *out1, float *out2, void *stream);
/* pmp_predict_maps == one batch of Metrics.inference_pre_QBD (Metrics.py:387-419):
 * Q net -> MSBD net (fed the raw qt) -> regroup.  qt [B,1,8,8], bt [B,3,16,16] (ch0 of out0/1/2),
 * dire [B,3,16,16] (ch1 of out0/1/2), all f32 device. */
int pmp_predict_maps(pmp_handle *h, int wset_q, int wset_msbd, const void *blocks, int in_dtype, int B,
                     float *qt, float *bt, float *dire, void *stream);

/* ---- post-process + decode ---------------------------------------------------------------
 * pmp_qt_postprocess == Metrics.eli_structual_error (Metrics.py:612-637).  qt [B,1,8,8] f32 ->
 * out_f32 [B,1,8,8] f32 holding 0..3 and/or out_u8 [B,64] (either may be NULL). */
int pmp_qt_postprocess(pmp_handle *h, const float *qt, int B, float *out_f32, uint8_t *out_u8, void *stream);
/* pmp_map2partition == Map2Partition.map_to_parititon over a batch (Map2Partition.py:98-373).
 * qt_u8 [B,64] values 0..3 (post-processed), bt/dire [B,3,16,16] f32 (un-rounded), chroma_factor 1|2.
 * hor/ver [B,16,16] u8 {0,1}; dire_out [B,3,16,16] i8 {-1,0,1}; flags [B] u32 (may be NULL):
 * bit0 = the argmin over candidate partitions had a runner-up within the float32 evaluation noise
 * of the reference (result may legitimately differ from a float32 evaluation); bit1 = a depth value lies
 * within near_tol of a rounding threshold k+0.5 (np.round, Map2Partition.py:104); bit2 = a direction
 * value lies within near_tol of +-0.5 (th_round, :30-35,:105); bit3 = a 2x2-pooled raw qt value lies
 * within near_tol of 0.5/1.5/2.5 (Metrics.py:631-632; only when qt_raw is given); bits 4..6 = the tests of
 * bits 1..3 at the tighter tolerance near_tol / 100; bits 8.. = number of MTT regions decoded.
 * near_tol = the handle's (pmp_set_near_tol). */
int pmp_map2partition(pmp_handle *h, const uint8_t *qt_u8, const float *bt, const float *dire, int B,
                      int chroma_factor, uint8_t *hor, uint8_t *ver, int8_t *dire_out, uint32_t *flags,
                      void *stream);
/* Same with the constructor thresholds of Map_to_Partition (Map2Partition.py:100: lamb1..lamb5 as 5 doubles, NULL = the
 * reference defaults 0.7, 0.7, 1.5, 0.3, 0.7), the raw qt maps [B,64] f32 for flags bit3 (may be NULL) and an explicit
 * near_tol. */
int pmp_map2partition_ex(pmp_handle *h, const uint8_t *qt_u8, const float *bt, const float *dire, int B,
                         int chroma_factor, const double *lamb, const float *qt_raw, float near_tol, uint8_t *hor,
                         uint8_t *ver, int8_t *dire_out, uint32_t *flags, void *stream);
/* pmp_assemble_frames == the scatter + per-frame vector order of get_sequence_partition_for_VTM
 * (Map2Partition.py:389-412).  Blocks are frame-major raster (bh x bw per frame).  out: per frame
 * hor[R*C] | ver[R*C] | qt[(R/2)*(C/2)] | dire[3*R*C] as int8, R=16*bh, C=16*bw; frames contiguous.
 * pmp_frame_values(bh,bw) gives the per-frame count. */
int pmp_assemble_frames(pmp_handle *h, const uint8_t *hor, const uint8_t *ver, const uint8_t *qt_u8,
                        const int8_t *dire, int frames, int bh, int bw, int8_t *out, void *stream);
int64_t pmp_frame_values(int bh, int bw);
/* pmp_format_text == the text body written at Map2Partition.py:405-412: one decimal integer and '\n'
 * per value.  values: n int8 in {-1,0,1,2,3}; text: device buffer of capacity >= 3*n; *n_bytes_host
 * receives the byte count (synchronises the stream). */
int pmp_format_text(pmp_handle *h, const int8_t *values, int64_t n, char *text, int64_t *n_bytes_host,
                    void *stream);
/* pmp_format_texts: the same text for m (1..8) vectors in ONE launch, byte-identical to pmp_format_text per vector, and
 * without a synchronisation.  values[i] (n[i] int8 in {-1,0,1,2,3}, 0 <= n[i] <= 2^30), text[i] (capacity >= 3*n[i])
 * and n_bytes (int64[m]): DEVICE pointers, held in host arrays; n: host.  n_bytes[i] is valid when `stream` reaches
 * this point.  A single-pass scan with per-tile status words that belong to the handle: launches of one handle must not
 * overlap on different streams.  The first launch of a larger total than before allocates (synchronising the device). */
int pmp_format_texts(pmp_handle *h, int m, const int8_t *const *values, const int64_t *n, char *const *text,
                     int64_t *n_bytes, void *stream);

/* ---- input prep ----------------------------------------------------------------------------
 * pmp_cut_blocks == Inference_QBD.output_block_yuv + the chroma input assembly
 * (Inference_QBD.py:104-149,:194-200) on device.  y [F,H,W], u/v [F,H/2,W/2]; sample_bytes 1 (8-bit)
 * or 2 (little-endian 16-bit holding 10-bit samples, reduced with round-half-even(y/4), clip 255).
 * luma_blocks [F*bh*bw,68,68] u8; chroma_blocks [F*bh*bw,3,34,34] u8 = (maxpool2(luma block), U, V). */
int pmp_cut_blocks(pmp_handle *h, const void *y, const void *u, const void *v, int sample_bytes, int frames,
                   int width, int height, uint8_t *luma_blocks, uint8_t *chroma_blocks, void *stream);

/* ---- whole-path convenience ------------------------------------------------------------------
 * pmp_run_component: cut blocks are already on device; runs predict_maps -> qt_postprocess ->
 * map2partition -> assemble_frames for one component (luma=1|0) in chunks of `chunk` blocks.
 * out: frames * pmp_frame_values(bh,bw) int8 (device).  Optional map outputs (device, may be NULL):
 * qt_raw [N,64] f32, bt/dire [N,768] f32, flags [N] u32. */
int pmp_run_component(pmp_handle *h, int wset_q, int wset_msbd, int luma, const uint8_t *blocks, int frames,
                      int bh, int bw, int chunk, int8_t *out, float *qt_raw, float *bt, float *dire,
                      uint32_t *flags, void *stream);

/* pmp_predict_host == the per-QP body of Inference_QBD.py:190-241 from host planes to host PartitionMat vectors
 * (get_sequence_partition_for_VTM order, Map2Partition.py:389-412), for callers without CUDA of their own.
 * wsets: luma Q, luma MSBD, chroma Q, chroma MSBD weight sets of one QP; -1,-1 skips that component.
 * y [F][H][pitch_y], u/v [F][H/2][pitch_c]: HOST pointers (pageable or pinned); pitches in bytes, 0 = dense; sample_bytes
 * as in pmp_cut_blocks (u and v may be NULL when chroma is skipped).  luma_out / chroma_out: HOST, frames *
 * pmp_frame_values(H/64, W/64) int8 each, the text file's values and the .bin payload.  Width or height below 64 means
 * zero blocks: PMP_OK, nothing written.
 * Frames are processed in windows of max(1, chunk / blocks-per-frame) whole frames (chunk <= 0: 4800), staged through
 * library-owned pinned buffers; the next window's upload and the previous one's download overlap the current window's
 * kernels.  Synchronous: returns when both outputs are in host memory.
 * report (may be NULL): decode-flag counts of this call summed over both components (flags of pmp_map2partition;
 * near_threshold = bits 1..3, tight = bits 4..6) and the fp16 saturation events of this call (the sticky counter of
 * pmp_saturation_count is not reset).  Saturation events make the call return PMP_ERR_STATE: rerun with PMP_TC_BF16
 * (Inference_QBD.py:192-194 of this package refuses the same way).
 * Repeated blocks: within a window, the nets run once per distinct cut block (68x68 luma, 3x34x34 chroma input bytes);
 * byte-identical blocks get the first one's results (pmp_block_stats counts the work).  Values, flags and every report
 * field but one are byte-identical to a run without reuse.  fp16_saturation_events (and the sticky counter) count the
 * epilogue events of the blocks computed: a repeated block saturates exactly when its first occurrence does, so the
 * PMP_ERR_STATE stop is unchanged, but the count is that of the distinct blocks. */
typedef struct pmp_report {
    long long blocks, near_tie_blocks, near_threshold_blocks, near_threshold_blocks_tight, fp16_saturation_events;
} pmp_report;
int pmp_predict_host(pmp_handle *h, const int wsets[4], const void *y, const void *u, const void *v, int sample_bytes,
                     int64_t pitch_y, int64_t pitch_c, int frames, int width, int height, int chunk, int8_t *luma_out,
                     int8_t *chroma_out, pmp_report *report);

/* pmp_predict_stream: a sequence of any length from frames to PartitionMat data in bounded memory, for every QP of an
 * encoder run at once (the whole of Inference_QBD.py:190-241 plus the text of Map2Partition.py:405-412).
 * wsets: [n_qps][4], each row as pmp_predict_host's (n_qps 1..4; -1,-1 skips a component of that QP, not both).
 * Frames are processed in windows of window_frames whole frames (<= 0: max(1, 4800 / blocks per frame)).
 *   read(user, first_frame, frames, y, u, v) fills frames [first_frame, first_frame + frames) as dense planes straight
 *     into library-owned page-locked memory: y [frames][H][W], u/v [frames][H/2][W/2], sample_bytes per sample; u and v
 *     are NULL when every QP skips chroma.
 *   write(user, w) is called once per window, in frame order, on the calling thread, while the GPU computes the next
 *     window.  w->values[q][c] (c: 0 luma, 1 chroma) holds w->n_values[q][c] = frames * pmp_frame_values(H/64, W/64)
 *     int8 with PMP_OUT_VALUES; w->text[q][c] holds w->text_bytes[q][c] bytes of file text with PMP_OUT_TEXT.  Pointers
 *     of a skipped component or an output not asked for are NULL (counts 0).  All are valid only during the callback.
 *     w->report counts this window only: decode flags of all its results and its fp16 saturation events.
 * outputs: PMP_OUT_VALUES, PMP_OUT_TEXT or both.  Window k+1 is read and uploaded and window k-1 downloaded and written
 * while window k computes; each window is cut into blocks once for all its QPs and components, and its texts are
 * formatted in one launch.  The host waits only on events of finished windows.  Page-locked and device staging scale
 * with window_frames, not frames; the handle owns them and pmp_destroy frees them.
 * A non-zero return of either callback stops the call with PMP_ERR_ABORTED.  A window with fp16 saturation events is
 * still written; the call then stops with PMP_ERR_STATE (message as pmp_predict_host's).  *report (may be NULL) is the
 * sum over the windows written.  Every return, errors included, leaves no work queued and the handle usable.  Width or
 * height below 64 (zero blocks) returns PMP_OK without calling either callback.
 * Repeated blocks within a window are computed once, as in pmp_predict_host: fp16_saturation_events counts the events of
 * the distinct blocks, every other output is byte-identical to a run without reuse.  This holds for
 * pmp_predict_stream_multi and pmp_predict_stream_ex too. */
enum { PMP_OUT_VALUES = 1, PMP_OUT_TEXT = 2 };
typedef struct pmp_window {
    int first_frame, frames, n_qps;
    const int8_t *values[4][2];
    int64_t n_values[4][2];       /* [qp index][0 luma, 1 chroma] */
    const char *text[4][2];
    int64_t text_bytes[4][2];
    pmp_report report;
} pmp_window;
typedef int (*pmp_read_cb)(void *user, int first_frame, int frames, void *y, void *u, void *v);
typedef int (*pmp_write_cb)(void *user, const pmp_window *w);
int pmp_predict_stream(pmp_handle *h, int n_qps, const int *wsets, int frames, int width, int height, int sample_bytes,
                       int window_frames, int outputs, pmp_read_cb read, pmp_write_cb write, void *user,
                       pmp_report *report);

/* pmp_predict_stream_multi: pmp_predict_stream over several handles at once, on one or several devices (the same
 * sequence and files, several GPUs busy).  handles: n_handles (1..16) distinct non-NULL handles; they may share a device,
 * each keeps its own streams and staging.  wsets: [n_handles][n_qps][4]; row [i][q] names handles[i]'s weight sets for
 * QP q (ids are per handle).
 * Before any callback the call checks that every handle computes what handles[0] computes: the same skip pattern, net
 * kinds and weights (an FNV-1a-64 fingerprint of each weight set's fp32 parameters, taken once per handle and weight set),
 * the same engine and tc_dtype (pmp_set_engine) and the same near_tol (pmp_set_near_tol).  Otherwise it returns
 * PMP_ERR_ARG, calls no callback, and the message names the handle index and the first item that differs.
 * Window k runs on handles[k % n_handles]; each handle keeps its two window slots busy, so up to 2 * n_handles windows
 * are in flight, and the host blocks only on the download of the oldest window not yet written.  window_frames <= 0:
 * max(1, min(4800 / blocks per frame, ceil(frames / n_handles))), so that a short sequence still reaches every handle.
 * The callbacks run on the calling thread, with the calling thread's current device made current before each of them
 * (the call switches devices in between and restores the device on return): read in ascending, contiguous frame order,
 * each frame once; write once per window, in frame order.  All other arguments, the callbacks' contract, the errors,
 * the saturation stop and *report are those of pmp_predict_stream: every return leaves no work queued on any handle and
 * every handle usable.  The values and text are byte-identical to pmp_predict_stream on handles[0]. */
int pmp_predict_stream_multi(pmp_handle *const *handles, int n_handles, int n_qps, const int *wsets, int frames,
                             int width, int height, int sample_bytes, int window_frames, int outputs, pmp_read_cb read,
                             pmp_write_cb write, void *user, pmp_report *report);

/* pmp_predict_stream_ex: pmp_predict_stream_multi where a row is a pair (weight sets, decode thresholds) instead of a QP,
 * so that one call writes PartitionMat data under several threshold settings of Map_to_Partition (Map2Partition.py:100),
 * or several QPs under several settings.
 * n_rows: 1..4; wsets: [n_handles][n_rows][4] as pmp_predict_stream_multi's; lamb: [n_rows][5] doubles, row r's lamb1..lamb5
 * (NULL: the reference defaults 0.7, 0.7, 1.5, 0.3, 0.7 for every row).  A threshold that is not finite returns
 * PMP_ERR_ARG before any callback; the message names the row and the index.  w->values/text[r][c] and w->n_qps (= n_rows)
 * of pmp_window refer to rows; w->report counts each row's blocks, and its near-tie count (flags bit 0) depends on the
 * row's thresholds.
 * Rows of a handle whose (Q, MSBD) weight-set ids for a component are equal share that component's net pass: per window
 * and chunk, pmp_predict_maps and pmp_qt_postprocess run once, then pmp_map2partition_ex and pmp_assemble_frames run once
 * per row.  Four settings of one QP cost one net pass per window plus four decodes, assemblies and texts.
 * Everything else (callbacks, consistency check across handles, errors, saturation stop, report, bounded staging, every
 * return leaving no work queued) is pmp_predict_stream_multi's.  With lamb NULL, or rows equal to the defaults, the output
 * is byte-identical to pmp_predict_stream_multi on the same arguments; pmp_predict_stream_multi is this call with
 * lamb NULL. */
int pmp_predict_stream_ex(pmp_handle *const *handles, int n_handles, int n_rows, const int *wsets, const double *lamb,
                          int frames, int width, int height, int sample_bytes, int window_frames, int outputs,
                          pmp_read_cb read, pmp_write_cb write, void *user, pmp_report *report);

/* pmp_block_stats: sticky per-handle counters of the window pipeline (pmp_predict_host, pmp_predict_stream(_multi,
 * _ex)), summed over the net passes this handle ran since creation / the last reset: *blocks = the blocks of the passes'
 * windows, *computed = the distinct blocks the nets actually ran on (a pass is one component of one window for one
 * weight-set pair; rows sharing weight sets share it).  With 4 QPs, one window of N blocks with d distinct luma blocks
 * adds 4N and 4d for luma.  Host counters: no synchronisation. */
int pmp_block_stats(pmp_handle *h, long long *blocks, long long *computed, int reset);

/* Self-test of the TC conv engine against the SIMT engine on random data (GPU).  Returns 0 and the
 * max-abs error in *max_err, or an error.  flags: bit0 ReLU, bit1 identity residual, bit2 attention product,
 * bit3 bf16 operands; kernel variants: bits 8..9 accumulator scheme of the single-CTA kernel (1 unstacked, 2 stacked),
 * bit10 CTA-pair (cta_group::2) kernel, bit11 force the single-CTA kernel, bit12 unstacked accumulators for the
 * 3x3 Cout = 64 layers (A/B of the default stacked scheme), bits 13..15 cap on the number of whole-tile
 * activation buffers (0: default); bit16 verbose mismatch report on stderr; bit17 fused 1x1 shortcut conv on a second
 * input with ((flags >> 20) & 0xff, default 32) channels (checked against conv + separate 1x1 conv; excludes bit1); bit18 2x2 max-pool with the horizontal half
 * fused into the conv epilogue (checked against the exact conv with fused pooling; excludes bit2). */
int pmp_selftest_conv(pmp_handle *h, int cin, int cout, int ksize, int hw, int batch, int flags,
                      double *max_err, double *ref_absmax, double *ms_tc, double *ms_simt);

/* Test hook: one TC-engine convolution (ResidualBlock conv variants of Model_QBD.py:23-44) on caller-supplied fp32
 * data, so that tests can check the tcgen05 kernels against an independent convolution (torch F.conv2d on the CPU).
 * in [B,cin,hw,hw], res/mul [B,cout,..] (may be NULL), in2 [B,cin2,hw,hw] (fused 1x1 shortcut input, may be NULL): DEVICE
 * fp32 NCHW; w_host [cout,cin,k,k], w_sc_host [cout,cin2]: HOST fp32.  flags: bit0 ReLU, bit3 bf16 operands, bit18 2x2
 * max-pool.  out [B,cout,Ho,Wo] device fp32.  Synchronises the stream. */
int pmp_debug_conv(pmp_handle *h, const float *in, const float *w_host, const float *res, const float *mul,
                   const float *in2, const float *w_sc_host, int cin, int cout, int ksize, int hw, int batch, int cin2,
                   int flags, float *out, void *stream);

/* Test hook: only the first-layer conv(s) of weight set `wset`'s net (conv_q1 with padding_rb, Model_QBD.py:79-80; or
 * conv_b1_1..3 on cat[x, pad_lu(up(qt))] concatenated, :130-135) through the TC engine's stem path (TMA-assembled K
 * chunks), bias + ReLU applied.  qt [B,1,8,8] f32 for the MSBD nets, NULL for the Q nets.  out [B,32,S,S] device fp32
 * (S = 64 luma / 32 chroma). */
int pmp_debug_stem(pmp_handle *h, int wset, const void *blocks, int in_dtype, const float *qt, int B, float *out,
                   void *stream);

/* Test hook: the window pipeline's grouping of repeated blocks (block_reuse.cu) on caller-supplied blocks.  blocks: n
 * blocks of block_bytes bytes each (a positive multiple of 4; DEVICE, 4-byte aligned); rep: DEVICE int[n] receives, for
 * every block i, the lowest index j with blocks j and i byte-identical.  hash_bits (0..64) keeps only that many low bits
 * of the 64-bit fingerprints (0: every block collides), so that tests reach the byte comparison that confirms every
 * fingerprint match.  *n_distinct_host (may be NULL): the number of i with rep[i] == i.  Synchronises the stream. */
int pmp_debug_block_groups(pmp_handle *h, const uint8_t *blocks, int n, int block_bytes, int hash_bits, int *rep,
                           int *n_distinct_host, void *stream);

/* Debug/profiling aid: per-CTA barrier-stall cycle counters of the CTA-pair conv kernel (filled when the environment
 * variable PMP_TC_DBG has bit 6 set; 16 uint64 per CTA, see conv_tc.cu).  n = number of uint64 to copy (<= 2560). */
int pmp_debug_tc_stalls(unsigned long long *out, int n);

#ifdef __cplusplus
}
#endif
#endif /* PMP_B200_H */
