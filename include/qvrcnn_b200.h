/*
 * qvrcnn_b200.h -- C ABI of the B200-native QVRCNN int8 luma-enhancement pass.
 *
 * This is the drop-in boundary for ONE path of binbinmeng/QCNN_GPU: the static-BLU
 * quantised VRCNN forward (`qvrcnn::forward_blu`) with its model / quant-param / YUV
 * formats and its PSNR report.  The reference has no FFI of its own -- its operator
 * surface is the C++ class `qvrcnn` (inference/qvrcnn.cuh:25-59) plus `vrcnn_data`
 * (inference/yuv_data.h:11-27) -- so every entry point below names the reference
 * member/function it replaces (paths relative to the reference repository).
 * A header-only C++ shim with the reference's own class and method names sits on top
 * of this ABI in qcnn_gpu_b200/csrc/qvrcnn.cuh and yuv_data.h.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success
 * and a negative QV_ERR_* code on failure (the reference prints and exit(1)s --
 * inference/cnn.cuh:8-15, inference/qvrcnn.cu:50-54 -- the C++ shim restores that);
 * qv_last_error() returns a thread-local message for the last failure.
 * A handle owns all of its device memory and streams, is bound to one CUDA device,
 * and is not thread-safe; distinct handles may be used from distinct threads.
 * There is no CPU fallback: without a CUDA device qv_create fails.
 */
#ifndef QVRCNN_B200_H
#define QVRCNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define QV_API __attribute__((visibility("default")))
#else
#define QV_API
#endif

typedef struct qv_net qv_net;

enum {
    QV_OK = 0,
    QV_ERR_ARG = -1,      /* bad argument / null pointer / wrong size */
    QV_ERR_IO = -2,       /* file cannot be opened / short read / bad format */
    QV_ERR_CUDA = -3,     /* CUDA runtime failure (message in qv_last_error) */
    QV_ERR_RANGE = -4,    /* model violates the exact-integer envelope (see qv_load_static_para) */
    QV_ERR_STATE = -5     /* call order: e.g. forward before a model is loaded */
};

/* Kernel implementation selector (qv_set_impl). */
enum {
    QV_IMPL_AUTO = 0,     /* fused tcgen05 path when available, else per-layer */
    QV_IMPL_LAYERED = 1,  /* per-layer CUDA-core dp4a kernels, activations in HBM */
    QV_IMPL_FUSED = 2     /* whole net fused per strip, tcgen05.mma kind::i8 + TMEM */
};

/* Layer indices, order of the records in the model file (inference/qvrcnn.cu:55-60). */
enum { QV_C1 = 0, QV_C2_1 = 1, QV_C2_2 = 2, QV_C3_1 = 3, QV_C3_2 = 4, QV_C4 = 5, QV_NLAYER = 6 };

QV_API const char *qv_last_error(void);
QV_API const char *qv_version(void);

/* ---- network object: qvrcnn (inference/qvrcnn.cuh:25-59) -------------------------------- */

/* qvrcnn::qvrcnn(gpu_num, batch, channel, height, width)   inference/qvrcnn.cu:4-29.
   channel must be 1 (luma).  `batch` frames are held in the handle's own x / x_rec buffers. */
QV_API int qv_create(int gpu_num, int batch, int channel, int height, int width, qv_net **out);
/* qvrcnn::~qvrcnn   inference/qvrcnn.cu:331-335 */
QV_API int qv_destroy(qv_net *net);

/* qvrcnn::load_static_para(char*)   inference/qvrcnn.cu:47-63 -> CovLayer::load_static_para
   inference/cnn.cu:90-112.  Reads the 60 028-byte NCHW_VECT_C static model file.
   Returns QV_ERR_RANGE if some output channel has 128*sum|w| + |b| >= 2^24: beyond that the
   reference's fp32 materialisation of u (inference/mat.cuh:69-70) stops being exact integer
   arithmetic and this integer implementation would not be bit-identical. */
QV_API int qv_load_static_para(qv_net *net, const char *filename);
/* Same record stream from memory (for callers that hold the model image already). */
QV_API int qv_load_static_para_mem(qv_net *net, const void *image, size_t len);
/* HWCN-flavoured static model file (input of model_qfp_HWCN2NCHW_VECT_C,
   inference/qvrcnn.cu:535-585), converted on load. */
QV_API int qv_load_static_para_hwcn(qv_net *net, const char *filename);

/* Per-QP scale file written by training/quantization.py:90-96 -- either the pickle
   `quant_params<QP>.data` or the raw `quant_params_cpp_<QP>.data` (6 x 6 doubles).
   Installs blu_q / mul / shift for the six layers (the only fields inference consumes,
   inference/cnn.cu:101-103). */
QV_API int qv_load_quant_params(qv_net *net, const char *filename);
/* Parse only: out18 = {blu, mul, shift} x 6. */
QV_API int qv_read_quant_params(const char *filename, int32_t *out18);
/* Install weights of one layer as plain [K][C][R][S] int8 + int32 bias[K]
   (what CovLayer::load_static_para leaves in w / b, inference/cnn.cu:99-106, minus the
   NCHW_VECT_C packing). */
QV_API int qv_set_weights(qv_net *net, int layer, const int8_t *w_kcrs, const int32_t *bias);
/* Read back what inference will use: out18 = {blu, mul, shift} x 6. */
QV_API int qv_get_quant_params(const qv_net *net, int32_t *out18);

/* qvrcnn::load_data(datatype*)   inference/qvrcnn.cu:64-68 -> InputLayer::load cnn.cu:439-443.
   Copies batch*height*width bytes of luma from host memory into the handle. */
QV_API int qv_load_data(qv_net *net, const uint8_t *host_luma);
/* qvrcnn::forward_blu()   inference/qvrcnn.cu:168-242.  Synchronous like the reference
   (which synchronises after every layer); on return x_rec is complete. */
QV_API int qv_forward_blu(qv_net *net);
/* Replaces the driver's direct poke `cudaMemcpy(recon, qvrcnn1.I1.x_rec, ...)`
   inference/kernel.cu:96: copies batch*height*width bytes of reconstructed luma to host. */
QV_API int qv_get_recon(qv_net *net, uint8_t *host_out);

/* The hot loop of testqvrcnn (inference/kernel.cu:91-97: per frame load_data, forward_blu,
   sync, D2H) over n_frames host frames, pipelined: pinned staging, H2D / compute / D2H
   overlapped on private streams, `batch` frames per chunk.  h_in / h_out may be pageable. */
QV_API int qv_forward_frames_host(qv_net *net, const uint8_t *h_in, uint8_t *h_out, int n_frames);
/* The whole of testqvrcnn's data path for sequences that need not fit in host memory (SURVEY 8 f2): frames
   [first_frame, first_frame + n_frames) of the anchor YUV 4:2:0 file are read chunk by chunk into pinned
   buffers by a reader thread (luma only, file stride h*w*3/2: inference/yuv_data.cpp:32-38), uploaded,
   enhanced, downloaded and written by a writer thread into `recon_yuv` in save_recon_as' layout (Y plane +
   h*w/2 zero bytes per frame, inference/yuv_data.cpp:119-125, at the frame's own offset) -- file reads,
   copies, compute and file writes of different chunks overlap.  With `ori_yuv` the exact integer SSE of the
   anchor and of the reconstruction against the original are accumulated on the device (the integer core of
   vrcnn_data::psnr, inference/yuv_data.cpp:87-97).  ori_yuv, recon_yuv, sse_before, sse_after may be NULL. */
QV_API int qv_stream_yuv(qv_net *net, const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv,
                         int first_frame, int n_frames, int64_t *sse_before, int64_t *sse_after);
/* qv_stream_yuv with the SSEs per frame, the integer core of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112):
   sse_before_pf[j] / sse_after_pf[j] = SSE of the anchor / the reconstruction against the original for frame
   first_frame + j.  Both are host arrays of n_frames (either may be NULL; both need ori_yuv).  qv_stream_yuv returns
   their sums. */
QV_API int qv_stream_yuv_pf(qv_net *net, const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv,
                            int first_frame, int n_frames, int64_t *sse_before_pf, int64_t *sse_after_pf);
/* Same pass on frames already resident in device memory (n_frames may exceed `batch`);
   asynchronous on `cuda_stream` (a cudaStream_t, NULL = the handle's own stream, in which
   case the call synchronises before returning). */
QV_API int qv_forward_frames_device(qv_net *net, const uint8_t *d_in, uint8_t *d_out, int n_frames,
                                    void *cuda_stream);
/* qv_forward_frames_device plus the per-frame quality report of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112):
   for every frame f the exact sum of (anchor - ori)^2 is ADDED to d_sse[2f] and the sum of (out - ori)^2 to
   d_sse[2f + 1] (device int64, [n_frames][2]; incremented like qv_sse_device, so chunks and repeated calls add up).
   d_ori holds the original luma of the same n_frames frames.  The output is byte-identical to qv_forward_frames_device.
   The fused path computes the sums in the kernel's output stage (one extra byte read per pixel; there is no SSE form of
   the opt-in QV_FUSED_TMA input ring, so with it set this call runs the kernel without TMA); the layered path runs a
   separate SSE pass per frame.  Null d_ori / d_sse: QV_ERR_ARG; on the fused path frame heights above 66051 are refused
   (QV_ERR_ARG), the layered path takes any height. */
QV_API int qv_forward_frames_device_sse(qv_net *net, const uint8_t *d_in, const uint8_t *d_ori, uint8_t *d_out,
                                        int n_frames, int64_t *d_sse, void *cuda_stream);
/* Spatially partitioned pass for one very large frame (multi-GPU strips): the frame has
   img_height x width pixels (width = the handle's); d_in points at image row `in_row0` and holds
   `in_rows` rows (the strip plus up to 6 halo rows each side); rows [out_row0, out_row1) are
   written to d_out (whose first row is out_row0).  Activations outside the IMAGE are zero
   (each layer's own SAME padding, inference/cnn.cu:44-49); rows outside the strip but inside
   the image are recomputed from the halo.  (The caller has gathered the halo rows; qv_strip_* below
   is the variant in which the kernel reads them from the neighbour GPUs' memory.) */
QV_API int qv_forward_rows_device(qv_net *net, const uint8_t *d_in, int img_height, int in_row0, int in_rows,
                                  uint8_t *d_out, int out_row0, int out_row1, void *cuda_stream);

/* Synchronises `cuda_stream` (NULL = the handle's own stream) and reports what the kernels that ran on it found:
   QV_ERR_CUDA if a CTA of the fused kernel gave up on a wait (the output of that launch is not valid), QV_OK otherwise.
   The asynchronous entry points (a non-NULL cuda_stream) cannot report this themselves; a NULL cuda_stream names the
   handle's own stream and makes the call synchronous -- to run on the legacy default stream pass cudaStreamLegacy. */
QV_API int qv_synchronize(qv_net *net, void *cuda_stream);

/* ---- one very large frame over several GPUs: horizontal strips, halo rows read over NVLink (SURVEY 8e-ii) ------------
   The reference runs on device 0 only (inference/kernel.cu:86); forward_blu's receptive field is 2+2+1+1 = 6 rows, so
   a GPU that owns image rows [row0, row1) needs 6 more rows from the GPU above and 6 from the GPU below.  They are
   never copied: every handle keeps its rows in a block of its own device memory which the two neighbours MAP (same
   process: CUDA peer access; another process: CUDA IPC) and the fused kernel's input stage loads the halo rows straight
   from the neighbour's HBM.  Ordering is by sequence numbers in the same block, written and polled by the kernels
   themselves (system-scope release / acquire): no collective, no host synchronisation between frames.  All handles of a
   frame must make the same sequence of qv_strip_forward calls.  Fused path only.
   One strip per GPU is the layout this is for.  Kernels of different launches must never wait for each other on ONE GPU
   (nothing guarantees that they run at the same time), so strips that share a GPU -- a test layout -- are ordered by
   stream order instead: the caller drives all of them on one stream, all loads of a frame before its forwards (a different
   stream is refused), and strips of different PROCESSES on one GPU are refused by qv_strip_attach.

     each GPU:  qv_create(gpu, 1, 1, rows, W) ; load model ; qv_strip_setup(net, H, row0, row1) ; qv_strip_export(net, &d)
     exchange the 192-byte descriptors once (threads: a shared array; processes: any byte transport)
     each GPU:  qv_strip_attach(net, QV_STRIP_ABOVE, &d[above]) ; qv_strip_attach(net, QV_STRIP_BELOW, &d[below])
     per frame k: qv_strip_load(net, k & 1, host_rows, st) ; qv_strip_forward(net, k & 1, d_out, st)                     */
typedef struct { unsigned char opaque[192]; } qv_strip_desc;
enum { QV_STRIP_ABOVE = 0, QV_STRIP_BELOW = 1 };
/* This handle owns image rows [row0, row1) of an img_height x width frame (width = the handle's). */
QV_API int qv_strip_setup(qv_net *net, int img_height, int row0, int row1);
QV_API int qv_strip_export(qv_net *net, qv_strip_desc *out);
/* Maps the neighbour's block.  Fails if the rows are not adjacent, or if the neighbour holds fewer than 6 rows. */
QV_API int qv_strip_attach(qv_net *net, int side, const qv_strip_desc *neighbour);
/* Device pointer of input slot 0 / 1 ((row1-row0) * width bytes) for callers that fill it on the device. */
QV_API int qv_strip_input(qv_net *net, int slot, void **d_rows);
/* Before overwriting a slot: waits (on the stream) until both neighbours have finished the step that read it. */
QV_API int qv_strip_acquire(qv_net *net, int slot, void *cuda_stream);
/* qv_strip_acquire + H2D copy of this GPU's rows into the slot (InputLayer::load, inference/cnn.cu:439-443). */
QV_API int qv_strip_load(qv_net *net, int slot, const uint8_t *host_rows, void *cuda_stream);
/* forward_blu on this GPU's rows of the frame in `slot`; rows [row0, row1) of the reconstruction go to d_out. */
QV_API int qv_strip_forward(qv_net *net, int slot, uint8_t *d_out, void *cuda_stream);
/* qv_strip_forward plus this GPU's share of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112) for the frame: d_ori_rows
   holds the original's rows [row0, row1) (device memory of this GPU), and the SSEs of the anchor and of the reconstruction
   over those rows are ADDED to d_sse2[0] and d_sse2[1] (device int64).  The caller adds the strips' values together.
   Null d_ori_rows / d_sse2: QV_ERR_ARG; not the fused path: QV_ERR_STATE, as qv_strip_forward. */
QV_API int qv_strip_forward_sse(qv_net *net, int slot, const uint8_t *d_ori_rows, uint8_t *d_out, int64_t *d_sse2,
                                void *cuda_stream);
/* qv_stream_yuv_pf through the strip partition: frames [first_frame, first_frame + n_frames) of a YUV 4:2:0 sequence,
   enhanced by the strip handles of THIS process (set up, exported and attached; on one device or several).  Each handle
   reads only its own rows of each frame from the anchor (and original) file with pread -- luma row r of frame f at byte
   f*H*W*3/2 + r*W -- and writes its rows of the reconstruction at the same offsets with pwrite; the handle that owns the
   last image row also writes the frame's H*W/2 zero bytes of chroma (save_recon_as' layout).  recon_yuv is opened like
   qv_stream_yuv's (created if missing, never truncated): frames outside the range and other processes' rows are left as
   they are.  A reader thread keeps one frame ahead and a writer thread one frame behind, over a ring of three page-locked
   slots per strip; one GPU thread per device drives that device's strips (one strip: two streams, upload of frame k+1
   overlapping the compute of frame k; several strips: one stream, all loads of a frame before its forwards).  Host and
   device memory are O(strip rows x W), whatever n_frames is.  The call waits for the devices of `nets` to be idle before it
   starts and leaves the handles idle, free to be driven on any stream.
   With ori_yuv, sse_before_pf[j] / sse_after_pf[j] are the SSEs of the anchor / the reconstruction against the original
   over this call's rows of frame first_frame + j (qv_strip_forward_sse per strip); with every strip of the frame in one call
   they are the frame's, as qv_stream_yuv_pf returns them, and across processes the caller adds them up.  Either may be NULL.
   Every process that holds strips of the frame must make the same call (same first_frame and n_frames): the strips' handles
   must see the same sequence of forwards.  Checked before any file is opened: QV_ERR_ARG for null or empty nets, a handle
   given twice, handles of different widths or image heights, a negative first_frame / n_frames, an SSE pointer without
   ori_yuv, or with ori_yuv an image taller than 66051 rows; QV_ERR_STATE for a handle without qv_strip_setup, without a
   neighbour on an interior edge or without the fused path, and for a device that also holds a strip handle of this process
   that is not in nets (strips that share a GPU are driven together).  QV_ERR_IO: open failure, short read, failed write.
   QV_ERR_CUDA: a CUDA call failed or a CTA reported a failure.  n_frames == 0: QV_OK, no file touched. */
QV_API int qv_strip_stream_yuv_pf(qv_net *const *nets, int n_nets, const char *anchor_yuv, const char *ori_yuv,
                                  const char *recon_yuv, int first_frame, int n_frames,
                                  int64_t *sse_before_pf, int64_t *sse_after_pf);
/* Unmaps the neighbours and frees the block (all GPUs must be idle). */
QV_API int qv_strip_release(qv_net *net);

/* Explicit device-pointer accessor for drivers that, like the reference's, read the object's
   buffers directly (`qvrcnn1.I1.x_rec`, inference/kernel.cu:96; InputLayer::x / x_rec,
   inference/cnn.cuh:98).  The pointers stay owned by the handle. */
QV_API int qv_device_buffers(qv_net *net, void **d_x, void **d_x_rec);

/* Sum of squared errors between two device luma buffers of n bytes (exact int64), the integer
   core of vrcnn_data::psnr (inference/yuv_data.cpp:87-97).  *d_sse_accum (device int64) is
   incremented; asynchronous on cuda_stream. */
QV_API int qv_sse_device(const uint8_t *d_a, const uint8_t *d_b, size_t n, int64_t *d_sse_accum, void *cuda_stream);

/* Implementation / debug controls (no reference counterpart). */
QV_API int qv_set_impl(qv_net *net, int impl);
QV_API int qv_get_impl(const qv_net *net);
/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
QV_API long long qv_launch_count(const qv_net *net);
/* Debug taps of the LAYERED path, valid after qv_forward_blu: copies frame 0's activations to
   host as planar int8 [C][H][W] (a1: 64, a2: 48, a3: 48 channels) -- the contents of C1.v,
   Conc1.conc, Conc2.conc in the reference (inference/qvrcnn.cu:183,202,218). */
QV_API int qv_get_activation(qv_net *net, int which /*1,2,3*/, int8_t *host_out);

/* Test hook, needs no GPU: what the host builds for the fused kernel from a static model image (Appendix B format) --
   the shared-memory weight image, the per-phase tcgen05 operand table (for window base 0 / TMEM base 0) and the layout
   and requantiser constants.  sizes[3] = capacities in elements on entry, actual element counts on return; a buffer that
   is null or too small is not written.  tests/test_fused_tables.py emulates the kernel's dataflow on these. */
QV_API int qv_debug_fused_tables(const void *model_image, size_t len, uint8_t *wimg, uint32_t *ops, int32_t *consts, size_t sizes[3]);

/* Test hook, needs no GPU: how the fused kernel's launch for n_frames frames of height x width (output rows [row0, row1);
   row_window != 0: a row-window launch of one frame, as the strip entry points issue) is dealt out to sm_count persistent
   CTAs -- the host's plan (equal row segments, or one equal chunk of the row line per SM when allow_line != 0 and that is
   cheaper) read back through the same unit_geo() the kernel uses.  units: 5 ints per work unit (cta, frame, strip column, y0, y1);
   *n_units = capacity in units on entry, count on return (a null or too small buffer is not written).
   tests/test_fused_units.py checks that every (frame, column, row) is covered exactly once and the load is balanced. */
QV_API int qv_debug_fused_units(int sm_count, int n_frames, int height, int width, int row0, int row1, int row_window, int allow_line,
                                int32_t *units, size_t *n_units, int *grid);

/* ---- model-file converters (SURVEY 8f1) ------------------------------------------------- */
/* model_qfp_HWCN2NCHW_VECT_C   inference/qvrcnn.cu:558-585 */
QV_API int qv_convert_model_hwcn_to_vect_c(const char *file_in, const char *file_out);

/* ---- quant-parameter solver and float -> int8 model quantiser (SURVEY 8f4) ----------------- */
/* adjust_quant(stepw_in, blu_in)   training/quantization.py:55-64 (with mul_shift :5-14, mul_shift_f :15-24,
   quant_qfp_layer :25-31, quant_qfp_concat :32-49, quant_qfp_last :50-53), same IEEE-754 operation order.
   stepw_in[6], blu_in[6] (order C1, C2_1, C2_2, C3_1, C3_2, C4) -> rows_out[6][6] =
   [stepw, ratio, blu_adj, blu_q, mul, shift] per layer, i.e. the content of quant_params<QP>.data. */
QV_API int qv_solve_quant_params(const double *stepw_in, const double *blu_in, double *rows_out36);
/* The raw flavour quantNsave also writes: quant_params_cpp_<QP>.data, 6 x struct.pack('6d')
   (training/quantization.py:93-96). */
QV_API int qv_write_quant_params_cpp(const char *filename, const double *rows36);
/* Float weights/biases of one layer -> the int8 / int32 the inference path loads:
   w_q = clip(round(w / stepw), -128, 127)   (training/model.py:167,201; round = half-to-even like numpy.around)
   b_q = round(b * ratio / stepw)            (training/quantization.py:104, the integer part of it)
   w is plain [K][C][R][S] float, n_w = K*C*R*S, n_b = K. */
QV_API int qv_quantize_layer(const float *w, size_t n_w, const float *b, size_t n_b, double stepw, double ratio,
                             int8_t *w_q, int32_t *b_q);

/* Host frame buffers for the vrcnn_data shim (the reference mallocs ori / input / recon, inference/yuv_data.cpp:3-14):
   page-locked when a CUDA device is present, so that the driver's per-frame load_data and its cudaMemcpy of x_rec
   (inference/kernel.cu:93,96) are plain DMA; plain malloc otherwise.  Free with qv_host_free. */
QV_API void *qv_host_alloc(size_t bytes);
QV_API void qv_host_free(void *p);

/* ---- luma frame I/O + PSNR: vrcnn_data (inference/yuv_data.h:11-27) ---------------------- */
/* vrcnn_data::read_data   inference/yuv_data.cpp:15-42: luma of the first `frames` frames of
   a YUV 4:2:0 8-bit planar file. */
QV_API int qv_yuv_read_luma(const char *filename, int frames, int height, int width, uint8_t *out);
/* vrcnn_data::read_frame   inference/yuv_data.cpp:44-66: luma of frame n. */
QV_API int qv_yuv_read_frame(const char *filename, int n, int height, int width, uint8_t *out);
/* vrcnn_data::save_recon_as   inference/yuv_data.cpp:113-128: Y plane then h*w/2 zero bytes. */
QV_API int qv_yuv_write_recon(const char *filename, const uint8_t *luma, int frames, int height, int width);
/* vrcnn_data::psnr   inference/yuv_data.cpp:87-97 (pooled over n samples). */
QV_API double qv_psnr(const uint8_t *data, const uint8_t *ori, size_t n, int64_t *sse_out);
/* PSNR from an (all-reduced) integer SSE: mse = sse/n; 10*log10(65025/mse). */
QV_API double qv_psnr_from_sse(int64_t sse, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* QVRCNN_B200_H */
