/*
 * rip_cuda.h -- C ABI of librip_cuda.so, the B200 (sm_100a) replacement for the OpenCL layer of
 * Arief-AK/OpenCL-Development-Real-time-Image-Processing.
 *
 * This is the drop-in boundary: plain C types only (no STL, no OpenCV, no torch).  The reference's
 * host classes (Controller / ProgramHandler / Comparator / FileHandler, re-implemented in
 * <package>/host/) call these entry points where the reference calls the OpenCL C API; each
 * declaration names the reference code it replaces (paths relative to the reference checkout,
 * "RT/" = src/RealtimeImageProcessing/).
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t value on a CUDA failure, or a
 *     negative RIP_E* code; rip_last_error_string() describes the last failure of the calling thread.
 *   - rip_stream is a cudaStream_t (NULL = the device's default stream).  Device ops are
 *     asynchronous on their stream; pointers named d_* are device pointers on the stream's device.
 *   - images are interleaved u8, row-major, tightly packed (pitch = width * channels); batches are
 *     n_frames consecutive frames.
 *   - device buffers may start at any byte: rip_gray, rip_convert, rip_sobel and rip_fused take any alignment of d_in
 *     and d_out (aligned buffers run the wider kernels, with the same results).  The one exception is RGBA rip_gauss
 *     (channels = 4), whose d_in and d_out must be 4-byte aligned; otherwise it returns RIP_EINVAL and writes nothing.
 *   - results are defined by the reference's CPU paths (bit-exact): gray = Comparator.cpp:30-45,
 *     blur = GaussianBlur.cpp:231-261, Sobel = EdgeDetection.cpp:219-240, fused = their
 *     composition with a u8 image between stages.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef RIP_CUDA_H
#define RIP_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RIP_ABI_VERSION 1

enum {
    RIP_OK = 0,
    RIP_EINVAL = -1,   /* bad argument (null pointer, non-positive size, even kernel size ...) */
    RIP_ENODEV = -2,   /* no usable CUDA device */
    RIP_ENOMEM = -3,   /* host allocation failed */
    RIP_EUNSUPPORTED = -4
};

typedef void *rip_stream;              /* cudaStream_t;   replaces cl_command_queue */
typedef struct rip_ctx rip_ctx;        /* device set + cached buffers; replaces cl_context */
typedef struct rip_module rip_module;  /* loaded kernel image;  replaces cl_program */
typedef struct rip_kernel rip_kernel;  /* kernel variant handle; replaces cl_kernel */
typedef struct rip_event rip_event;    /* cudaEvent_t wrapper;  replaces cl_event */
typedef struct rip_ticket rip_ticket;  /* one job in flight in the host-buffer pipeline (rip_submit / rip_collect) */

/* pixel formats of the interleaved u8 images */
enum { RIP_FMT_GRAY8 = 1, RIP_FMT_RGB8 = 3, RIP_FMT_RGBA8 = 4, RIP_FMT_BGR8 = 5, RIP_FMT_BGRA8 = 6, RIP_FMT_NV12 = 7,
       RIP_FMT_NV12_COLOR = 8, RIP_FMT_YUYV = 9, RIP_FMT_UYVY = 10, RIP_FMT_I420 = 11,
       RIP_FMT_BAYER_RGGB8 = 12, RIP_FMT_BAYER_BGGR8 = 13, RIP_FMT_BAYER_GRBG8 = 14, RIP_FMT_BAYER_GBRG8 = 15,
       RIP_FMT_BAYER_RGGB10 = 16, RIP_FMT_BAYER_BGGR10 = 17, RIP_FMT_BAYER_GRBG10 = 18, RIP_FMT_BAYER_GBRG10 = 19,
       RIP_FMT_BAYER_RGGB12 = 20, RIP_FMT_BAYER_BGGR12 = 21, RIP_FMT_BAYER_GRBG12 = 22, RIP_FMT_BAYER_GBRG12 = 23,
       RIP_FMT_BAYER_RGGB14 = 24, RIP_FMT_BAYER_BGGR14 = 25, RIP_FMT_BAYER_GRBG14 = 26, RIP_FMT_BAYER_GBRG14 = 27,
       RIP_FMT_BAYER_RGGB16 = 28, RIP_FMT_BAYER_BGGR16 = 29, RIP_FMT_BAYER_GRBG16 = 30, RIP_FMT_BAYER_GBRG16 = 31,
       RIP_FMT_BAYER_RGGB10P_MIPI = 40, RIP_FMT_BAYER_BGGR10P_MIPI = 41, RIP_FMT_BAYER_GRBG10P_MIPI = 42,
       RIP_FMT_BAYER_GBRG10P_MIPI = 43,
       RIP_FMT_BAYER_RGGB12P_MIPI = 44, RIP_FMT_BAYER_BGGR12P_MIPI = 45, RIP_FMT_BAYER_GRBG12P_MIPI = 46,
       RIP_FMT_BAYER_GBRG12P_MIPI = 47,
       RIP_FMT_BAYER_RGGB10P_GENICAM = 48, RIP_FMT_BAYER_BGGR10P_GENICAM = 49, RIP_FMT_BAYER_GRBG10P_GENICAM = 50,
       RIP_FMT_BAYER_GBRG10P_GENICAM = 51,
       RIP_FMT_BAYER_RGGB12P_GENICAM = 52, RIP_FMT_BAYER_BGGR12P_GENICAM = 53, RIP_FMT_BAYER_GRBG12P_GENICAM = 54,
       RIP_FMT_BAYER_GBRG12P_GENICAM = 55 };
/* RIP_FMT_NV12 (the reference's camera format, RT/RealtimeImageProcessing.cpp:153): per frame a W*H luma plane
 * followed by the W*H/2 interleaved chroma plane (frame = W*H*3/2 bytes, H even).  Accepted by the EDGE and FUSED
 * operations only; the luma plane is the gray image (one byte per pixel leaves HBM instead of three or four),
 * the chroma plane is never read.  Row bands of an NV12 frame are passed as plain luma rows.
 * RIP_FMT_NV12_COLOR: the same bytes (W and H even), decoded to colour first, exactly as OpenCV's
 * cvtColor(COLOR_YUV2RGB_NV12) does (BT.601 limited range, 20-bit fixed point, one U,V pair per 2x2 block); every
 * operation then gives the reference's result on that colour image: GRAYSCALE its gray, GAUSSIAN the blur of the
 * RGBA image with alpha 255 (W*H*4 bytes out), EDGE / FUSED their result on its gray.  Whole frames only (no row bands);
 * rip_gray and rip_convert take it on device buffers, rip_sobel / rip_fused do not (decode with rip_gray first).
 * RIP_FMT_YUYV, RIP_FMT_UYVY and RIP_FMT_I420 are the other common camera and video layouts, decoded to colour exactly as
 * NV12_COLOR is (OpenCV's cvtColor(COLOR_YUV2RGB_YUYV / _UYVY / _I420), the same arithmetic) and taken everywhere
 * NV12_COLOR is, with the same results on the decoded image (GAUSSIAN: W*H*4 bytes out):
 *   YUYV: packed 4:2:2, bytes Y0 U Y1 V per horizontal pixel pair, 2*W bytes per row (frame = W*H*2 bytes); W even,
 *         any H.  What a UVC webcam delivers (V4L2 with CAP_PROP_CONVERT_RGB off: a CV_8UC2 Mat).
 *   UYVY: the same with bytes U Y0 V Y1 (HDMI / SDI capture cards, many CSI sensors); W even, any H.
 *   I420: planar 4:2:0: the W*H luma plane, then the (W/2)*(H/2) U plane, then the V plane (frame = W*H*3/2 bytes);
 *         W and H even.  FFmpeg's yuv420p, GStreamer's I420.
 * None of the four has a luma-only meaning (RIP_FMT_NV12 is that for NV12).
 * RIP_FMT_BAYER_RGGB8 / _BGGR8 / _GRBG8 / _GBRG8: 8-bit Bayer raw frames, W*H bytes per frame (one byte per pixel,
 * row-major, frames consecutive), W >= 3 and H >= 3 of any parity; what machine-vision cameras (GenICam BayerRG8 ...) and
 * raw CSI sensors (V4L2 SRGGB8 ...) deliver.  Named by the sensor's top-left 2x2, as V4L2 and GenICam name them; OpenCV
 * names a pattern by the 2x2 at (1, 1), so the same result comes from its COLOR_BayerBG2RGB (RGGB), COLOR_BayerRG2RGB (BGGR),
 * COLOR_BayerGB2RGB (GRBG) and COLOR_BayerGR2RGB (GBRG), and their 2BGR / 2RGBA / 2BGRA forms.  Demosaiced exactly as
 * OpenCV's default (bilinear) cvtColor does it, border pixels copying their interior neighbour, and taken everywhere
 * NV12_COLOR is, with the same results on the decoded image (GAUSSIAN: W*H*4 bytes out).
 * RIP_FMT_BAYER_<pattern>10 / 12 / 14 / 16 (codes 16-31, patterns in the same order as 12-15 within each depth): Bayer raw
 * frames of b = 10, 12, 14 or 16 bits per sample, W*H little-endian 16-bit words per frame (2*W*H bytes, row-major, frames
 * consecutive), W >= 3 and H >= 3 of any parity; what V4L2 SRGGB10 / 12 / 14 / 16 ... and GenICam BayerRG10 / 12 / 14 / 16 ...
 * (unpacked) deliver.  Samples are LSB-aligned, as V4L2 and GenICam store them; a stream whose samples are MSB-aligned is a
 * 16-bit stream to this decode (use the *16 code).  The decode is OpenCV's cvtColor(COLOR_Bayer**2RGB) on the CV_16U frame
 * (the 8-bit formulas on the full samples, the same pattern names) followed by convertTo(CV_8U, 1.0 / (1 << (b - 8))): each
 * channel divided by 2^(b-8), rounded half to even, saturated (a full-scale sample gives 255; padding bits above bit b-1 are
 * used as they are, and saturate); alpha 255.  Taken everywhere the 8-bit Bayer formats are, with the same results on that
 * 8-bit image.
 * Packed 10- and 12-bit Bayer raw frames (codes 40-55, patterns in the order of 12-15 within each packing): rows of exactly
 * W*5/4 bytes (10-bit) or W*3/2 bytes (12-bit), no row padding, frames consecutive (H*W*5/4 or H*W*3/2 bytes each), any
 * alignment; W a multiple of 4 (10-bit) or of 2 (12-bit) and at least 4, H at least 3 (else RIP_EINVAL).
 *   RIP_FMT_BAYER_<pattern>10P_MIPI (40-43): MIPI CSI-2 RAW10 (V4L2 SRGGB10P ..., libcamera SRGGB10_CSI2P ...), 4 pixels in
 *     5 bytes:
 *         byte 0      byte 1      byte 2      byte 3      byte 4
 *         P0[9:2]     P1[9:2]     P2[9:2]     P3[9:2]     P3[1:0] P2[1:0] P1[1:0] P0[1:0]   (bit 7 ... bit 0)
 *   RIP_FMT_BAYER_<pattern>12P_MIPI (44-47): MIPI CSI-2 RAW12 (V4L2 SRGGB12P ..., libcamera SRGGB12_CSI2P ...), 2 pixels in
 *     3 bytes:
 *         byte 0      byte 1      byte 2
 *         P0[11:4]    P1[11:4]    P1[3:0] P0[3:0]                                         (bit 7 ... bit 0)
 *   RIP_FMT_BAYER_<pattern>10P_GENICAM (48-51), RIP_FMT_BAYER_<pattern>12P_GENICAM (52-55): GenICam PFNC BayerRG10p /
 *     BayerRG12p ... (and BayerBG, BayerGR, BayerGB), an LSB-first bit stream: pixel i occupies stream bits b*i .. b*i+b-1,
 *     stream bit k is bit k % 8 of byte k / 8.  At 10 bits:
 *         byte 0      byte 1              byte 2              byte 3              byte 4
 *         P0[7:0]     P1[5:0] P0[9:8]     P2[3:0] P1[9:6]     P3[1:0] P2[9:4]     P3[9:2]   (bit 7 ... bit 0)
 *     at 12 bits:
 *         byte 0      byte 1              byte 2
 *         P0[7:0]     P1[3:0] P0[11:8]    P1[11:4]                                        (bit 7 ... bit 0)
 *     A width off these multiples would start rows inside a byte.
 * The decode unpacks the b-bit samples and applies exactly the decode of RIP_FMT_BAYER_<pattern>10 / 12 (cvtColor on the
 * 16-bit frame, then convertTo(CV_8U, 1.0 / (1 << (b - 8)))); packed samples have no padding bits, so full scale (1023 /
 * 4095) gives 255.  Taken everywhere the other Bayer formats are, with the same results on that 8-bit image. */

/* operations (the reference's METHOD strings "GRAYSCALE" / "GAUSSIAN" / "EDGE", plus "FUSED") */
enum { RIP_OP_GRAY = 0, RIP_OP_EDGE = 1, RIP_OP_GAUSSIAN = 2, RIP_OP_FUSED = 3 };

/* gray output layouts: one byte per pixel, or the reference's buffer-path container
 * (g,g,g,255) of W*H*4 bytes (RT/src/ProgramHandler.cpp:185, RT/RealtimeImageProcessing.cpp:114) */
enum { RIP_GRAY_OUT_U8 = 0, RIP_GRAY_OUT_RGBA = 1 };

typedef struct rip_device_info {
    char name[128];
    int sm_count;
    int cc_major, cc_minor;
    int clock_khz;
    int l2_bytes;
    size_t global_mem_bytes;
    size_t smem_per_sm_bytes;
} rip_device_info;

/* ---- library / device discovery  (replaces clGetPlatformIDs / clGetDeviceIDs / clGetDeviceInfo:
 *      RT/src/Controller.cpp:13-64, RT/src/ProgramHandler.cpp:62-66) ---- */
int rip_abi_version(void);
const char *rip_last_error_string(void);
int rip_device_count(int *count);
int rip_device_name(int device, char *buf, size_t buf_len);
int rip_device_get_info(int device, rip_device_info *info);
/* "domain:bus:device.function" of the device (cudaDeviceGetPCIBusId): lets a one-process-per-GPU launcher put its
 * host thread and its pinned frame buffers on the NUMA node the GPU hangs off (/sys/bus/pci/devices/<id>/numa_node),
 * which the end-to-end (host-buffer) throughput of an 8-GPU box depends on. */
int rip_device_pci_bus_id(int device, char *buf, size_t buf_len);

/* ---- context / program / kernel handles (replace clCreateContext, clCreateProgramWithSource +
 *      clBuildProgram, clCreateKernel: RT/src/Controller.cpp:97-191).  The kernels are compiled
 *      into the library (sm_100a SASS), so "loading" a module validates the variant name
 *      ("grayscale_base.cl", "gaussian_base.cl", "edge_base.cl", "fused" ...) and "getting" a
 *      kernel binds the entry ("grayscale", "gaussian_blur", "sobel_edge_detection", "fused"). ---- */
int rip_ctx_create(const int *devices, int n_devices, rip_ctx **ctx);
int rip_ctx_destroy(rip_ctx *ctx);
int rip_ctx_device_count(const rip_ctx *ctx, int *n_devices);
int rip_ctx_device(const rip_ctx *ctx, int index, int *device);
int rip_module_load(rip_ctx *ctx, const char *variant, rip_module **module);
int rip_module_release(rip_module *module);
int rip_kernel_get(rip_module *module, const char *kernel_name, rip_kernel **kernel);
int rip_kernel_release(rip_kernel *kernel);
int rip_kernel_op(const rip_kernel *kernel, int *op);

/* ---- streams, events, memory (replace clCreateCommandQueue, cl_event profiling, clCreateBuffer,
 *      clEnqueueWriteBuffer / clEnqueueReadBuffer: RT/src/Controller.cpp:115-129, 66-74, 234-324) ---- */
int rip_stream_create(int device, rip_stream *stream);
int rip_stream_destroy(int device, rip_stream stream);
int rip_stream_sync(int device, rip_stream stream);
int rip_device_sync(int device);
int rip_event_create(int device, rip_event **event);
int rip_event_destroy(rip_event *event);
int rip_event_record(rip_event *event, rip_stream stream);
int rip_event_sync(rip_event *event);
int rip_event_elapsed_ns(rip_event *start, rip_event *stop, uint64_t *ns);
int rip_malloc_device(int device, size_t bytes, void **d_ptr);
int rip_free_device(int device, void *d_ptr);
int rip_malloc_pinned(size_t bytes, void **h_ptr);
int rip_free_pinned(void *h_ptr);
int rip_memcpy_h2d_async(int device, void *d_dst, const void *h_src, size_t bytes, rip_stream stream);
int rip_memcpy_d2h_async(int device, void *h_dst, const void *d_src, size_t bytes, rip_stream stream);
int rip_memset_device_async(int device, void *d_dst, int value, size_t bytes, rip_stream stream);

/* ---- Gaussian weights, typed like the reference generator
 *      (RT/src/Controller.cpp:352-372 == src/GaussianBlur/src/Controller.cpp:342-362) ---- */
int rip_gauss_weights(int ksize, float sigma, float *weights /* ksize*ksize, host */);

/* ---- device-resident operations (replace clSetKernelArg + clEnqueueNDRangeKernel of
 *      kernel/grayscale_base.cl, gaussian_base.cl, edge_base.cl; RT/src/Controller.cpp:429-744).
 *      All asynchronous on `stream` of `device`. ---- */

/* d_out[i] = (uchar)(0.299*r + 0.587*g + 0.114*b) (double, truncation).  in_format: RGB8 / RGBA8 /
 * BGR8 / BGRA8, or NV12_COLOR / YUYV / UYVY / I420 / BAYER_* of any depth or packing (decoded in the same kernel; 16-bit
 * samples: 2*w*h bytes in per frame, packed: w*h*5/4 or w*h*3/2; any alignment).  out_mode: RIP_GRAY_OUT_U8 (w*h bytes per frame) or
 * RIP_GRAY_OUT_RGBA (w*h*4). */
int rip_gray(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width,
             int height, int n_frames, int in_format, int out_mode);

/* Colour conversion of whole frames: in_format RIP_FMT_NV12_COLOR or RIP_FMT_I420 (width and height even), RIP_FMT_YUYV or
 * RIP_FMT_UYVY (width even), RIP_FMT_BAYER_* of 8 to 16 bits (width and height at least 3) or packed at 10 and 12 bits
 * (width a multiple of 4 or 2 and at least 4, height at least 3), out_format RGB8 / BGR8 / RGBA8
 * (alpha 255) / BGRA8: OpenCV's cvtColor(COLOR_YUV2RGB_NV12 / _BGR / _RGBA / _BGRA, and the same for _I420, _YUYV, _UYVY;
 * the Bayer conversions listed with the formats, followed for 10 to 16 bits and packed samples by
 * convertTo(CV_8U, 1.0 / (1 << (b - 8)))),
 * bit for bit.  d_in and d_out may have any alignment.  d_out: w*h*3 or w*h*4 bytes per frame. */
int rip_convert(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width, int height,
                int n_frames, int in_format, int out_format);

/* K x K float32 convolution per channel in the reference's summation order, clamp-to-edge,
 * truncation.  channels: 1 (gray, any alignment) or 4 (RGBA, all four channels blurred; d_in and d_out
 * 4-byte aligned, else RIP_EINVAL).  weights: host pointer to ksize*ksize floats (copied before the call
 * returns).  ksize odd, 1..RIP_MAX_KSIZE. */
#define RIP_MAX_KSIZE 31
int rip_gauss(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width,
              int height, int n_frames, int channels, int ksize, const float *weights);

/* 3x3 Sobel magnitude, BORDER_REFLECT_101, round-half-even, saturate (OpenCV semantics).
 * in_format GRAY8 runs on the image as is; RGB8/RGBA8/BGR8/BGRA8 first convert with rip_gray's
 * arithmetic inside the same kernel; NV12 (even height, any width) runs on the luma plane of each frame.  d_out: w*h bytes
 * per frame.  NV12_COLOR, YUYV, UYVY, I420, BAYER_*: RIP_EUNSUPPORTED (rip_gray
 * with RIP_GRAY_OUT_U8 first, then GRAY8); the same holds for rip_fused. */
int rip_sobel(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width,
              int height, int n_frames, int in_format);

/* Fused gray -> K x K Gaussian -> Sobel in one kernel, one HBM round trip per frame, for every
 * shape and kernel size.  Processes output rows [out_row0, out_row0 + out_rows) of
 * frames whose true height is `height`; d_in holds input rows [in_row0, in_row0 + in_rows) of each
 * frame (a row band with halo: it must cover out rows extended by ksize/2 + 1 rows each side, clipped to
 * the image, and may hold more rows than that, up to the whole frame; a band that misses a needed row, or
 * reaches past row height - 1, fails with RIP_EINVAL).  For whole frames pass in_row0 = out_row0 = 0 and
 * in_rows = out_rows = height.
 * d_out holds out_rows * width bytes per frame.  d_workspace and workspace_bytes are unused (pass
 * NULL, 0); they stay in the signature for ABI compatibility. */
int rip_fused(int device, rip_stream stream, const uint8_t *d_in, uint8_t *d_out, int width,
              int height, int n_frames, int in_format, int ksize, const float *weights,
              int in_row0, int in_rows, int out_row0, int out_rows, void *d_workspace,
              size_t workspace_bytes);
/* bytes of d_workspace rip_fused needs for this shape: always 0 (rip_fused needs no workspace);
 * still rejects a non-positive shape */
int rip_fused_workspace_bytes(int width, int in_rows, int n_frames, int ksize, size_t *bytes);

/* counters: kernels launched by this library in this process (all threads) */
int rip_launch_count(uint64_t *launches);
/* diagnostics: count the pixels of rip_fused that took the exact 25-tap replay instead of the
 * separable fast path.  enable != 0 starts (and zeroes) the counter on `device`; every call
 * returns the count accumulated since the previous call.  Not for production (adds an atomic). */
int rip_debug_slow_path_stats(int device, int enable, uint64_t *slow_pixels);
/* diagnostics: exhaustive on-device check of the fused kernel's arithmetic shortcuts (approximate
 * sqrt + magic-number rounding for every reachable gx^2+gy^2; dot-product gray for all 2^24
 * triples) against the plain exact formulations.  mismatches must come back 0. */
int rip_debug_selftest(int device, uint64_t *checked, uint64_t *mismatches);
/* diagnostics: experiment switches (kernel selection for A/B runs and for the tests that compare kernels).  They are
 * read from the environment once, at first use (RIP_FUSED_SEG, RIP_FUSED_NPX, RIP_FUSED_GENERIC,
 * RIP_BLUR_EXACT, RIP_BLUR_TILED, RIP_BLUR_STREAM); afterwards only this call changes them, so no launch path calls
 * getenv().  `name` is the variable name with or without the RIP_ prefix.  The reference has no counterpart (its
 * switches are file-scope globals, RealtimeImageProcessing.cpp:10-30). */
int rip_debug_set_option(const char *name, int value);

/* ---- host-buffer pipeline: what Controller::PerformCL* calls.  Shards n_frames over the devices of
 *      ctx (contiguous blocks of frames per device, no inter-device traffic), and per device runs
 *      H2D -> kernel -> D2H on cached device buffers with the copies of consecutive chunks
 *      overlapped.  Every device of a context has one persistent worker thread that owns its streams,
 *      device buffers and pinned staging buffers: no call creates a thread, and any number of host
 *      threads may use one context concurrently.  h_in / h_out may be pinned (rip_malloc_pinned,
 *      rip_host_register: copied by DMA directly) or pageable (std::vector, cv::Mat: staged through
 *      the context's pinned buffers, the staging copy of one chunk overlapping the DMA of the previous).
 *      rip_process_host is blocking: it returns with h_out filled, like the reference's PerformCL*
 *      (RT/src/Controller.cpp:429-744: three blocking waits per call).  rip_submit / rip_collect is
 *      the same pipeline split in two, so that the frames of a stream overlap: frame i+1 uploads while
 *      frame i computes and frame i-1 downloads (ProgramHandler.cpp:259-329 is called once per camera
 *      frame, RealtimeImageProcessing.cpp:355-403).  Jobs of one context complete in submission order.
 *      prof_ns (may be NULL) receives [write_start, write_end, kernel_start, kernel_end, read_start,
 *      read_end] in ns relative to the start of the job, measured with CUDA events on device 0 of
 *      the context for its first chunk -- the layout of the reference's profiling_events
 *      (RT/src/Controller.cpp:66-74). ---- */
typedef struct rip_op_desc {
    int op;          /* RIP_OP_* */
    int in_format;   /* RIP_FMT_* of h_in */
    int gray_out;    /* RIP_GRAY_OUT_* (RIP_OP_GRAY only) */
    int ksize;       /* GAUSSIAN / FUSED */
    const float *weights; /* ksize*ksize host floats (GAUSSIAN / FUSED) */
} rip_op_desc;

int rip_out_bytes_per_frame(const rip_op_desc *desc, int width, int height, size_t *bytes);
int rip_process_host(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                     int width, int height, int n_frames, uint64_t prof_ns[6]);
/* asynchronous form.  rip_submit copies the descriptor and the weights, queues the job on the device workers and
 * returns at once; h_in must stay valid and h_out untouched until rip_collect(ticket) has returned.  flags:
 * RIP_SUBMIT_BANDED = one frame split into row bands (as rip_process_host_banded), RIP_SUBMIT_PROFILE = record the
 * events behind prof_ns.  rip_collect blocks until the job is done, frees the ticket and returns the job's status;
 * rip_ticket_done polls.  Every ticket must be collected exactly once, before rip_ctx_destroy. */
#define RIP_SUBMIT_BANDED 1
#define RIP_SUBMIT_PROFILE 2
int rip_submit(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in, uint8_t *h_out, int width, int height,
               int n_frames, int flags, rip_ticket **ticket);
int rip_ticket_done(rip_ticket *ticket, int *done);
int rip_collect(rip_ticket *ticket, uint64_t prof_ns[6]);
/* page-lock / release memory the caller owns (cudaHostRegister), so that the pipeline copies it by DMA without the
 * staging copy -- for a std::vector or cv::Mat that is reused across calls (the reference's iteration loop hands the
 * same input_data to PerformCL* 100 times, ProgramHandler.cpp:157-216). */
int rip_host_register(void *h_ptr, size_t bytes);
int rip_host_unregister(void *h_ptr);
/* The partitions the two host pipelines use (pure host arithmetic, exported so that callers and tests
 * see exactly the split that runs): part `index` of `n_parts` owns frames [first, first + count) of a
 * batch, or output rows [out_row0, out_row0 + out_rows) of a frame, for which it needs input rows
 * [in_row0, in_row0 + in_rows) (halo = ksize/2 + 1 for FUSED, 1 for EDGE; clipped to the image). */
int rip_shard_frames(int n_frames, int n_parts, int index, int *first, int *count);
int rip_band_rows(int height, int n_parts, int index, int halo, int *in_row0, int *in_rows,
                  int *out_row0, int *out_rows);
/* one large frame split into row bands (one per device of ctx, halo rows replicated from the
 * source frame; SURVEY.md 8e).  RIP_OP_FUSED and RIP_OP_EDGE only. */
int rip_process_host_banded(rip_ctx *ctx, const rip_op_desc *desc, const uint8_t *h_in,
                            uint8_t *h_out, int width, int height, uint64_t prof_ns[6]);

#ifdef __cplusplus
}
#endif
#endif /* RIP_CUDA_H */
