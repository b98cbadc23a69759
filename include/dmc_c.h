/* dmc_c.h -- C ABI of libdmc_b200.so: the B200 (sm_100a) implementation of the post filter set for decoded
 * depth maps of Wavelet303/DepthMapCompression.
 *
 * The reference has no FFI layer: its boundary is the C++ header PostFilterSetForDepthCoding/filter.h (plus the
 * converter declarations of util.h that the chain uses).  include/filter.h in this repo keeps those declarations
 * byte-for-byte and forwards every call to the entry points below; each entry point names the reference
 * declaration it replaces (paths relative to /root/reference/PostFilterSetForDepthCoding/).
 *
 * Conventions
 *   - plain pointers and sizes only; no exceptions cross this boundary; every call returns a dmc_status.
 *   - an image is {data, rows, cols, cvtype, step, mem}; cvtype is OpenCV's encoding depth + ((channels-1) << 3)
 *     with depth 0 = 8U, 2 = 16U, 3 = 16S, 5 = 32F, 6 = 64F; step is the row pitch in bytes (0 = dense);
 *     mem says whether `data` is host or device memory.  Host images are staged through device memory by the
 *     library (H2D, kernels, D2H) and the call returns when `dst` is valid, like the reference's synchronous API.
 *     Device images are processed in stream order on the context's stream; call dmc_synchronize() (or use your own
 *     stream via dmc_set_stream) before reading them.
 *   - src and dst may alias (in-place is legal for every operator, as in the reference).
 *   - the library never allocates caller-visible memory: dst must be allocated by the caller (include/filter.h does
 *     the `dst.create()` the reference does).
 *   - DMC_UNSUPPORTED mirrors the reference's silent no-ops (e.g. 8U + FULL_KERNEL_PAIR): dst is left untouched.
 *   - one dmc_ctx per (host thread, device); a context is not thread-safe (neither is a PostFilterSet instance).
 *   - there is NO CPU fallback: without a CUDA device dmc_create fails with DMC_ERR_CUDA.
 */
#ifndef DMC_C_H
#define DMC_C_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    DMC_OK = 0,
    DMC_UNSUPPORTED = 1,   /* reference's silent no-op for this (type, method) pair; dst untouched */
    DMC_ERR_TYPE = -1,     /* CV_Assert on type would have fired in the reference */
    DMC_ERR_SIZE = -2,     /* size / step / null-pointer problem */
    DMC_ERR_CUDA = -3,     /* CUDA runtime error (see dmc_last_error) */
    DMC_ERR_ARG = -4       /* invalid parameter (even median size, radius out of range, ...) */
} dmc_status;

enum { DMC_MEM_HOST = 0, DMC_MEM_DEVICE = 1 };
enum { DMC_8U = 0, DMC_16U = 2, DMC_16S = 3, DMC_32F = 5, DMC_64F = 6 };
/* filter.h:23-28 */
enum { DMC_FULL_KERNEL = 0, DMC_FULL_KERNEL_PAIR = 1, DMC_SEPARABLE_KERNEL = 2 };
/* util.h:19-23 */
enum { DMC_FILL_DISPARITY = 0, DMC_FILL_DEPTH = 1 };
/* cv::BORDER_REPLICATE: the only border the reference's range filter is ever called with (filter.h:29 default) */
enum { DMC_BORDER_REPLICATE = 1 };

#define DMC_MAKETYPE(depth, cn) (((depth) & 7) + (((cn) - 1) << 3))
#define DMC_MAX_RADIUS 10   /* trackbar maxima main.cpp:87-93 */

typedef struct dmc_image {
    void* data;
    int rows, cols;
    int cvtype;
    size_t step;   /* bytes per row; 0 = cols * elemSize */
    int mem;       /* DMC_MEM_HOST or DMC_MEM_DEVICE */
} dmc_image;

typedef struct dmc_ctx dmc_ctx;

/* ---- context -------------------------------------------------------------------------------------------- */
int dmc_device_count(void);
int dmc_create(int device, dmc_ctx** out);
void dmc_destroy(dmc_ctx* ctx);
const char* dmc_last_error(const dmc_ctx* ctx);           /* valid until the next call on ctx; ctx may be NULL */
int dmc_set_stream(dmc_ctx* ctx, void* cuda_stream);      /* use the caller's cudaStream_t (NULL = own stream) */
void* dmc_get_stream(dmc_ctx* ctx);
int dmc_synchronize(dmc_ctx* ctx);
uint64_t dmc_kernel_launches(const dmc_ctx* ctx);         /* kernels launched by this context so far */
void* dmc_host_alloc(size_t bytes);                       /* pinned host memory for the streaming entry points */
void dmc_host_free(void* p);
/* Pins and device-maps memory the caller already owns (a cv::Mat's buffer, a numpy array): cudaHostRegister.  Host images of
 * up to 2 MB that lie in pinned memory (this call, dmc_host_alloc, cudaMallocHost) are processed in place over the host link
 * by the single-image entry points -- no staging copies (640x480 filterDisp8U2Depth32F host to host: 152 -> about 50 us).
 * Unregister before the memory is freed. */
int dmc_host_register(void* p, size_t bytes);
int dmc_host_unregister(void* p);
int dmc_version(void);
/* Device-resident frame batches: number of frame groups in flight on separate streams (1..3, default 1). */
int dmc_set_lanes(dmc_ctx* ctx, int lanes);

/* Optional CUDA-event timing of the chain's stages (used by bench.py for the live roofline figure): while a stage's
 * bit is set in stage_mask, every launch of that stage inside the chain entry points is bracketed by an event pair
 * on the launching stream.  dmc_profile_read synchronises, folds the finished pairs into per-stage totals and
 * returns them (pixels = frames x rows x cols the launches covered). */
enum { DMC_STAGE_MEDIAN = 0, DMC_STAGE_GAUSS = 1, DMC_STAGE_MINMAX = 2, DMC_STAGE_RANGE = 3, DMC_STAGE_COUNT = 4 };
int dmc_profile_enable(dmc_ctx* ctx, int stage_mask);
int dmc_profile_read(dmc_ctx* ctx, int stage, double* total_ms, uint64_t* launches, uint64_t* pixels, int reset);

/* ---- PostFilterSet (filter.h:32-42, postFilterSet.cpp:21-63) --------------------------------------------- */
/* PostFilterSet::operator() filter.h:41: 8UC1 -> 8UC1 */
int dmc_post_filter_set(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int median_r, int gaussian_r,
                        int minmax_r, int brange_r, int brange_th, int brange_method);
/* PostFilterSet::filterDisp8U2Depth32F filter.h:38: 8UC1 -> 32FC1 */
int dmc_filter_disp8u_depth32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, double focus, double baseline,
                               double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th,
                               int brange_method);
/* PostFilterSet::filterDisp8U2Depth16U filter.h:39: 8UC1 -> 16UC1 */
int dmc_filter_disp8u_depth16u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, double focus, double baseline,
                               double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th,
                               int brange_method);
/* PostFilterSet::filterDisp8U2Disp32F filter.h:40: 8UC1 -> 16UC1 (sic) */
int dmc_filter_disp8u_disp32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int median_r, int gaussian_r,
                              int minmax_r, int brange_r, float brange_th, int brange_method);

/* Frame batches (video / multi-view): n_frames dense rows x cols frames, back to back, in host or device memory.
 * chain: 0 = operator() (u8 out), 1 = Depth32F (f32 out), 2 = Depth16U (u16 out), 3 = Disp32F (u16 out).
 * With host memory the frames are streamed through the device in chunks over several CUDA streams (H2D of chunk
 * i+1, kernels of chunk i and D2H of chunk i-1 overlap); pinned memory (dmc_host_alloc) is needed for overlap. */
enum { DMC_CHAIN_DISP8U = 0, DMC_CHAIN_DEPTH32F = 1, DMC_CHAIN_DEPTH16U = 2, DMC_CHAIN_DISP32F = 3 };
typedef struct dmc_chain_params {
    int chain;
    int median_r, gaussian_r, minmax_r, brange_r;
    float brange_th;           /* operator(): integer threshold, passed as float like postFilterSet.cpp:62 */
    int brange_method;
    double focus, baseline, amp;   /* depth chains only */
} dmc_chain_params;
int dmc_chain_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols,
                    const dmc_chain_params* p, int mem);
/* The same chain on a batch given as arrays of image descriptors: n_frames CV_8UC1 images of one size, each anywhere in
 * host or device memory with its own row step (e.g. a std::vector<cv::Mat> of video frames or camera views); dsts[i] has
 * the chain's output type.  Frames are packed into dense device buffers chunk by chunk and streamed through the same
 * H2D / kernel / D2H pipeline.  Returns when every dsts[i] is valid. */
int dmc_chain_batch_images(dmc_ctx* ctx, const dmc_image* srcs, dmc_image* dsts, int n_frames, const dmc_chain_params* p);
/* Frame-batch scheduler across the GPUs of one box, in one process (the reference scales by row-striping one image
 * over CPU threads -- cv::parallel_for_, binalyWeightedRangeFilter.cpp:1080; here whole frames go to whole GPUs):
 * one context per listed device, kept between runs; every run cuts the batch into contiguous shards
 * (dmc_shard_frames) and streams each shard through its device on its own host thread, as dmc_chain_batch does.
 * src/dst are HOST buffers (pinned for full overlap).  No data-path exchange between devices: frames are independent. */
typedef struct dmc_sched dmc_sched;
int dmc_sched_create(const int* devices, int n_devices, dmc_sched** out);
void dmc_sched_destroy(dmc_sched* sched);
int dmc_sched_device_count(const dmc_sched* sched);
const char* dmc_sched_last_error(const dmc_sched* sched);
int dmc_sched_chain_batch(dmc_sched* sched, const void* src, void* dst, int n_frames, int rows, int cols, const dmc_chain_params* p);
/* one-shot convenience: create, run, destroy; on error the message is copied into err (may be NULL) */
int dmc_multi_chain_batch(const int* devices, int n_devices, const void* src, void* dst, int n_frames, int rows, int cols,
                          const dmc_chain_params* p, char* err, size_t err_len);
/* Host-link topology.  Every frame of a host-resident batch crosses the host link twice, and on a multi-GPU box the
 * link is not uniform (profiles/r02_hostlink.json: one group of four B200s shares ~51 GB/s each way, the other four reach
 * ~94 GB/s together, all eight together only ~64 GB/s).  dmc_hostlink_probe copies 64 MB blocks both ways on all listed
 * devices at once (~0.1 s, call it while the devices are otherwise idle), then on the subset with the best per-device rate
 * alone, and proposes a routing: gateway[i] is the device whose link should carry device[i]'s host traffic (itself when
 * its own link is as good as any).  dmc_set_gateway makes the host-memory batch entry points of a context stage through
 * the gateway's HBM: H2D / D2H run on the gateway's copy engines, the context's kernels read their input from and write
 * their output to the gateway's memory directly over NVLink / NVSwitch (peer access), no extra copy.  Results are
 * unchanged (bit-identical); -1 restores the context's own link.  dmc_sched_create probes and routes by itself
 * (DMC_NO_TOPOLOGY=1 disables that). */
#define DMC_MAX_DEVICES 16
typedef struct dmc_hostlink_info {
    int n_devices;
    int device[DMC_MAX_DEVICES];
    int gateway[DMC_MAX_DEVICES];        /* proposed routing */
    double loaded_gbs[DMC_MAX_DEVICES];  /* GB/s each way of device[i] while ALL listed devices copy both ways at once */
    double all_gbs;                      /* aggregate GB/s each way, all listed devices on their own links */
    double best_gbs;                     /* aggregate GB/s each way of the proposed link set (== all_gbs if nothing is re-routed) */
    int n_link;                          /* devices whose links carry traffic under the proposed routing */
} dmc_hostlink_info;
int dmc_hostlink_probe(const int* devices, int n_devices, dmc_hostlink_info* info);
/* cudaDeviceReset of a device this process only probed (no live allocations / contexts of the caller on it); the calling
 * thread's current device is `device` afterwards */
int dmc_release_device(int device);
int dmc_set_gateway(dmc_ctx* ctx, int gateway_device);
int dmc_get_gateway(const dmc_ctx* ctx);
/* routing chosen by the scheduler at creation: gateways[i] for the i-th device, -1 = own link */
int dmc_sched_get_routing(const dmc_sched* sched, int* gateways, double* all_gbs, double* best_gbs);

/* Frame-parallel sharding of a batch over `world` ranks (one process per GPU, no collective): frames
 * [*begin, *begin + *count) belong to `rank` (contiguous blocks, sizes differ by at most one). */
int dmc_shard_frames(int n_frames, int rank, int world, int* begin, int* count);

/* ---- decode feeding the chain (SURVEY.md 8f-1) ------------------------------------------------------------ */
/* Frame-parallel baseline JPEG decode (SOF0, 8-bit, single component), bit-identical to libjpeg(-turbo)'s default
 * JDCT_ISLOW decoder, i.e. to the reference's imdecode(buf, 0) (main.cpp:284, :521) and jpeg_decode()
 * (jpegTurboDemo.cpp:217-271).  `blob` is HOST memory holding the n_frames bitstreams; stream i occupies
 * [offsets[i], offsets[i+1]).  All frames must be rows x cols.  dst receives n_frames dense 8UC1 frames
 * (dst_mem: host or device; with device memory the chain entry points can consume it without leaving the GPU). */
int dmc_jpeg_decode_gray_batch(dmc_ctx* ctx, const void* blob, const uint64_t* offsets, int n_frames, int rows, int cols,
                               void* dst, int dst_mem);
/* Streamed bitstream -> chain (the reference's pointcloudTest loop main.cpp:276-303 for a whole batch): JPEG streams in
 * HOST memory (pinned for full overlap) are copied to the device (about 1/30 of the bytes of the decoded frames), decoded
 * there and run through the chain of *p without leaving the device; dst receives n_frames frames of the chain's output type
 * (dst_mem: host -- pinned for overlap -- or device).  Chunks of frames flow through the same 4-slot H2D / kernels / D2H
 * pipeline as dmc_chain_batch, with no host synchronisation between chunks.  Returns when dst is valid (host) or when the
 * work is queued (device: dmc_synchronize before reading). */
int dmc_chain_batch_jpeg(dmc_ctx* ctx, const void* blob, const uint64_t* offsets, int n_frames, int rows, int cols,
                         void* dst, int dst_mem, const dmc_chain_params* p);
/* Host-only: parses the headers of one stream, reports its size and whether this library can decode it (DMC_OK) or why
 * not (DMC_ERR_TYPE + message in err, may be NULL).  Needs no context and no GPU.  Malformed, truncated or hostile
 * streams (bad segment lengths, Huffman tables that are not prefix codes, ...) are refused here, never crashed on. */
int dmc_jpeg_probe(const void* stream, size_t len, int* rows, int* cols, char* err, size_t err_len);
/* Frame-parallel baseline colour JPEG decode.  The output of frame i is a dense rows x cols 8UC3 BGR image equal to
 * cv::imdecode(buf, IMREAD_COLOR | IMREAD_IGNORE_ORIENTATION) with libjpeg-turbo 3.1.2 (cv2 4.13): islow IDCT, fancy
 * upsampling, libjpeg's YCbCr -> RGB tables; pixels as stored, so for streams without an EXIF orientation tag (cv2's own
 * streams never carry one) it is plain IMREAD_COLOR.  Accepted: SOF0 / SOF1 at 8-bit precision with three components in
 * one interleaved scan, chroma sampled 1x1 and luma 1x1, 2x1, 2x2, 1x2 or 4x1 (4:4:4, 4:2:2, 4:2:0, 4:4:0, 4:1:1: every
 * sampling cv::imencode writes), standard or optimised Huffman tables, with or without restart intervals; and
 * one-component streams, which decode to B = G = R = Y.  Refused with a reason (DMC_ERR_TYPE): progressive, arithmetic,
 * lossless, 12-bit, non-interleaved multi-scan colour, CMYK / YCCK, and streams libjpeg treats as RGB (Adobe transform 0
 * without JFIF, or component IDs 'R' 'G' 'B' without JFIF or Adobe markers).  blob / offsets as for
 * dmc_jpeg_decode_gray_batch; one batch may mix samplings, table kinds and component counts at one rows x cols.
 * dst receives n_frames x rows x cols x 3 bytes (dst_mem: host or device; a device dst is a texture batch that
 * dmc_render_view_batch takes as it is).  Returns when dst is valid. */
int dmc_jpeg_decode_color_batch(dmc_ctx* ctx, const void* blob, const uint64_t* offsets, int n_frames, int rows, int cols,
                                void* dst, int dst_mem);
/* Host-only: whether dmc_jpeg_decode_color_batch can decode this stream (DMC_OK, with its size and component count, 1 or
 * 3) or why not (DMC_ERR_TYPE + message in err, may be NULL).  Needs no context and no GPU. */
int dmc_jpeg_probe_color(const void* stream, size_t len, int* rows, int* cols, int* components, char* err, size_t err_len);

/* ---- encode (SURVEY.md 8f-5) ----------------------------------------------------------------------------------- */
/* Baseline JPEG encoding of 8UC1 frames, byte-identical to cv::imencode(".jpg", img, {IMWRITE_JPEG_QUALITY, quality}) with
 * libjpeg-turbo (the encoder behind the reference's degradeJPEG): standard luminance tables scaled by quality, islow FDCT,
 * no restart intervals, the standard Huffman tables of ITU T.81 K.3 / K.5.  The _ex entry points take `flags`:
 *   0                          the calls without _ex, same bytes;
 *   DMC_JPEG_OPTIMIZE_HUFFMAN  every frame gets its own optimal Huffman tables, built from its own symbol counts as
 *                              libjpeg's optimize_coding builds them: byte-identical to cv::imencode(".jpg", img,
 *                              {IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_OPTIMIZE, 1}).  The same decoded pixels
 *                              in fewer bytes (the header's two DHT segments and the scan differ).
 * Any other flag bit is DMC_ERR_ARG.
 *
 * Host only, needs no GPU: the worst-case stream size of one rows x cols frame.  DMC_ERR_SIZE for sizes outside
 * 1..65535 and for frames whose bound exceeds 256 MB (the decoder's scan limit; *bytes still holds the bound). */
enum { DMC_JPEG_OPTIMIZE_HUFFMAN = 1 };   /* cv::IMWRITE_JPEG_OPTIMIZE = 1 */
int dmc_jpeg_encode_bound(int rows, int cols, uint64_t* bytes);
/* The bound of a stream encoded with `flags` (with DMC_JPEG_OPTIMIZE_HUFFMAN a little larger: 1661 instead of 1658 bits
 * per 8x8 block). */
int dmc_jpeg_encode_bound_ex(int rows, int cols, int flags, uint64_t* bytes);
/* src: n_frames dense rows x cols frames (src_mem: host or device).  The streams are written back to back into blob
 * (blob_mem: host or device); offsets (host, n_frames + 1 entries) receives their layout -- stream i occupies
 * [offsets[i], offsets[i+1]) -- which dmc_jpeg_decode_gray_batch and dmc_chain_batch_jpeg take as it is.  quality in
 * 0..100 (0 acts as 1, as in cv::imencode), anything else is DMC_ERR_ARG.  If the streams do not fit into `capacity`
 * bytes the call returns DMC_ERR_SIZE and writes nothing at or past blob + capacity; n_frames x dmc_jpeg_encode_bound
 * always suffices.  Returns when offsets and blob are valid. */
int dmc_jpeg_encode_gray_batch(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, int quality,
                               void* blob, int blob_mem, uint64_t capacity, uint64_t* offsets);
/* The same with flags; n_frames x dmc_jpeg_encode_bound_ex(rows, cols, flags) always suffices. */
int dmc_jpeg_encode_gray_batch_ex(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, int quality, int flags,
                                  void* blob, int blob_mem, uint64_t capacity, uint64_t* offsets);
/* The reference's degradeJPEG for a batch, entirely on the device: dst = cv::imdecode(cv::imencode(src, quality), 0) for
 * every frame (src, dst: n_frames dense 8UC1 frames in `mem`; they may alias).  bytes (host, n_frames entries, may be NULL)
 * receives the stream sizes, i.e. the bitrate.  The streams themselves never leave the device.  Returns when dst and
 * bytes are valid. */
int dmc_jpeg_degrade_gray_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, int quality, int mem,
                                uint64_t* bytes);
/* The same with flags: with DMC_JPEG_OPTIMIZE_HUFFMAN dst is unchanged (the coefficients are the same) and bytes receives
 * the sizes of the optimised streams. */
int dmc_jpeg_degrade_gray_batch_ex(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, int quality, int flags,
                                   int mem, uint64_t* bytes);

/* Baseline colour JPEG encoding of dense 8UC3 BGR frames, byte-identical to cv::imencode(".jpg", img,
 * {IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_SAMPLING_FACTOR, sampling}) with libjpeg-turbo 3.1.2 (cv2 4.13): libjpeg's
 * RGB -> YCbCr conversion and chroma downsampling (no smoothing), the standard luminance and chrominance tables of ITU
 * T.81 K.1-K.6 scaled by quality, one interleaved scan, no restart intervals.  `sampling` is one of cv::IMWRITE_JPEG_SAMPLING_
 * FACTOR_*'s values below (anything else is DMC_ERR_ARG); cv::imencode's default is 4:2:0.  Other rules as for the gray
 * encoder: quality 0..100, sizes 1..65535, DMC_ERR_SIZE for frames whose bound exceeds 256 MB. */
enum {
    DMC_JPEG_SAMPLING_444 = 0x111111,
    DMC_JPEG_SAMPLING_422 = 0x211111,
    DMC_JPEG_SAMPLING_420 = 0x221111,
    DMC_JPEG_SAMPLING_440 = 0x121111,
    DMC_JPEG_SAMPLING_411 = 0x411111
};
/* Host only, needs no GPU: the worst-case stream size of one rows x cols colour frame (1660 bits per 8x8 block, the dummy
 * blocks of partial MCUs included). */
int dmc_jpeg_encode_color_bound(int rows, int cols, int sampling, uint64_t* bytes);
/* src: n_frames dense rows x cols x 3 frames (src_mem: host or device).  blob, capacity and offsets as for
 * dmc_jpeg_encode_gray_batch (n_frames x dmc_jpeg_encode_color_bound always suffices); dmc_jpeg_decode_color_batch takes
 * blob and offsets as they are.  Returns when offsets and blob are valid. */
int dmc_jpeg_encode_color_batch(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, int quality, int sampling,
                                void* blob, int blob_mem, uint64_t capacity, uint64_t* offsets);
/* A colour JPEG round trip for a batch, entirely on the device: dst = cv::imdecode(cv::imencode(src, {QUALITY, quality,
 * SAMPLING_FACTOR, sampling}), IMREAD_COLOR) for every frame (src, dst: n_frames dense 8UC3 frames in `mem`; they may
 * alias).  bytes (host, n_frames entries, may be NULL) receives the stream sizes.  Returns when dst and bytes are valid. */
int dmc_jpeg_degrade_color_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, int quality, int sampling,
                                 int mem, uint64_t* bytes);

/* ---- distortion and the JPEG rate-distortion sweep ---------------------------------------------------------- */
/* Per-frame sum of squared differences of two batches of n dense rows x cols 8UC1 frames (both in `mem`), exact:
 * sse[i] = sum over the pixels of (a_i - b_i)^2 (host, n_frames entries).  a and b may be the same pointer.
 * Returns when sse is valid. */
int dmc_sse_gray_batch(dmc_ctx* ctx, const void* a, const void* b, int n_frames, int rows, int cols, int mem, uint64_t* sse);
/* Host only, no GPU: PSNR in dB of an 8-bit frame of `pixels` pixels with sum of squared differences `sse`, by the formula of
 * cv::PSNR: 20*log10(255 / (sqrt(sse / pixels) + DBL_EPSILON)) -- identical frames give 361.20199909921956, as cv2.PSNR does. */
double dmc_psnr_from_sse(uint64_t sse, uint64_t pixels);
/* The rate-distortion sweep: for every quality qualities[k] and every frame i of src (n dense 8UC1 frames, src_mem host or
 * device): bytes[k*n+i]        = size of cv::imencode(frame, {QUALITY, q} [+ OPTIMIZE with DMC_JPEG_OPTIMIZE_HUFFMAN]),
 *          sse_coded[k*n+i]    = SSE(frame, imdecode(that stream)),
 *          sse_filtered[k*n+i] = SSE(frame, chain(imdecode(that stream))) -- only when p != NULL; p->chain must be DMC_CHAIN_DISP8U.
 * No stream and no decoded or filtered frame leaves the device.  Outputs are host arrays of n_q * n_frames entries.
 * DMC_ERR_ARG (nothing written): n_q < 1, a quality outside 0..100 (0 acts as 1, as in cv::imencode), unknown flag bits,
 * a chain other than DMC_CHAIN_DISP8U, a bad radius, or a brange_method other than FULL_KERNEL / SEPARABLE_KERNEL (the
 * 8-bit chain writes nothing for the others).  p == NULL: sse_filtered may be NULL and is not written.  Sizes follow
 * dmc_jpeg_encode_bound_ex.  Returns when the outputs are valid. */
int dmc_jpeg_rd_sweep(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, const int* qualities, int n_q,
                      int flags, const dmc_chain_params* p, uint64_t* bytes, uint64_t* sse_coded, uint64_t* sse_filtered);

/* ---- the boundary reconstruction filter on frame batches, and as a third arm of both sweeps ---------------------------- */
/* Parameters of boundaryReconstructionFilter(src, dest, Size(kernel_w, kernel_h), frec, color, space) (filter.h:45). */
typedef struct dmc_brf_params { int kernel_w, kernel_h; float frec, color, space; } dmc_brf_params;
/* boundaryReconstructionFilter (filter.h:45) on n dense single-channel frames of one depth (DMC_8U/16U/16S/32F/64F), host or device memory.
 * src and dst hold n_frames dense rows x cols frames back to back in `mem`; each frame of dst equals dmc_boundary_reconstruction
 * of that frame.  Device memory: one launch per group of frames, in stream order (dmc_synchronize before reading dst).  Host
 * memory: chunks stream through the device as in dmc_chain_batch (pinned memory for overlap); returns when dst is valid.
 * src == dst is legal, and so is any overlap.  Device memory: where dst overlaps src, each group of frames (~256 MB) is filtered
 * into scratch of the group's size and copied to dst, so an in-place batch costs one group of device memory and one extra
 * device-to-device copy of the batch.  Host memory: in place needs nothing extra; a partly overlapping source is copied on the
 * host first.  DMC_ERR_ARG: b == NULL, a kernel side < 1 or a radius
 * (side / 2) above DMC_MAX_RADIUS, a window the kernel cannot take; DMC_ERR_TYPE: another depth; nothing is written on error. */
int dmc_brf_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, int depth, const dmc_brf_params* b, int mem);
/* dmc_jpeg_rd_sweep with a third arm.  b == NULL: exactly dmc_jpeg_rd_sweep (sse_brf may be NULL and is not written).  With b,
 * B(x) = boundaryReconstructionFilter(x, Size(b->kernel_w, b->kernel_h), b->frec, b->color, b->space) on the 8-bit decoded
 * disparity and
 *          sse_brf[k*n+i]      = SSE(frame_i, B(imdecode(that stream))).
 * The reference never runs this comparison: pointcloudTest keeps the call boundaryReconstructionFilter(disp, disp, Size(13,13),
 * 1, 1, 1) on the decoded disparity commented out (main.cpp:306-311).  Placing B there, in place of the post filter set, is this
 * library's definition.  b's argument rules are those of dmc_brf_batch (DMC_ERR_ARG, nothing written); p may be NULL with b set. */
int dmc_jpeg_rd_sweep_ex(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, const int* qualities, int n_q,
                         int flags, const dmc_chain_params* p, const dmc_brf_params* b, uint64_t* bytes, uint64_t* sse_coded,
                         uint64_t* sse_filtered, uint64_t* sse_brf);

/* ---- structural similarity (SSIM) ---------------------------------------------------------------------------------------- */
/* Per-frame mean structural similarity of two batches of n dense rows x cols 8-bit frames of `channels` interleaved channels
 * (1: 8UC1, 3: 8UC3 such as the sweeps' BGR views), both in `mem`; mssim (host, n_frames entries).  The definition is that of
 * Wang, Bovik, Sheikh and Simoncelli (2004), ssim_index.m, and of skimage.metrics.structural_similarity(a, b, data_range=255,
 * gaussian_weights=True, sigma=1.5, use_sample_covariance=False[, channel_axis=-1]):
 *   window   w = g g^T, g_i = exp(-i^2 / 4.5) for i = -5..5, normalised to sum 1 in double;
 *   at every window position that lies wholly inside the frame ((rows - 10) x (cols - 10) of them), per channel:
 *            mu_x = sum w x, mu_y = sum w y, s_x = sum w x^2 - mu_x^2, s_y = sum w y^2 - mu_y^2, s_xy = sum w x y - mu_x mu_y,
 *            S = ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_x + s_y + C2)),  C1 = (0.01 * 255)^2, C2 = (0.03 * 255)^2;
 *   MSSIM    the mean of S over the positions; with 3 channels the mean of the three channels' MSSIMs.
 * Computed in FP64 (in FP32, E[x^2] - mu^2 cancels to about 4e-3 on sigma^2 near 255).  Deterministic: a frame's result is
 * the same bits alone, in any batch, inside a sweep, from host or device memory.  a == b and any alignment are legal.
 * DMC_ERR_ARG: channels not 1 or 3, a bad mem; DMC_ERR_SIZE: rows or cols below 11, a negative count, a NULL pointer;
 * nothing is written on error.  Returns when mssim is valid. */
int dmc_ssim_batch(dmc_ctx* ctx, const void* a, const void* b, int n_frames, int rows, int cols, int channels, int mem, double* mssim);
/* dmc_jpeg_rd_sweep_ex with SSIM outputs, in the layout of the SSE arrays ([k*n+i]): ssim_coded = MSSIM(frame, decoded),
 * ssim_filtered = MSSIM(frame, chain(decoded)), ssim_brf = MSSIM(frame, B(decoded)).  SSIM is computed iff ssim_coded != NULL;
 * then ssim_filtered is required iff p != NULL and ssim_brf iff b != NULL (DMC_ERR_SIZE), and frames below 11 x 11 are
 * DMC_ERR_SIZE.  With ssim_coded == NULL this is dmc_jpeg_rd_sweep_ex: the same launches, the same results.  bytes and the SSE
 * outputs are the same with and without SSIM. */
int dmc_jpeg_rd_sweep_ssim(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, const int* qualities, int n_q,
                           int flags, const dmc_chain_params* p, const dmc_brf_params* b, uint64_t* bytes, uint64_t* sse_coded,
                           uint64_t* sse_filtered, uint64_t* sse_brf, double* ssim_coded, double* ssim_filtered, double* ssim_brf);
/* dmc_jpeg_view_rd_sweep_ex with SSIM outputs of the 8UC3 views, in the layout of the SSE arrays ([(k*n_views + v)*n + i]):
 * MSSIM(view(D(disp_i)), the arm's view).  SSIM is computed iff ssim_view_coded != NULL; then ssim_view_filtered is required and
 * ssim_view_brf iff b != NULL (DMC_ERR_SIZE), and frames below 11 x 11 are DMC_ERR_SIZE.  With ssim_view_coded == NULL this is
 * dmc_jpeg_view_rd_sweep_ex. */
int dmc_jpeg_view_rd_sweep_ssim(dmc_ctx* ctx, const void* disp, const void* texture, int src_mem, int n_frames, int rows, int cols,
                                const int* qualities, int n_q, int flags, const dmc_chain_params* p, const dmc_brf_params* b, double f,
                                const double* R, const double* t, int n_views, const double* K, int is_sub, int render_flags,
                                uint64_t* bytes, uint64_t* sse_view_coded, uint64_t* sse_view_filtered, uint64_t* sse_view_brf,
                                double* ssim_view_coded, double* ssim_view_filtered, double* ssim_view_brf);

/* ---- stand-alone operators of filter.h ------------------------------------------------------------------- */
/* binalyWeightedRangeFilter filter.h:29 (binalyWeightedRangeFilter.cpp:1106): 8U/16S/16U/32F x C1/C3 */
int dmc_bwrf(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kernel_w, int kernel_h, float threshold,
             int method, int border_type);
/* Joint (guided) binary-weighted range filter -- an EXTENSION with no counterpart in the reference (SURVEY.md section 8f-4):
 * src (CV_8UC1) is averaged over the window of binalyWeightedRangeFilter with the binary weights computed on `guide`
 * (CV_8UC3: saturated L1 colour distance of binalyWeightedRangeFilter.cpp:297-301; CV_8UC1: absolute difference) instead
 * of on src itself.  Same window, border (REPLICATE), (uchar)threshold, division and rounding as the 8UC1 filter; with
 * guide == src the result equals dmc_bwrf.  method must be DMC_FULL_KERNEL. */
int dmc_joint_bwrf(dmc_ctx* ctx, const dmc_image* src, const dmc_image* guide, dmc_image* dst, int kernel_w, int kernel_h,
                   float threshold, int method);
/* blurRemoveMinMax filter.h:19 (minmaxFilter.cpp:176), blurRemoveMinMaxBase filter.h:20 (:216): same result */
int dmc_blur_remove_minmax(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int r);
/* maxFilter / minFilter filter.h:17-18 (minmaxFilter.cpp:314, :394): single channel 8U/16S/16U/32F */
int dmc_max_filter(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kernel_w, int kernel_h, int border_type);
int dmc_min_filter(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kernel_w, int kernel_h, int border_type);
/* boundaryReconstructionFilter filter.h:45 (boundaryReconstructionFilter.cpp:133): single channel, 5 depths */
int dmc_boundary_reconstruction(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kernel_w, int kernel_h,
                                float frec, float color, float space);
/* Fused min-max -> boundary reconstruction -- an EXTENSION (SURVEY.md section 8f-4, BASELINE north_star): the result of
 * dmc_blur_remove_minmax(src, tmp, minmax_r) followed by dmc_boundary_reconstruction(tmp, dst, ...) in ONE kernel: the
 * min-max image is produced tile by tile in shared memory and never written to HBM, so src is read once.  Single channel
 * 8U / 16U / 16S (the integer depths of minmaxFilter.cpp:48-174); bit-identical to the two calls. */
int dmc_minmax_boundary_reconstruction(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int minmax_r, int kernel_w, int kernel_h,
                                       float frec, float color, float space);
/* smallGaussianBlur filter.h:14 (postFilterSet.cpp:4-16): 8UC1 */
int dmc_small_gaussian(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int d, double sigma);
/* cv::medianBlur as called at postFilterSet.cpp:23,36,47,59: 8UC1, odd ksize */
int dmc_median_blur(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int ksize);

/* ---- depthmapUtil.cpp helpers on the filter path (util.h:16-28) ------------------------------------------- */
int dmc_disp8u2depth32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float focal_baseline, float a, float b);   /* util.h:28 */
int dmc_depth32f2disp8u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float focal_baseline, float a, float b);   /* util.h:25 */
int dmc_depth16u2disp8u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float focal_baseline, float a, float b);   /* util.h:27 */
int dmc_disp16s2depth16u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float focal_baseline, float a, float b);  /* util.h:26 */
int dmc_fill_occlusion(dmc_ctx* ctx, dmc_image* img, int invalid_value, int disp_or_depth);                           /* util.h:24 */
/* cv::transpose as used between the two fillOcclusion passes of pointcloudTest (main.cpp:258, :260); single channel */
int dmc_transpose(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst);
/* reprojectXYZ(depth, xyz, f) util.h:11: xyz is (rows*cols) x 1 32FC3, dense */
int dmc_reproject_xyz(dmc_ctx* ctx, const dmc_image* depth, dmc_image* xyz, double f);

/* splitBGRLineInterleave filter.h:12 (split.cpp:167-177): 8UC3 / 32FC3 -> single channel 3*rows x cols (a B, a G and an R
 * row per image row: the layout the reference's SSE range filter works on); other types are a silent no-op */
int dmc_split_bgr_line_interleave(dmc_ctx* ctx, const dmc_image* src, dmc_image* dest);

/* ---- point-cloud render (SURVEY.md 8f-3; util.h:12-13, :25, :33) ------------------------------------------- */
/* R (3x3), t (3), K (3x3) are row-major doubles (the reference asserts CV_64F, depthmapUtil.cpp:290-294).
 * flags: DMC_RENDER_EXACT_DIVIDE replaces the reference's _mm_rcp_ps (depthmapUtil.cpp:78, emulated from Intel's table)
 * by a true division for every point (the reference's own scalar twin myProjectPoint_BF :99-146). */
enum { DMC_RENDER_EXACT_DIVIDE = 1 };
/* projectPointsSimple util.h:33 (depthmapUtil.cpp:148): xyz 32FC3 (n x 1, dense) -> pt 32FC2 (n x 1, dense) */
int dmc_project_points(dmc_ctx* ctx, const dmc_image* xyz, const double* R, const double* t, const double* K, dmc_image* pt, int flags);
/* projectImagefromXYZ util.h:12-13 (depthmapUtil.cpp:285-448): z-buffer splat of `image` (8UC3) at the projected positions
 * of xyz (32FC3, one point per pixel, dense) into destimage (8UC3, cleared first); depth (32FC1) and pt (32FC2) are the
 * optional outputs of the second overload (NULL to skip).  The reference's SERIAL raster-order semantics (a point tries its
 * neighbour pixels only if it won its own pixel at that moment; isSub quirks included) are reproduced exactly, see
 * csrc/dmc_render.cu.  Synchronous: returns when the outputs are complete. */
int dmc_project_image_from_xyz(dmc_ctx* ctx, const dmc_image* image, dmc_image* destimage, const dmc_image* xyz, const double* R,
                               const double* t, const double* K, int is_sub, dmc_image* depth, dmc_image* pt, int flags);
/* fillSmallHole util.h:25 (depthmapUtil.cpp:187-283): 8UC3; only hole pixels (green == 0) of the interior are written,
 * dest keeps everything else (call it in place, like main.cpp:355, or with dest pre-filled). */
int dmc_fill_small_hole(dmc_ctx* ctx, const dmc_image* src, dmc_image* dest);

/* ---- the view-synthesis rate-distortion sweep ------------------------------------------------------------------- */
/* Scores coded depth by the views it renders, as pointcloudTest (main.cpp:276-373) consumes a decoded depth map.  For every
 * frame i of disp (n dense 8UC1 disparity frames) with its texture i (n dense 8UC3 images, the pixels that are splatted, in
 * the same memory src_mem as disp), every camera v (R + 9v, t + 3v: row-major doubles; K shared) and every qualities[k]:
 *   D(x)     = disp8U2depth32F(x, (float)(p->focus * p->baseline), (float)p->amp, 0), the unfiltered depth.  It equals the
 *              32F chain with all four radii 0 except where x is 0: there D is +inf and the chain NaN, and neither point is
 *              drawn, so the views are the same;
 *   view(z)  = fillSmallHole(projectImagefromXYZ(texture_i, reprojectXYZ(z, f), R_v, t_v, K, is_sub)), the fill in place
 *              as at main.cpp:355;
 *   dec      = imdecode(imencode(disp_i, {QUALITY, q} [+ OPTIMIZE with DMC_JPEG_OPTIMIZE_HUFFMAN]));
 *   bytes[k*n + i]                          = the size of that stream (as dmc_jpeg_rd_sweep reports it);
 *   sse_view_coded[(k*n_views + v)*n + i]    = SSE(view(D(disp_i)), view(D(dec))), over all 3*rows*cols bytes;
 *   sse_view_filtered[(k*n_views + v)*n + i] = SSE(view(D(disp_i)), view(filterDisp8U2Depth32F(dec, p))).
 * PSNR of a view is dmc_psnr_from_sse(sse, 3*rows*cols), which is cv::PSNR of the two 8UC3 images.  p->chain must be
 * DMC_CHAIN_DEPTH32F (focus, baseline, amp and the radii of pointcloudTest's filter); render_flags: DMC_RENDER_EXACT_DIVIDE
 * or 0, as the flags of dmc_project_image_from_xyz.  No frame, stream or view leaves the device.
 * DMC_ERR_ARG (nothing written): n_q < 1, a quality outside 0..100, unknown flags or render_flags bits, p == NULL, a chain
 * other than DMC_CHAIN_DEPTH32F, a bad radius, a brange_method for which the 32F chain writes nothing, n_views < 1 or a NULL
 * camera.  Sizes follow dmc_jpeg_encode_bound_ex and rows * cols < 2^29 (DMC_ERR_SIZE).  Returns when the outputs are valid. */
int dmc_jpeg_view_rd_sweep(dmc_ctx* ctx, const void* disp, const void* texture, int src_mem, int n_frames, int rows, int cols,
                           const int* qualities, int n_q, int flags, const dmc_chain_params* p, double f,
                           const double* R, const double* t, int n_views, const double* K, int is_sub, int render_flags,
                           uint64_t* bytes, uint64_t* sse_view_coded, uint64_t* sse_view_filtered);
/* dmc_jpeg_view_rd_sweep with a third arm.  b == NULL: exactly dmc_jpeg_view_rd_sweep (sse_view_brf may be NULL and is not
 * written).  With b, B as for dmc_jpeg_rd_sweep_ex on the 8-bit decoded disparity, and D and view the sweep's own:
 *   sse_view_brf[(k*n_views + v)*n + i] = SSE(view(D(disp_i)), view(D(B(dec)))).
 * p stays required: it supplies focus, baseline and amp for D.  As for the gray sweep, the reference never runs this: the BRF
 * call on the decoded disparity is commented out at main.cpp:306-311, and putting B before D is this library's definition. */
int dmc_jpeg_view_rd_sweep_ex(dmc_ctx* ctx, const void* disp, const void* texture, int src_mem, int n_frames, int rows, int cols,
                              const int* qualities, int n_q, int flags, const dmc_chain_params* p, const dmc_brf_params* b, double f,
                              const double* R, const double* t, int n_views, const double* K, int is_sub, int render_flags,
                              uint64_t* bytes, uint64_t* sse_view_coded, uint64_t* sse_view_filtered, uint64_t* sse_view_brf);

/* ---- pointcloudTest's frame loop on batches: preparation and views ------------------------------------------------ */
/* Preparation of sensor depth (main.cpp:254-260, :511-512) on n_frames dense 16UC1 frames (depth16) into n_frames dense 8UC1
 * frames (disp8), both in `mem`:
 *   passes = 1: disp8_i = fillOcclusion(depth16U2disp8U(depth16_i, focal_baseline, a, b), 0, FILL_DISPARITY)  (simpleTest);
 *   passes = 2: that, then transpose, fillOcclusion(0, FILL_DISPARITY) and transpose back                       (pointcloudTest).
 * Every frame equals, bit for bit, that sequence of single-image calls on the frame alone: the converter's SIMD body and
 * scalar tail split per frame, and no frame reads its neighbour.  Device memory: groups of frames (~256 MB, DMC_GROUP_MB)
 * in stream order (dmc_synchronize before reading disp8).  Host memory: chunks stream through the device as in
 * dmc_chain_batch; returns when disp8 is valid.  DMC_ERR_ARG: passes not 1 or 2, depth16 and disp8 overlapping, a bad mem;
 * DMC_ERR_SIZE: cols < 2, rows < 2 with passes = 2, a negative count or size, a NULL buffer; nothing is written on error. */
int dmc_prepare_disp_batch(dmc_ctx* ctx, const void* depth16, void* disp8, int n_frames, int rows, int cols, float focal_baseline,
                           float a, float b, int passes, int mem);
/* Views of frame batches (main.cpp:321-355): for every frame i of depth (n_frames dense rows x cols frames of depth_type
 * DMC_8U, DMC_16S, DMC_16U or DMC_32F, the depths reprojectXYZ takes; dmc_chain_batch's DMC_CHAIN_DEPTH32F output as it is)
 * with its texture i (dense 8UC3) and every camera v (R + 9v, t + 3v: row-major doubles; K shared),
 *   views[v*n_frames + i] = fillSmallHole(projectImagefromXYZ(texture_i, reprojectXYZ(depth_i, f), R_v, t_v, K, is_sub)),
 * the fill in place as at main.cpp:355; each view is a dense rows x cols 8UC3 image.  This is the view of
 * dmc_jpeg_view_rd_sweep, through the same render.  depth, texture and views are all in `mem`.  render_flags:
 * DMC_RENDER_EXACT_DIVIDE or 0.  Frames run in groups sized like the sweep's.  Device memory: in stream order; host
 * memory: returns when views is valid.  DMC_ERR_ARG (nothing written): n_views < 1, a NULL camera, unknown render_flags,
 * views overlapping depth or texture, another depth_type, a bad mem; DMC_ERR_SIZE: rows * cols >= 2^29, a negative count
 * or size, a NULL buffer. */
int dmc_render_view_batch(dmc_ctx* ctx, const void* depth, int depth_type, const void* texture, int mem, int n_frames, int rows, int cols,
                          double f, const double* R, const double* t, int n_views, const double* K, int is_sub, int render_flags, void* views);

#ifdef __cplusplus
}
#endif
#endif
