/* hbcu.h -- C-ABI of the B200 (sm_100a) implementation of libhb's per-pixel
 * video-filter hot path.  Plain pointers and sizes only; no CUDA or torch types.
 *
 * This is the boundary a libhb maintainer binds: the filter objects in
 * handbrake_b200/libhb/ (nlmeans_cuda.c, ...) (drop-ins for hb_filter_nlmeans, ...) are
 * ordinary C that call ONLY the functions below.  Each group names the
 * reference code it replaces (paths relative to /root/reference/libhb).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure;
 *     hbcu_last_error() then describes the failure (thread-local string).
 *   - "planes"/"strides": arrays of 3 host pointers / byte strides in
 *     hb_buffer_t.plane[] order (Y, Cb, Cr).  Host memory may be pageable;
 *     page-locked memory from hbcu_host_alloc() makes the copies asynchronous.
 *   - a handle belongs to one thread at a time (libhb calls a filter's work() from that filter's own thread only,
 *     work.c:2527); different handles may be used from different threads concurrently.  All device work is queued
 *     on the handle's own non-blocking streams and ordered by events; calls return before the work has run unless
 *     they are named wait / sync / result.
 *   - nothing here falls back to the CPU: with no usable sm_100 device the
 *     create functions fail (=> filter init() returns non-zero, and libhb drops
 *     the filter exactly as for any failing init, work.c:1861-1868).
 */
#ifndef HBCU_H
#define HBCU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HBCU_ABI_VERSION 6

/* ------------------------------------------------------------------------- */
/* runtime                                                                    */
/* ------------------------------------------------------------------------- */
int          hbcu_abi_version(void);
const char * hbcu_last_error(void);
/* number of CUDA devices visible (0 when no driver / no GPU) */
int          hbcu_device_count(void);
/* page-locked host memory: the "pinned backing" of hb_buffer_t
 * (replaces av_malloc in hb_buffer_init_internal, fifo.c:358-441).  Freed blocks
 * are kept in power-of-two size pools like libhb's buffer pools (fifo.c:70-135)
 * because cudaHostAlloc costs milliseconds; hbcu_host_trim() releases them. */
void *       hbcu_host_alloc(size_t bytes);
void         hbcu_host_free(void *p);
void         hbcu_host_trim(void);
/* while on, hbcu_host_alloc hands out WRITE-COMBINED pinned memory: for buffers the CPU only writes and the GPU only reads
 * (a decoder's output frames); never for buffers the CPU reads back (filter outputs) */
void         hbcu_host_set_write_combined(int on);
/* pre-populates the pool with `count` blocks able to hold `bytes` each (steady state of a running
 * pipeline, where every frame buffer is a recycled one); returns the number of blocks added */
int          hbcu_host_reserve(size_t bytes, int count);
/* kernels launched by this library since load (bench.py's gpu_launches) */
uint64_t     hbcu_kernel_launches(void);

/* ------------------------------------------------------------------------- */
/* device frames: the HBCU_DEVICE backing of hb_buffer_t (SURVEY.md 8 f3)      */
/*   what AVFRAME / COREMEDIA storage is to the other hardware paths           */
/*   (handbrake/internal.h:152-153, fifo.c:1016-1034): between two CUDA        */
/*   filters a frame stays in HBM.  A frame is one allocation, planes back to   */
/*   back at the given strides (use hb_image_stride: the layout of a STANDARD  */
/*   hb_buffer_t).  Frames are pooled; release never blocks -- two CUDA events */
/*   per frame (producer done / readers done) order the streams that touch it. */
/* ------------------------------------------------------------------------- */
typedef struct hbcu_frame_s hbcu_frame_t;
int    hbcu_frame_alloc(hbcu_frame_t **f, int device, const int row_bytes[3], const int rows[3], const int strides[3]);
void   hbcu_frame_retain(hbcu_frame_t *f);             /* hb_buffer_shallow_dup(): one more reference (frames are written once) */
void   hbcu_frame_release(hbcu_frame_t *f);            /* hb_buffer_close() of an HBCU_DEVICE buffer (fifo.c:1037-1083); pooled at the last one */
void * hbcu_frame_plane(const hbcu_frame_t *f, int plane);      /* DEVICE pointer: never dereference on the host */
int    hbcu_frame_stride(const hbcu_frame_t *f, int plane);
int    hbcu_frame_device(const hbcu_frame_t *f);
long   hbcu_frames_alive(void);                         /* handed out and not released (leak check) */
/* The NVDEC / NVENC seam (libhb/nvenc_common.c:329-336 sets hw_pix_fmt = AV_PIX_FMT_CUDA; libhb/hwaccel.c:15-60):
 * a frame that already lives in device memory SOMEBODY ELSE owns -- what an AVFrame of AV_PIX_FMT_CUDA carries,
 * data[i] = device pointer, linesize[i] = pitch -- becomes an hbcu_frame_t without a copy.
 *   dplanes / strides    AVFrame.data / AVFrame.linesize (16-byte aligned, as every decoder surface is)
 *   readable_tail_bytes  how far past each plane's last row the allocation stays readable (>= 256: the stencil kernels
 *                        read whole vectors; decoder surfaces are height-aligned and satisfy it)
 *   producer_stream      the CUstream the planes were written on (AVCUDADeviceContext.stream), or NULL when the
 *                        writer has already been synchronised: consumers order themselves behind it, nobody blocks
 *   release(opaque)      called once, after the last hb_buffer_t reference is gone AND every queued device reader has
 *                        finished (av_frame_free / unmapping the surface goes here)
 * hbcu_frame_acquire/done let an external consumer (the encoder's stream) read ANY device frame in stream order. */
typedef void (*hbcu_frame_release_fn)(void *opaque);
int    hbcu_frame_wrap(hbcu_frame_t **f, int device, void *const dplanes[3], const int row_bytes[3], const int rows[3],
                       const int strides[3], size_t readable_tail_bytes, void *producer_stream,
                       hbcu_frame_release_fn release, void *opaque);
int    hbcu_frame_acquire(hbcu_frame_t *f, void *cuda_stream);
int    hbcu_frame_done(hbcu_frame_t *f, void *cuda_stream);

void   hbcu_frame_trim(void);                           /* frees the pooled frames */
/* the two ends of a device-resident chain (the role of libhb's adapter filters,
 * platform/macosx/adapter_vt.c): host frame -> device frame in front of the first CUDA filter,
 * device frame -> host frame in front of the encoder.  Asynchronous; `ticket`s complete in order,
 * `depth` of them may be in flight. */
typedef struct hbcu_xfer_s hbcu_xfer_t;
int    hbcu_xfer_create(hbcu_xfer_t **x, int device, int depth);
void   hbcu_xfer_destroy(hbcu_xfer_t *x);
int    hbcu_xfer_upload(hbcu_xfer_t *x, int64_t ticket, hbcu_frame_t *f, const void *const planes[3], const int strides[3]);
int    hbcu_xfer_download(hbcu_xfer_t *x, int64_t ticket, hbcu_frame_t *f, void *const planes[3], const int strides[3]);
int    hbcu_xfer_wait(hbcu_xfer_t *x, int64_t ticket);
int    hbcu_xfer_poll(hbcu_xfer_t *x, int64_t ticket);  /* 1 done, 0 running, <0 error */

/* ------------------------------------------------------------------------- */
/* NLMeans      replaces nlmeans.c:464-664 + templates/nlmeans_template.c       */
/*              (nlmeans_alloc/border, build_integral_*, nlmeans_plane) and    */
/*              nlmeans_x86.c; taskset fork/join becomes stream ordering       */
/* ------------------------------------------------------------------------- */
#define HBCU_NLMEANS_EXPSIZE 128   /* NLMEANS_EXPSIZE, nlmeans.c:88 */

typedef struct hbcu_nlmeans_plane_s
{
    int    patch_size;      /* n, odd >= 1            (pv->patch_size[c]) */
    int    range;           /* r, odd >= 1            (pv->range[c])      */
    int    nframes;         /* temporal depth 1..32   (pv->nframes[c])    */
    int    bypass;          /* strength == 0: plane is copied (nlmeans.c:493-499) */
    double origin_tune;     /* pv->origin_tune[c] */
    float  weight_fact;     /* pv->weight_fact_table[c]  (nlmeans.c:352) */
    int    diff_max;        /* pv->diff_max[c]           (nlmeans.c:353) */
    float  exptable[HBCU_NLMEANS_EXPSIZE];   /* pv->exptable[c], computed by the host exactly as nlmeans.c:354-358 */
    int    prefilter;       /* pv->prefilter[c] (nlmeans.c:72-83): mean 1/2, median 4/8, csm 16/32, reduce 256/512, edgeboost 1024,
                             * passthru 2048; patch distances are taken from the pre-denoised image (template :103-543) */
} hbcu_nlmeans_plane_t;

typedef struct hbcu_nlmeans_config_s
{
    int width, height;          /* luma geometry */
    int depth;                  /* bits per sample: 8 -> uint8 planes, 9..16 -> uint16 planes */
    int chroma_shift_w;         /* log2 chroma subsampling (1,1 for yuv420p) */
    int chroma_shift_h;
    int device;                 /* CUDA device ordinal */
    int ring_frames;            /* input frames kept on the device (>= max nframes + in-flight outputs) */
    int out_slots;              /* device output frames in flight */
    hbcu_nlmeans_plane_t plane[3];
} hbcu_nlmeans_config_t;

typedef struct hbcu_nlmeans_s hbcu_nlmeans_t;

int  hbcu_nlmeans_create(hbcu_nlmeans_t **out, const hbcu_nlmeans_config_t *cfg);
void hbcu_nlmeans_destroy(hbcu_nlmeans_t *h);

/* nlmeans_add_frame (nlmeans.c:524-544): copy frame `index` to the device and
 * build its mirror-bordered planes.  Asynchronous when the source is pinned;
 * the source may be reused once hbcu_nlmeans_wait_upload(index) returned. */
int  hbcu_nlmeans_upload(hbcu_nlmeans_t *h, int64_t index,
                         const void *const planes[3], const int strides[3]);
int  hbcu_nlmeans_wait_upload(hbcu_nlmeans_t *h, int64_t index);

/* nlmeans_filter_work / nlmeans_plane (nlmeans.c:464-522): denoise frame
 * `index` from frames index .. index+navail-1 (navail is clamped per plane to
 * its nframes; the EOF flush passes the shrinking count, nlmeans.c:636-640)
 * and copy the result to the host planes.  Asynchronous; hbcu_nlmeans_wait()
 * blocks until the host planes hold the result. */
int  hbcu_nlmeans_filter(hbcu_nlmeans_t *h, int64_t index, int navail,
                         void *const planes[3], const int strides[3]);
int  hbcu_nlmeans_wait(hbcu_nlmeans_t *h, int64_t index);
/* non-blocking: 1 = the host planes of frame `index` are complete, 0 = still in flight, <0 = error */
int  hbcu_nlmeans_poll(hbcu_nlmeans_t *h, int64_t index);

/* device-resident entry points (frames never leave HBM): used by chained
 * filters and by bench.py's kernel-only arm.
 *   upload_device : src = device pointers to unbordered planes
 *   filter_device : result stays in the handle's output slot; pointers to it
 *                   are returned through out_planes/out_strides (may be NULL) */
int  hbcu_nlmeans_upload_device(hbcu_nlmeans_t *h, int64_t index,
                                const void *const dplanes[3], const int strides[3]);
int  hbcu_nlmeans_filter_device(hbcu_nlmeans_t *h, int64_t index, int navail,
                                void *out_planes[3], int out_strides[3]);
/* like filter_device, but the result is written straight into caller-owned DEVICE planes (the next
 * filter's input, or a buffer an NCCL send reads): the device-resident hand-off between filters */
int  hbcu_nlmeans_filter_into(hbcu_nlmeans_t *h, int64_t index, int navail,
                              void *const dplanes[3], const int strides[3]);
/* Multi-device dealing (the frame-parallel taskset of mt_frame_filter.c:169-237 spread over several GPUs): one handle
 * per device, each with its OWN contiguous index space; the filter deals blocks of frames to the handles in turn.
 *   upload_peer      : frame `src_index` of `src` (uploaded there already) becomes frame `dst_index` of `dst`, copied
 *                      device to device (NVLink peer copy): the temporal halo of a block crosses PCIe once, not twice.
 *                      Both handles must outlive the copy (destroy them together).
 *   set_stream_slice : mid_stream != 0 -- the handle's frame 0 is NOT the first frame of the stream, so the
 *                      start-of-stream rule of the prefilter path (templates/nlmeans_template.c:612 vs :628: the very
 *                      first frame's source patches come from the unfiltered image) does not apply to it. */
int  hbcu_nlmeans_upload_peer(hbcu_nlmeans_t *dst, int64_t dst_index, hbcu_nlmeans_t *src, int64_t src_index);
int  hbcu_nlmeans_set_stream_slice(hbcu_nlmeans_t *h, int mid_stream);

/* device-resident chain: frame `index` arrives in / leaves in an hbcu_frame_t.  Stream-ordered against the frame's
 * producer and readers, never blocks; the output needs no wait/poll -- its consumer orders itself behind it. */
int  hbcu_nlmeans_upload_frame(hbcu_nlmeans_t *h, int64_t index, hbcu_frame_t *in);
int  hbcu_nlmeans_filter_frame(hbcu_nlmeans_t *h, int64_t index, int navail, hbcu_frame_t *out);
/* orders a caller-owned CUDA stream (passed as void*) after all work queued on the handle so far */
int  hbcu_nlmeans_stream_wait(hbcu_nlmeans_t *h, void *cuda_stream);
int  hbcu_nlmeans_sync(hbcu_nlmeans_t *h);
/* implementation selector for tests: 0 = auto (per plane: the v3 tile kernels
 * where their conditions hold, else the integer tiled kernel where the patch
 * and range fit its halo, else the generic kernel), 1 = force generic,
 * 2 = as 0 but fail where 0 would take the generic kernel, 3 = integer tiled
 * kernel where it fits, generic otherwise (the one >10-bit planes use) */
int  hbcu_nlmeans_set_impl(hbcu_nlmeans_t *h, int impl);

/* CUDA-event timing on the handle's compute stream (bench.py):
 * mark 0 = start, mark 1 = stop; elapsed_ms synchronises on mark 1. */
int  hbcu_nlmeans_mark(hbcu_nlmeans_t *h, int which);
int  hbcu_nlmeans_elapsed_ms(hbcu_nlmeans_t *h, float *ms);
/* device time spent in the main kernel alone between the two marks */
int  hbcu_nlmeans_kernel_ms(hbcu_nlmeans_t *h, float *ms, int *launches);

/* ------------------------------------------------------------------------- */
/* Comb detect   replaces comb_detect.c:221-276,384-454,556-966,1051-1072 and  */
/*               templates/comb_detect_template.c:288-402,789-933 (the five     */
/*               tasksets become three kernels on one stream)                  */
/* ------------------------------------------------------------------------- */
typedef struct hbcu_comb_detect_config_s
{
    int width, height;        /* luma geometry (only luma is examined) */
    int depth;
    int device;
    int slots;                /* luma planes kept on the device (>= 4) */
    int mode;                 /* bit0 MODE_GAMMA, bit1 MODE_FILTER (comb_detect.c:23-26) */
    int spatial_metric;
    int filter_mode;          /* 1 FILTER_CLASSIC, 2 FILTER_ERODE_DILATE */
    int motion_threshold;     /* already shifted by depth-8 (comb_detect.c:1152-1153) */
    int spatial_threshold;
    int block_threshold, block_width, block_height;
    float gamma_motion_threshold, gamma_spatial_threshold, gamma_spatial_threshold6;
    int comb32detect_min, comb32detect_max;
    const float *gamma_lut;   /* (1<<depth) floats built by the host as comb_detect.c:1074-1081 */
} hbcu_comb_detect_config_t;

typedef struct hbcu_comb_detect_s hbcu_comb_detect_t;

int  hbcu_comb_detect_create(hbcu_comb_detect_t **out, const hbcu_comb_detect_config_t *cfg);
void hbcu_comb_detect_destroy(hbcu_comb_detect_t *h);
/* luma plane of frame `index` to the device (asynchronous from pinned memory) */
int  hbcu_comb_detect_upload(hbcu_comb_detect_t *h, int64_t index, const void *luma, int stride);
int  hbcu_comb_detect_upload_device(hbcu_comb_detect_t *h, int64_t index, const void *dluma, int stride);
int  hbcu_comb_detect_upload_frame(hbcu_comb_detect_t *h, int64_t index, hbcu_frame_t *in);   /* luma of a device frame */
/* comb_segmenter (comb_detect.c:1051-1072) for frame `cur` against `prev` and `next`; asynchronous */
int  hbcu_comb_detect_run(hbcu_comb_detect_t *h, int64_t prev, int64_t cur, int64_t next, int force_exhaustive);
/* blocks until the verdict of frame `cur` is known: HB_COMB_NONE 0 / LIGHT 1 / HEAVY 2 */
int  hbcu_comb_detect_result(hbcu_comb_detect_t *h, int64_t cur, int *combed);
/* test hook: raw and scored masks (width*height bytes each, may be NULL) of the latest run */
int  hbcu_comb_detect_masks(hbcu_comb_detect_t *h, uint8_t *raw, uint8_t *scored);
int  hbcu_comb_detect_sync(hbcu_comb_detect_t *h);
int  hbcu_comb_detect_mark(hbcu_comb_detect_t *h, int which);
int  hbcu_comb_detect_elapsed_ms(hbcu_comb_detect_t *h, float *ms);

/* ------------------------------------------------------------------------- */
/* Decomb        replaces decomb.c:500-571 (per-field work) and                 */
/*               templates/decomb_template.c:43-107,279-361,482-898 (cubic,     */
/*               blend, yadif line filters, segment driver, frame filter);      */
/*               EEDI2 (eedi2.c, templates/eedi2_template.c) plugs in below     */
/* ------------------------------------------------------------------------- */
#define HBCU_DECOMB_YADIF     1
#define HBCU_DECOMB_BLEND     2
#define HBCU_DECOMB_CUBIC     4
#define HBCU_DECOMB_EEDI2     8
#define HBCU_DECOMB_BOB       16
#define HBCU_DECOMB_SELECTIVE 32

typedef struct hbcu_decomb_config_s
{
    int width, height;
    int depth;
    int chroma_shift_w, chroma_shift_h;
    int device;
    int slots;                  /* input frames kept on the device (>= 4) */
    int out_slots;              /* output fields in flight */
    int mode;                   /* filter-level mode bits (selects whether EEDI2 buffers are needed) */
    /* EEDI2 thresholds, decomb.c:234-243 */
    int magnitude_threshold, variance_threshold, laplacian_threshold;
    int dilation_threshold, erosion_threshold, noise_threshold;
    int maximum_search_distance, post_processing;
} hbcu_decomb_config_t;

typedef struct hbcu_decomb_s hbcu_decomb_t;

int  hbcu_decomb_create(hbcu_decomb_t **out, const hbcu_decomb_config_t *cfg);
void hbcu_decomb_destroy(hbcu_decomb_t *h);
int  hbcu_decomb_upload(hbcu_decomb_t *h, int64_t index, const void *const planes[3], const int strides[3]);
int  hbcu_decomb_upload_device(hbcu_decomb_t *h, int64_t index, const void *const dplanes[3], const int strides[3]);
/* blocks until the host planes of frame `index` have been read (no-op if the frame left the device ring) */
int  hbcu_decomb_wait_upload(hbcu_decomb_t *h, int64_t index);
/* one output picture (filter_{8,16}, decomb template :810-898): `frame_mode` is the mode chosen for
 * this frame (BLEND for lightly combed frames, else the filter mode without SELECTIVE), `parity`
 * the field being rebuilt, `tff` the field order.  Result goes to the host planes asynchronously;
 * `ticket` is a caller-chosen id (monotonic) for wait/poll. */
int  hbcu_decomb_filter(hbcu_decomb_t *h, int64_t ticket, int64_t prev, int64_t cur, int64_t next,
                        int frame_mode, int parity, int tff, void *const planes[3], const int strides[3]);
int  hbcu_decomb_filter_device(hbcu_decomb_t *h, int64_t ticket, int64_t prev, int64_t cur, int64_t next,
                               int frame_mode, int parity, int tff, void *out_planes[3], int out_strides[3]);
/* device-resident chain (see hbcu_frame_t): input frame from / output picture into a device frame, stream-ordered */
int  hbcu_decomb_upload_frame(hbcu_decomb_t *h, int64_t index, hbcu_frame_t *in);
int  hbcu_decomb_filter_frame(hbcu_decomb_t *h, int64_t ticket, int64_t prev, int64_t cur, int64_t next,
                              int frame_mode, int parity, int tff, hbcu_frame_t *out);
int  hbcu_decomb_wait(hbcu_decomb_t *h, int64_t ticket);
int  hbcu_decomb_poll(hbcu_decomb_t *h, int64_t ticket);
int  hbcu_decomb_sync(hbcu_decomb_t *h);
/* test hook: EEDI2 work buffer `which` (0-3 field buffers SRCPF MSKPF TMPPF DSTPF, 4-8 frame buffers
 * DST2PF TMP2PF2 MSK2PF TMP2PF DST2MPF; decomb.c:64-74), three planes back to back with their strides */
int  hbcu_decomb_debug_eedi2(hbcu_decomb_t *h, int which, void *host, size_t host_bytes);
int  hbcu_decomb_mark(hbcu_decomb_t *h, int which);
int  hbcu_decomb_elapsed_ms(hbcu_decomb_t *h, float *ms);

/* ------------------------------------------------------------------------- */
/* Lapsharp      replaces lapsharp.c:125-182 (DEF_LAPSHARP_FUNC) and, for the   */
/*               frame batching, mt_frame_filter.c:169-237 (stream dispatch)    */
/* ------------------------------------------------------------------------- */
typedef struct hbcu_lapsharp_config_s
{
    int width, height, depth;
    int chroma_shift_w, chroma_shift_h;
    int device;
    int slots;                   /* frames in flight */
    double strength[3];          /* sanitised, lapsharp.c:289-296 */
    int    kernel[3];            /* 0 lap, 1 isolap, 2 log, 3 isolog (lapsharp.c:36-93) */
} hbcu_lapsharp_config_t;

typedef struct hbcu_lapsharp_s hbcu_lapsharp_t;

int  hbcu_lapsharp_create(hbcu_lapsharp_t **out, const hbcu_lapsharp_config_t *cfg);
void hbcu_lapsharp_destroy(hbcu_lapsharp_t *h);
/* one frame: host planes in (whole strides are transferred: the filter reads the stride region next
 * to the right picture edge, lapsharp.c:145-158), host planes out; asynchronous, `ticket` for wait/poll */
int  hbcu_lapsharp_filter(hbcu_lapsharp_t *h, int64_t ticket, const void *const in_planes[3], const int in_strides[3],
                          void *const out_planes[3], const int out_strides[3]);
/* device-resident variant: dplanes are device pointers with the given strides, result stays on the device */
int  hbcu_lapsharp_filter_device(hbcu_lapsharp_t *h, int64_t ticket, const void *const dplanes[3], const int strides[3],
                                 void *out_planes[3], int out_strides[3]);
/* device-resident chain: either side may be a device frame (NULL = use the host planes / strides of that side) */
int  hbcu_lapsharp_filter_frames(hbcu_lapsharp_t *h, int64_t ticket,
                                 hbcu_frame_t *in_frame, const void *const in_planes[3], const int in_strides[3],
                                 hbcu_frame_t *out_frame, void *const out_planes[3], const int out_strides[3]);
int  hbcu_lapsharp_wait(hbcu_lapsharp_t *h, int64_t ticket);
int  hbcu_lapsharp_poll(hbcu_lapsharp_t *h, int64_t ticket);
int  hbcu_lapsharp_sync(hbcu_lapsharp_t *h);
int  hbcu_lapsharp_mark(hbcu_lapsharp_t *h, int which);
int  hbcu_lapsharp_elapsed_ms(hbcu_lapsharp_t *h, float *ms);

/* ------------------------------------------------------------------------- */
/* unsharp / chroma smooth   replaces DEF_UNSHARP_FUNC (unsharp.c:88-168) and    */
/*              DEF_CHROMA_SMOOTH_FUNC (chroma_smooth.c:86-168), with lapsharp  */
/*              the three clients of mt_frame_filter.c (common.c:5497-5517)     */
/* ------------------------------------------------------------------------- */
typedef struct hbcu_unsharp_config_s
{
    int width, height, depth;
    int chroma_shift_w, chroma_shift_h;
    int device;
    int slots;              /* frames in flight */
    int smooth;             /* 0 = unsharp.c, 1 = chroma_smooth.c */
    int amount[3];          /* (int)(strength * 65536.0) per plane after the filter's sanitising; 0 copies the plane
                             * (chroma_smooth: always 0 for luma) */
    int steps[3];           /* size / 2 per plane, 1..7 */
} hbcu_unsharp_config_t;

typedef struct hbcu_unsharp_s hbcu_unsharp_t;

int  hbcu_unsharp_create(hbcu_unsharp_t **out, const hbcu_unsharp_config_t *cfg);
void hbcu_unsharp_destroy(hbcu_unsharp_t *h);
/* one frame; either side may be a device frame (NULL = the host planes / strides of that side); asynchronous */
int  hbcu_unsharp_filter_frames(hbcu_unsharp_t *h, int64_t ticket,
                                hbcu_frame_t *in_frame, const void *const in_planes[3], const int in_strides[3],
                                hbcu_frame_t *out_frame, void *const out_planes[3], const int out_strides[3]);
int  hbcu_unsharp_wait(hbcu_unsharp_t *h, int64_t ticket);
int  hbcu_unsharp_poll(hbcu_unsharp_t *h, int64_t ticket);
int  hbcu_unsharp_sync(hbcu_unsharp_t *h);
int  hbcu_unsharp_mark(hbcu_unsharp_t *h, int which);
int  hbcu_unsharp_elapsed_ms(hbcu_unsharp_t *h, float *ms);

/* ------------------------------------------------------------------------- */
/* hqdn3d       replaces hqdn3d_denoise_spatial/_temporal/_depth                 */
/*              (denoise.c:102-201); SURVEY.md 8 f4                              */
/* ------------------------------------------------------------------------- */
typedef struct hbcu_hqdn3d_config_s
{
    int width, height, depth;
    int chroma_shift_w, chroma_shift_h;
    int device;
    int slots;                 /* frames in flight */
    const int16_t *coef[6];    /* hqdn3d_precalc_coef tables (denoise.c:78-94), 512 << LUT_BITS entries each, computed by the host
                                * exactly as there: y-spatial, y-temporal, cb-spatial, cb-temporal, cr-spatial, cr-temporal */
} hbcu_hqdn3d_config_t;

typedef struct hbcu_hqdn3d_s hbcu_hqdn3d_t;

int  hbcu_hqdn3d_create(hbcu_hqdn3d_t **out, const hbcu_hqdn3d_config_t *cfg);
void hbcu_hqdn3d_destroy(hbcu_hqdn3d_t *h);
/* one frame, IN DISPLAY ORDER (the temporal state chains the frames); either side may be a device frame */
int  hbcu_hqdn3d_filter_frames(hbcu_hqdn3d_t *h, int64_t ticket,
                               hbcu_frame_t *in_frame, const void *const in_planes[3], const int in_strides[3],
                               hbcu_frame_t *out_frame, void *const out_planes[3], const int out_strides[3]);
int  hbcu_hqdn3d_wait(hbcu_hqdn3d_t *h, int64_t ticket);
int  hbcu_hqdn3d_poll(hbcu_hqdn3d_t *h, int64_t ticket);
int  hbcu_hqdn3d_sync(hbcu_hqdn3d_t *h);
int  hbcu_hqdn3d_mark(hbcu_hqdn3d_t *h, int which);
int  hbcu_hqdn3d_elapsed_ms(hbcu_hqdn3d_t *h, float *ms);

/* ------------------------------------------------------------------------- */
/* detelecine   replaces the data-parallel half of pullup (libhb/detelecine.c): */
/*              pullup_compute_metric + pullup_diff_y/licomb_y/var_y (:159-265), */
/*              the max-reductions inside pullup_compute_breaks (:345-380) and   */
/*              pullup_compute_affinity (:382-434), pullup_copy_field (:298-317) */
/* ------------------------------------------------------------------------- */
/* The field-queue state machine (what to compare with what, how long a frame is, which fields make it) is control
 * flow on a handful of integers; it stays on the host (handbrake_b200/libhb/detelecine_cuda.c) and drives these calls.
 * Pictures and the per-field metric arrays never leave the device.  Everything is queued on the handle's stream; only
 * hbcu_detelecine_fetch(), hbcu_detelecine_download() and hbcu_detelecine_download_end() wait. */
typedef struct hbcu_detelecine_config_s
{
    int width, height, depth;
    int chroma_shift_w, chroma_shift_h;
    int device;
    int pictures;              /* picture buffers (pullup's nbuffers, >= 10, detelecine.c:601-607) */
    int fields;                /* metric slots, one per node of the field queue (9 to start with, :623) */
    int results;               /* reduction result slots */
    int metric_plane;
    int junk_left, junk_right; /* in units of 8 pixels  (:615-618) */
    int junk_top, junk_bottom; /* in units of 2 lines */
} hbcu_detelecine_config_t;

typedef struct hbcu_detelecine_s hbcu_detelecine_t;

int  hbcu_detelecine_create(hbcu_detelecine_t **out, const hbcu_detelecine_config_t *cfg);
void hbcu_detelecine_destroy(hbcu_detelecine_t *h);
/* picture <- host planes with their strides (hb_image_copy_plane semantics: whole strides when they agree) */
int  hbcu_detelecine_upload(hbcu_detelecine_t *h, int picture, const void *const planes[3], const int strides[3]);
/* the three metric arrays of field slot `field` = field `parity` of `picture` (pullup_submit_field :973-978):
 *   diffs against the same-parity field of diff_picture: -1 leaves the array as it is (the partner has no buffer, :242),
 *         == picture zeroes it (the duplicate-field shortcut, :244-249);
 *   comb  between the top field of comb_top_picture and the bottom field of comb_bottom_picture; -1 leaves it as it is;
 *   var   of the field itself. */
int  hbcu_detelecine_metrics(hbcu_detelecine_t *h, int field, int picture, int parity,
                             int diff_picture, int comb_top_picture, int comb_bottom_picture);
/* result[slot] = { max(0, max_i l_i), max(0, max_i -l_i) } with
 *   breaks:   l_i = diffs2[i] - diffs3[i]                                                    (:369-374)
 *   affinity: l_i = max(0, comb[i] - (v+lv) + |v-lv|) - max(0, comb_next[i] - (v+rv) + |v-rv|),
 *             v = var[i], lv = var_prev[i], rv = var_next[i]                                  (:405-418) */
int  hbcu_detelecine_breaks(hbcu_detelecine_t *h, int field2, int field3, int slot);
int  hbcu_detelecine_affinity(hbcu_detelecine_t *h, int field_prev, int field, int field_next, int slot);
/* waits for everything queued so far; dst <- result slots [0, nslots) (2 ints each) */
int  hbcu_detelecine_fetch(hbcu_detelecine_t *h, int *dst, int nslots);
/* lines of `parity` (whole strides) of src_picture -> dst_picture */
int  hbcu_detelecine_copy_field(hbcu_detelecine_t *h, int dst_picture, int src_picture, int parity);
/* picture -> host planes (plane height x stride bytes each, as the reference's memcpy of size[p], :1250-1252); waits */
int  hbcu_detelecine_download(hbcu_detelecine_t *h, int picture, void *const planes[3], const int strides[3]);
/* the same without the wait: the copy runs on the handle's download stream behind everything queued so far, so it overlaps
 * the next picture's upload and metrics; _end waits for the most recent _begin.  The caller keeps the picture untouched
 * (and its host planes alive) until then.  (detelecine.c:1246-1258 is the copy-out this serves.) */
int  hbcu_detelecine_download_begin(hbcu_detelecine_t *h, int picture, void *const planes[3], const int strides[3]);
int  hbcu_detelecine_download_end(hbcu_detelecine_t *h);
/* device-resident chain (SURVEY.md 8 f3): the picture arrives in / leaves in an hbcu_frame_t -- a device-to-device copy on
 * the handle's stream, ordered against the frame's producer and readers through its events; nothing waits on the host
 * (the frame twins of upload / download; detelecine.c:1116-1277 is the work() these serve) */
int  hbcu_detelecine_upload_frame(hbcu_detelecine_t *h, int picture, hbcu_frame_t *in);
int  hbcu_detelecine_download_frame(hbcu_detelecine_t *h, int picture, hbcu_frame_t *out);
/* benchmark hooks as for the other handles */
int  hbcu_detelecine_mark(hbcu_detelecine_t *h, int which);
int  hbcu_detelecine_elapsed_ms(hbcu_detelecine_t *h, float *ms);

#ifdef __cplusplus
}
#endif

#endif /* HBCU_H */
