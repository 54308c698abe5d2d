/*
 * b2video.h — C-ABI of libb2video.so, the B200-native video-frame hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point replaces one
 * call the selkies reference makes into its out-of-tree native module
 * `pixelflux` (capture → colour-convert → H.264 encode → callback).  The
 * reference interface each entry replaces is cited as  path:line  relative to
 * the selkies tree.  The signatures carry plain pointers and sizes only; the
 * Python host side (selkies_b200/_native.py) binds them with ctypes.
 *
 * Threading: every function is safe to call from any host thread; setters may
 * race with b2v_ring_submit() (reference: control calls arrive on thread-pool
 * threads, media_pipeline.py:195,236,244,300,313).  b2v_set_resolution() locks
 * submitters out, drains, and returns B2V_ESTATE while a producer still holds an
 * acquired ring slot (its memory is about to be reallocated).  The frame callback fires on
 * the session's own output thread (a native, non-Python thread, as pixelflux's
 * does: media_pipeline.py:293 uses run_coroutine_threadsafe for that reason).
 *
 * Errors: functions returning int give 0 on success and a negative B2V_E* code
 * on failure; b2v_last_error() returns a thread-local message.
 */
#ifndef B2VIDEO_H_
#define B2VIDEO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2V_ABI_VERSION 3

enum {
  B2V_OK = 0,
  B2V_EINVAL = -1,   /* bad argument / unsupported size            */
  B2V_ECUDA = -2,    /* CUDA runtime error (see b2v_last_error)     */
  B2V_ENOMEM = -3,
  B2V_ESTATE = -4,   /* call not valid in the current state         */
  B2V_ETIMEOUT = -5
};

/* rate-control modes: reference CaptureSettings.h264_cbr_mode / h264_crf
 * (media_pipeline.py:266-269) */
enum { B2V_RC_CBR = 0, B2V_RC_CQP = 1 };

/* header_mode: what precedes the Annex-B access unit in b2v_frame.data.
 * 1 = the 10-byte pixelflux stripe header the reference strips at
 * media_pipeline.py:286 and keeps at selkies.py:3116
 * (0x04, frame_type, frame_id u16be, y_start u16be, width u16be, height u16be;
 * parser: addons/selkies-web-core/selkies-ws-core.js:3183-3196). */
enum { B2V_HDR_NONE = 0, B2V_HDR_PIXELFLUX = 1 };

/* Session configuration — the native image of pixelflux.CaptureSettings as
 * filled by MediaPipelinePixel.generate_capture_settings
 * (media_pipeline.py:251-273) and _get_capture_settings (selkies.py:3191-3242). */
typedef struct b2v_settings {
  int32_t src_w, src_h;     /* BGRA source size (even, 16..7680 x 16..4320; selkies.py:281) */
  int32_t dst_w, dst_h;     /* encoded size; 0 = same as source (no scaling)                */
  double  fps;              /* CaptureSettings.target_fps                                   */
  int32_t device;           /* CUDA ordinal (settings.py:162 gpu_id)                        */
  int32_t rc_mode;          /* B2V_RC_CBR | B2V_RC_CQP                                      */
  int32_t bitrate_kbps;     /* CaptureSettings.h264_bitrate_kbps                            */
  int32_t crf;              /* CaptureSettings.h264_crf → constant QP 0..51 in CQP mode; <0 = 26 */
  int32_t gop;              /* in FRAMES.  <=0: IDR only on request (settings.py:163 keyframe_distance=-1);
                               1: intra-only; N: IDR every N frames.  keyframe_distance itself is in SECONDS:
                               the host side passes round(seconds * fps) (pixelflux_compat.py)             */
  int32_t slice_rows;       /* macroblock rows per slice of a P picture (>=1); 0 = default: 8, or one slice per stripe in striped
                               mode (inside a slice P_Skip infers moving vectors: a scrolling picture costs half the bytes) */
  int32_t header_mode;      /* B2V_HDR_*                                                    */
  int32_t ring_slots;       /* pinned BGRA ingest ring depth (2..16); 0 = default 4          */
  int32_t flags;            /* B2V_FLAG_*                                                   */
  int32_t paintover_trigger_frames; /* after this many consecutive all-skipped pictures code paintover_burst_frames pictures
                                       at paintover_crf (CaptureSettings.paint_over_trigger_frames / use_paint_over_quality,
                                       selkies.py:3226-3229); in CBR mode the paint-over QP only applies when it is finer
                                       than the controller's; 0 = off */
  int32_t paintover_crf;            /* CaptureSettings.h264_paintover_crf */
  int32_t stripe_rows;      /* striped mode (CaptureSettings.h264_fullframe = False, selkies.py:3219; encoder
                               "x264enc-striped"): macroblock rows per stripe, a multiple of slice_rows.  Every stripe is
                               an independent H.264 stream (own SPS/PPS, own frame_num, motion confined to the stripe)
                               delivered by its own callback with y_start/height (10-byte header bytes 4..9,
                               selkies-ws-core.js:3183-3196); a stripe whose macroblocks were all skipped is not
                               delivered.  0 or >= picture rows = full frame */
  int32_t idr_slice_mbs;    /* IDR pictures only (whatever slice_rows is): macroblocks per slice INSIDE a row.  The macroblocks of an
                               intra slice are a serial chain (left-neighbour prediction), so shorter slices shorten the chain the
                               GPU has to walk (a 4K key frame: 3.3 ms with whole rows).  0 = default (about 540 slices per
                               picture, none under 30 macroblocks: 60 at 4K, 30 at 1080p), < 0 = whole rows, n = n macroblocks */
  int32_t paintover_burst_frames;   /* CaptureSettings.h264_paintover_burst_frames (selkies.py:3217): how many consecutive
                                       pictures are coded at paintover_crf once the trigger is reached; <= 0 = 1 */
} b2v_settings;

enum {
  B2V_FLAG_SPS_EVERY_IDR = 1,   /* in-band SPS/PPS before every IDR (rtc.py:394-401); always on */
  B2V_FLAG_NO_ENCODE     = 2,   /* CSC only (BASELINE config 4: 8K CSC roofline stress)         */
  B2V_FLAG_TIMING        = 4,   /* bracket every kernel with CUDA events (b2v_get_stats)        */
  B2V_FLAG_DEVICE_TIMER  = 8,   /* with TIMING: the CSC kernel also stamps %globaltimer (ms_csc_device) */
  B2V_FLAG_TIMING_CSC    = 16,  /* a CUDA-event pair around the CSC launch of every 4th picture (ms_csc / n_csc)  */
  B2V_FLAG_JPEG          = 32   /* CaptureSettings.output_mode = 0 (selkies.py:3209-3212): JPEG stripes instead of H.264.  The picture is cut
                                   into stripes of stripe_rows x 16 rows (0 = about eight stripes); each stripe that changed is delivered by its
                                   own callback as one baseline JFIF file (JFIF colour, 4:2:0), y_start/height set; with B2V_HDR_PIXELFLUX the
                                   file is preceded by frame_id u16be | y_start u16be (the reference adds 03 00 in front, selkies.py:3118).
                                   crf = jpeg_quality, paintover_crf = paint_over_jpeg_quality, paintover_trigger_frames as for H.264.
                                   A key-frame request re-sends every stripe. */
};

/* One encoded frame, the native image of the pixelflux callback result
 * (`result.data / result.size / result.frame_id`, media_pipeline.py:284-292).
 * `data` is owned by the library and valid only during the callback. */
typedef struct b2v_frame {
  const uint8_t* data;   /* [optional 10-byte header] + Annex-B access unit */
  int32_t  size;         /* bytes in data                                    */
  int32_t  frame_id;     /* +1 per emitted frame, wraps at 65536 (selkies.py:10) */
  int32_t  is_key;       /* 1 = IDR                                         */
  int32_t  qp;           /* slice QP used for this frame                     */
  int64_t  pts90k;       /* frame_id * (90000 // fps)  (media_pipeline.py:291-292) */
  int64_t  capture_ns;   /* value passed to b2v_ring_submit                  */
  int32_t  y_start;      /* first picture row of this stripe (0 when full-frame)           */
  int32_t  height;       /* visible rows in this stripe (the picture height when full-frame) */
} b2v_frame;

typedef void (*b2v_cb)(const b2v_frame* frame, void* user);

/* Per-session counters; kernel times are CUDA-event milliseconds accumulated on
 * the launching stream (only when B2V_FLAG_TIMING is set). */
typedef struct b2v_stats {
  int64_t frames_submitted, frames_delivered, key_frames;
  int64_t bytes_out, h2d_bytes, d2h_bytes;
  int64_t kernel_launches;
  double  ms_csc, ms_intra, ms_inter, ms_cavlc, ms_slice, ms_pack, ms_total_gpu;
  int64_t n_csc, n_intra, n_inter, n_cavlc, n_slice, n_pack;
  double  ms_csc_device;   /* same launches, timed by the kernel itself (%globaltimer: first block start .. last block end) */
  int64_t n_csc_device;
  /* host-side stopwatches (CLOCK_MONOTONIC ns, always on): where a session's wall time goes when it is not the GPU's */
  int64_t ns_wait_event;     /* output thread: waiting for the GPU to finish the next picture (polling, no interrupt)      */
  int64_t ns_wait_event_max; /*   longest single such wait                                                               */
  int64_t n_event_sleeps;    /*   waits that outlasted the 30 us busy phase and slept                                    */
  int64_t ns_wait_job;       /* output thread: idle, no picture in flight                                                */
  int64_t ns_callback;       /* output thread: inside the frame callback (Python holds the GIL there)                    */
  int64_t ns_wait_out_slot;  /* submitter: blocked on back-pressure (every output slot in flight)                        */
  int64_t ns_wait_ring;      /* producer: blocked in b2v_ring_acquire (every ingest slot in flight)                      */
  int64_t ns_submit;         /* submitter: inside the CUDA enqueue calls of a picture (launches, copies, event records)  */
} b2v_stats;

/* ---- lifecycle: replaces ScreenCapture() / start_capture / stop_capture
 *      (media_pipeline.py:298-300, 313; selkies.py:3163-3176, 2852) ---------- */
int  b2v_abi_version(void);
int  b2v_device_count(void);
int  b2v_create(const b2v_settings* s, b2v_cb cb, void* user, void** out_handle);
void b2v_destroy(void* h);                 /* blocks: drains frames, joins the output thread */

/* ---- frame ingest (a: pinned host ring → cudaMemcpyAsync).  The producer is
 *      whatever fills BGRA frames (pixelflux's XShm grab in the reference,
 *      SURVEY.md §3.2 hot loop #1). ------------------------------------------ */
void* b2v_ring_acquire(void* h, int32_t* slot);          /* blocks until a slot is free */
int   b2v_ring_submit(void* h, int32_t slot, int32_t stride_bytes, int64_t capture_ns);
/* Give an acquired slot back WITHOUT encoding it (the producer had no frame after all: end of a canned source, a grab that
 * failed).  Only the most recently acquired slot can be returned; the next b2v_ring_acquire hands out the same slot. */
int   b2v_ring_release(void* h, int32_t slot);
/* device-resident frames (bench `value`: inputs already in HBM) */
int   b2v_resident_upload(void* h, int32_t index, const void* bgra_host, int32_t stride_bytes);
int   b2v_submit_resident(void* h, int32_t index, int64_t capture_ns);
int   b2v_flush(void* h);                                /* wait until every submitted frame was delivered */

/* ---- live control: ScreenCapture.update_framerate (media_pipeline.py:236),
 *      update_video_bitrate (:195), request_idr_frame (:244); set_resolution is
 *      WebRTCApp.on_resize_handler → width/height (webrtc_mode.py:383-426). --- */
int  b2v_set_framerate(void* h, double fps);
int  b2v_set_bitrate_kbps(void* h, int32_t kbps);
int  b2v_set_qp(void* h, int32_t qp);                    /* CQP mode (restart-free set_crf) */
int  b2v_set_gop(void* h, int32_t frames);               /* b2v_settings.gop, live (the Python side converts keyframe_distance
                                                            SECONDS, settings.py:163, with the current fps) */
int  b2v_set_resolution(void* h, int32_t src_w, int32_t src_h, int32_t dst_w, int32_t dst_h);
int  b2v_request_idr(void* h);

/* ---- introspection / test hooks ------------------------------------------- */
int  b2v_get_stats(void* h, b2v_stats* out);
int  b2v_reset_stats(void* h);
int  b2v_coded_size(void* h, int32_t* coded_w, int32_t* coded_h);
/* synchronous fused CSC(+scale) of one host BGRA frame to host NV12 (dst_w*dst_h*3/2 bytes) */
int  b2v_csc_nv12(void* h, const void* bgra_host, int32_t stride_bytes, void* nv12_host);
/* reconstruction of the last encoded frame: NV12, coded_w*coded_h*3/2 bytes */
int  b2v_get_recon(void* h, void* nv12_host);
/* repeat the CSC kernel `iters` times over resident frames and return mean ms per launch
 * (CUDA events on the launching stream); used by bench.py for the roofline leg. */
int  b2v_bench_csc(void* h, int32_t n_resident, int32_t iters, float* ms_per_launch);
/* same, but `iters` launches back to back between ONE event pair (amortises the event/launch gap) */
int  b2v_bench_csc_burst(void* h, int32_t n_resident, int32_t iters, float* ms_per_launch);
/* device-side stopwatch on the encode stream: start = after everything submitted so far has drained;
 * stop = after every frame submitted since has been delivered.  bench.py times its K steps with it. */
int  b2v_timer_start(void* h);
int  b2v_timer_stop(void* h, float* ms);
const char* b2v_last_error(void);

/* ---- RTP H.264 payloader (SURVEY.md §8f row 1): replaces H264Encoder.pack -> _split_bitstream / _packetize
 *      (src/selkies/webrtc/codecs/h264.py:238-279, 331-335).  Splits the Annex-B access unit and writes the RTP
 *      payloads (single NAL, STAP-A, FU-A; RFC 6184 packetization-mode 1) back to back into `out`; lens[i] is the
 *      size of payload i.  Byte-identical to the reference (tests/golden/rtp_h264_golden.json).  Host code, no GPU.
 *      Returns B2V_ENOMEM when out/lens are too small (out_cap >= au_size + au_size/600 + 64 always suffices). */
int  b2v_rtp_h264_packetize(const uint8_t* au, int32_t au_size, int32_t packet_max, uint8_t* out, int32_t out_cap,
                            int32_t* lens, int32_t max_packets, int32_t* n_packets);

#ifdef __cplusplus
}
#endif
#endif /* B2VIDEO_H_ */
