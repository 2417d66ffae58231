/*
 * mmw_radar.h — C ABI of the B200-native mmWave radar processing chain.
 *
 * This is the NEW surface (plain pointers and sizes, no C++/torch types) for
 * everything the reference's single entry point cannot carry: batches of
 * frames, run-time cube dimensions, detection lists, power maps and multi-GPU
 * frame sharding.  The reference's own entry point
 *     double cudaProcessing(short*, Complex_t*, int, double*, double*, double*, double*)
 * (acceleration.h:32, C++ linkage) is kept as a drop-in in mmw_legacy.h.
 *
 * What each call replaces in the reference:
 *   mmw_create / mmw_destroy      the per-frame cudaMalloc x6 / cudaFree x6 of cudaProcessing
 *                                 (acceleration.cu:435-437,471,474,499 / :564-569): allocated once.
 *   mmw_process_host              the body of cudaProcessing (acceleration.cu:417-572): H2D of the
 *                                 int16 capture (:438), unpack (:446), reshape (:454), FFT (:503-510),
 *                                 peak search (:518-523) — here a batch of frames and the full
 *                                 range / Doppler / CFAR / angle chain instead of one flat FFT.
 *   mmw_process_device            same, for captures already resident in HBM.
 *   mmw_read_* / mmw_copy_*       the reference's D2H of the spectrum (acceleration.cu:519).
 *   mmw_set_base_frame            cudaDataExtension_kernel's base-frame subtraction (acceleration.cu:152-166), all antennas.
 *   mmw_process_capture_file      the fopen / fread / one-call-per-frame loop of cudaTiming() (cudaBenchMarking.cpp:339-378).
 *   mmw_to_physical               the distance formula (cudaBenchMarking.cpp:301-303) and the constants of :10-19.
 *   mmw_legacy_*                  see mmw_legacy.h.
 *
 * Frame format (identical to the reference capture files, cudaBenchMarking.cpp:156-180):
 * little-endian int16, per frame [chirp][antenna][sample], samples in groups of four shorts
 * [I(2m) I(2m+1) Q(2m) Q(2m+1)]; frames concatenated without header.
 *
 * Threading: a context is not thread-safe — drive it from one host thread at a time; different contexts (also on
 * different GPUs, mmw_config.device) are independent and may be used concurrently.  mmw_last_error() is per thread.
 *
 * All functions return MMW_OK (0) or a negative error code; mmw_last_error() gives the text
 * of the calling thread's last failure.  There is no CPU fallback: without a CUDA device every
 * processing call fails with MMW_ERR_CUDA.
 */
#ifndef MMW_RADAR_H
#define MMW_RADAR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMW_OK 0
#define MMW_ERR_ARG (-1)          /* bad argument / unsupported shape */
#define MMW_ERR_CUDA (-2)         /* CUDA runtime failure (text in mmw_last_error) */
#define MMW_ERR_STATE (-3)        /* call not valid in this state (e.g. cube not kept) */
#define MMW_ERR_OVERFLOW (-4)     /* more detections than the destination can hold (list truncated) */

#define MMW_FLAG_PEAK 0x1u        /* detection is the strict 3x3 maximum among detected cells */

typedef struct mmw_ctx mmw_ctx;

/* 24-byte detection record (SURVEY.md §8a n8) */
typedef struct mmw_detection {
    uint32_t frame;        /* frame index inside the batch (plus frame_offset, see mmw_set_frame_offset) */
    uint16_t range_bin;    /* 0 .. Sp-1 */
    uint16_t doppler_bin;  /* 0 .. Cp-1, no fftshift: bins >= Cp/2 are negative velocities */
    float power;           /* integrated |X|^2 over antennas */
    float noise;           /* CA-CFAR training mean */
    int16_t angle_bin;     /* arg-max of the angle FFT wrapped to [-Ntheta/2, Ntheta/2) */
    uint16_t flags;        /* MMW_FLAG_* */
    float angle_rad;       /* asin(angle_bin * lambda_over_d / Ntheta) */
} mmw_detection;

typedef struct mmw_config {
    int n_samples;          /* S, samples per chirp (multiple of 4; zero-padded to Sp = nextPow2(S), 64..1024) */
    int n_chirps;           /* C, chirps per frame (multiple of 2; zero-padded to Cp = nextPow2(C), 64..1024) */
    int n_antennas;         /* A, virtual antennas (1..256) */
    int max_frames;         /* batch capacity: frames per mmw_process_* call */
    int cfar_guard_r, cfar_guard_d;   /* guard half-widths (range, Doppler) */
    int cfar_train_r, cfar_train_d;   /* training half-widths beyond the guard */
    float cfar_alpha;       /* detect iff P > alpha * mean(training cells) */
    int max_det_per_frame;  /* capacity of each frame's detection list (<= 65536; max_frames * this <= 2^28) */
    int keep_doppler_cube;  /* 1: write the full Doppler cube to HBM (mmw_copy_doppler_cube works);
                               0: fused — the angle stage re-derives only the detected cells */
    float lambda_over_d;    /* wavelength / element spacing, 2.0 for a half-wavelength array */
    int device;             /* CUDA device ordinal, -1 = current device */
} mmw_config;

typedef struct mmw_info {
    int Sp, Cp, n_theta;
    int sm_count;
    long long adc_bytes_per_frame;      /* 4*S*C*A */
    long long algorithmic_bytes_per_frame; /* 28*N + 8*M, SURVEY.md §8d, N = Sp*Cp*A, M = Sp*Cp */
    long long workspace_bytes;          /* HBM held by the context */
    int kernels_per_batch;              /* launches one mmw_process_device() issues */
} mmw_info;

/* defaults: CFAR guard (2,2) train (8,4) alpha 15, 1024 detections/frame, fused cube, lambda/d = 2 */
void mmw_default_config(mmw_config *cfg, int n_samples, int n_chirps, int n_antennas, int max_frames);

int mmw_create(const mmw_config *cfg, mmw_ctx **out);
void mmw_destroy(mmw_ctx *ctx);
const char *mmw_last_error(void);
int mmw_get_info(const mmw_ctx *ctx, mmw_info *info);

/* Window tables (fp32, host pointers). NULL keeps the default periodic Hann
 * w[n] = 0.5 - 0.5 cos(2 pi n / L).  win_range has S entries, win_doppler C. */
int mmw_set_windows(mmw_ctx *ctx, const float *win_range, const float *win_doppler);
/* copies the tables currently in use back to the host (either pointer may be NULL) */
int mmw_get_windows(const mmw_ctx *ctx, float *win_range, float *win_doppler);
/* Static-clutter removal: `base_host` is one frame in capture format (2*S*C*A int16); it is subtracted sample by
 * sample, in integers, from every frame before the range window — the reference's base-frame subtraction
 * (acceleration.cu:152-166, cudaBenchMarking.cpp:277-280: rx0 of frame 0) applied to every antenna.  NULL turns it off. */
int mmw_set_base_frame(mmw_ctx *ctx, const int16_t *base_host);
/* value added to mmw_detection.frame (the global index of the batch's first frame on this GPU) */
int mmw_set_frame_offset(mmw_ctx *ctx, uint32_t first_frame);

/* CUDA-graph mode for launch-bound use (one or a few frames per call, e.g. per-sensor streaming): the launch sequence
 * of a batch is captured once per distinct (capture address, n_frames, base frame, stream) and replayed with a single
 * cudaGraphLaunch.  The frame offset is not part of that key: a new value is patched into the instantiated graph
 * (one kernel-node parameter update on the host), so a stream of frames with advancing indices replays one graph.
 * Off by default; results are identical either way. */
int mmw_set_graph_mode(mmw_ctx *ctx, int enable);

/* How the detection records get their antenna snapshots when the Doppler cube is not kept (fused mode).
 * MMW_DETECT_PER_CELL: every detection re-derives its Doppler bin from the range spectrum, one DFT per detection per antenna
 *   (detections of one range bin share the rows they read) — one kernel, the lowest latency for a few frames per call.
 * MMW_DETECT_REFFT: every (frame, range bin) row that has a hit is Doppler-transformed once more by the FFT stage's own code
 *   and the detected bins are picked out of it (snapshots bit-identical to what the cube would hold), then the angle spectra
 *   are FFTs — three kernels, the cheaper path for large batches (256 x 128 x 4 x 1024 frames: 0.135 -> 0.08 ms).
 * MMW_DETECT_AUTO (default): _REFFT for arrays of 32 antennas and more, _PER_CELL below.
 * The two paths agree on everything but angle bins at near ties of the angle spectrum; a job that shards frames over
 * several contexts must give all of them the same path to get byte-identical lists.  Call between batches.
 * (The reference has no detection stage; acceleration.cu:518-523 picks one range peak on the host.) */
#define MMW_DETECT_AUTO 0
#define MMW_DETECT_PER_CELL 1
#define MMW_DETECT_REFFT 2
int mmw_set_detect_path(mmw_ctx *ctx, int path);

/* The CUDA stream every call of this context runs on (a cudaStream_t). */
void *mmw_stream(mmw_ctx *ctx);
/* Run on a caller-owned stream instead (e.g. torch's current stream); NULL restores the context's own. */
int mmw_use_stream(mmw_ctx *ctx, void *cuda_stream);

/* ADC cube already in HBM -> detections in HBM. Asynchronous on the context stream.
 * adc_dev: n_frames * 2*S*C*A int16, 16-byte aligned. */
int mmw_process_device(mmw_ctx *ctx, const int16_t *adc_dev, int n_frames);

/* Host capture -> detections on the host: H2D, the whole chain, D2H; synchronous.
 * dets receives up to det_capacity records ordered by (frame, range_bin, doppler_bin);
 * *n_det is the number written. Returns MMW_ERR_OVERFLOW (after filling dets) if some
 * frame exceeded max_det_per_frame or the total exceeded det_capacity. */
int mmw_process_host(mmw_ctx *ctx, const int16_t *adc_host, int n_frames,
                     mmw_detection *dets, int det_capacity, int *n_det);

/* The two halves of mmw_process_host, for streaming with several batches in flight (one context per batch in flight,
 * each with its own stream): mmw_submit_host queues the upload, the chain and the read-back of the result block and
 * returns without waiting; mmw_wait blocks until that batch is done and hands out its detections.  The capture buffer
 * must stay valid until mmw_wait returns and should be pinned (a pageable buffer makes the upload synchronous).
 * One batch per context at a time: between a submit and its wait, a second submit and every other call that would run or
 * read a batch on this context (mmw_process_device, mmw_time_device, mmw_read_detections, mmw_process_capture_file) return
 * MMW_ERR_STATE. */
int mmw_submit_host(mmw_ctx *ctx, const int16_t *adc_host, int n_frames);
int mmw_wait(mmw_ctx *ctx, mmw_detection *dets, int det_capacity, int *n_det);

/* After mmw_process_device: synchronises, then copies the ordered detection list. */
int mmw_read_detections(mmw_ctx *ctx, mmw_detection *dets, int det_capacity, int *n_det);
/* per-frame TRUE detection counts of the last batch (may exceed max_det_per_frame) */
int mmw_read_counts(mmw_ctx *ctx, uint32_t *counts, int n_frames);
/* Device views for zero-copy consumers (e.g. an NCCL gather): after mmw_process_device,
 * *dense_dets points at the packed ordered list and *header at {uint32 n_written, uint32 n_total,
 * uint32 n_frames, uint32 overflow}. Valid until the next process call. */
int mmw_device_results(mmw_ctx *ctx, const mmw_detection **dense_dets, const uint32_t **header);

/* The header and the dense list are one contiguous device block: MMW_RESULT_HEADER_BYTES bytes of header
 * {uint32 n_written, n_total, n_frames, overflow, 4 x reserved} followed by the records.  A fixed-size prefix of
 * this block is what a multi-GPU gather sends (no host round trip to learn the count first). */
#define MMW_RESULT_HEADER_BYTES 32
int mmw_device_result_block(mmw_ctx *ctx, const void **block, long long *capacity_bytes);
/* Rank-0 side of the gather: `gathered_dev` holds n_ranks result blocks (header + records) at a stride of
 * stride_bytes, in rank order (= frame order).  Writes one merged block (header + all records, still ordered by
 * (frame, range, doppler)) to merged_dev, which can hold merged_capacity records.  Asynchronous on the context
 * stream; one kernel. */
int mmw_merge_gathered(mmw_ctx *ctx, const void *gathered_dev, int n_ranks, long long stride_bytes,
                       void *merged_dev, int merged_capacity);

/* ---- multi-GPU: a frame-sharded group of GPUs driven by ONE host process (SURVEY.md §8e) ----
 * The reference is single-GPU, one frame per call (acceleration.h:32, cudaBenchMarking.cpp:374-378); frames are independent,
 * so a batch shards by frame.  A group owns one context per device (same config; cfg->max_frames is the capacity PER GPU)
 * and one NCCL communicator over them (single process, one rank per device; NCCL is loaded at run time from libnccl.so.2,
 * the library has no link-time dependency on it).  A batch of n frames is cut into contiguous blocks — GPU i gets frames
 * [first_i, first_i + n_i), remainders to the low ranks — every GPU runs the whole chain on its block with no data-path
 * collective, and the one exchange step gathers the ordered detection lists to GPU 0: the 32-byte headers first, then
 * exactly count_i records from each rank (grouped ncclSend / ncclRecv over NVLink), landing at their final offsets of one
 * merged block [32-byte header | records ordered by (frame, range, doppler)] in GPU 0's memory.  mmw_detection.frame
 * counts from the start of the batch (plus mmw_group_set_frame_offset).  The NCCL kernels are held to one CTA per peer
 * (ncclConfig_t.maxCTAs) so that they do not evict the persistent FFT kernels of a batch in flight.
 * One-process-per-GPU launchers (torchrun) use mmw_device_result_block / mmw_merge_gathered with their own communicator
 * instead (sharding.py).  Not thread-safe: drive a group from one host thread. */
typedef struct mmw_group mmw_group;
int mmw_group_create(const mmw_config *cfg, const int *devices, int n_devices, mmw_group **out);
void mmw_group_destroy(mmw_group *group);
int mmw_group_size(const mmw_group *group);
/* the context on the i-th device of the group (windows, base frame, intermediates of its shard); owned by the group */
mmw_ctx *mmw_group_context(mmw_group *group, int i);
/* index of the batch's first frame (added to every record's frame field) */
int mmw_group_set_frame_offset(mmw_group *group, uint32_t first_frame);
/* frames [first, first + count) of an n-frame batch owned by rank `rank` of `n_ranks` (the rule the group uses) */
void mmw_shard_frames(int n_frames, int n_ranks, int rank, int *first, int *count);
/* Host capture of n_frames frames (n_frames <= n_devices * max_frames; should be pinned) -> sharded upload -> chain on
 * every GPU -> NCCL gather to GPU 0 -> ordered detection list on the host.  Same result, byte for byte, as one GPU
 * processing the whole batch.  Returns MMW_OK or MMW_ERR_OVERFLOW as mmw_process_host does. */
int mmw_group_process_host(mmw_group *group, const int16_t *adc_host, int n_frames,
                           mmw_detection *dets, int det_capacity, int *n_det);
/* Device-resident shards: adc_dev[i] points at n_frames[i] frames in the memory of the group's i-th device (n_frames[i]
 * may be 0).  Runs the chain and the gather; the merged block stays on GPU 0. */
int mmw_group_process_device(mmw_group *group, const int16_t *const *adc_dev, const int *n_frames);
/* after mmw_group_process_device: the merged block on GPU 0 ([MMW_RESULT_HEADER_BYTES header | records]); the gather has
 * been queued on GPU 0's stream (mmw_stream(mmw_group_context(group, 0))) — synchronise that stream before reading */
int mmw_group_merged_block(mmw_group *group, const void **block_dev0, long long *capacity_bytes);
/* after mmw_group_process_device: waits for the gather and copies the merged list to the host */
int mmw_group_read_detections(mmw_group *group, mmw_detection *dets, int det_capacity, int *n_det);

/* ---- capture-file ingest (the caller side of the boundary: the fopen/fread loop of cudaBenchMarking.cpp:339-378) ----
 * Reads a raw capture (frames of 2*S*C*A little-endian int16, no header — the fhy_direct.bin format) from `path`,
 * starting at frame `first_frame`, at most `max_frames` frames (<= 0: to the end of the file), and runs the chain over
 * it in batches of the context's max_frames.  The file is read into pinned double buffers so that the fread of batch
 * k+1 overlaps the H2D copy and kernels of batch k.  mmw_detection.frame counts from the start of the FILE.
 * A trailing partial frame is zero-filled and processed (the reference passes the short count on and processes the
 * frame anyway, cudaBenchMarking.cpp:374-377).  use_first_as_base != 0: the first frame read becomes the base frame
 * (mmw_set_base_frame) and is not itself processed — the reference's cudaTiming() convention (:357-365); it replaces any
 * base frame set before and STAYS installed after the call returns (mmw_set_base_frame(ctx, NULL) turns it off).
 * *n_frames_done receives the number of frames processed.  Returns MMW_OK, MMW_ERR_OVERFLOW (list truncated) or an
 * error (MMW_ERR_ARG if the file cannot be opened). */
int mmw_process_capture_file(mmw_ctx *ctx, const char *path, long long first_frame, int max_frames, int use_first_as_base,
                             mmw_detection *dets, int det_capacity, int *n_det, int *n_frames_done);

/* ---- detections in physical units (SURVEY.md §8f row 3) ----
 * The reference declares the radar constants for exactly this but only ever computes a range (cudaBenchMarking.cpp:
 * 10-19, 301-303).  Host arithmetic on the (small) detection list; no device work. */
typedef struct mmw_radar_params {
    double f0_hz;            /* carrier, 77e9           (cudaBenchMarking.cpp:10  F0) */
    double slope_hz_per_s;   /* chirp slope, 5.987e12   (:11 mu)                      */
    double fs_hz;            /* ADC sample rate, 2e6    (:13 Fs)                      */
    double chirp_period_s;   /* chirp repetition, 64e-6 (:15 Tr)                      */
    double light_speed;      /* 3.0e8 as the reference writes it (:12 c)              */
} mmw_radar_params;
typedef struct mmw_target {
    uint32_t frame;
    float range_m;           /* c * (range_bin * Fs / Sp) / (2 mu) — the reference's distance formula per chirp */
    float velocity_mps;      /* (lambda / 2) * d' / (Cp * Tr), d' = doppler_bin wrapped to [-Cp/2, Cp/2) */
    float angle_deg;         /* angle_rad in degrees */
    float snr_db;            /* 10 log10(power / noise) */
    uint32_t flags;          /* MMW_FLAG_* of the detection */
} mmw_target;
void mmw_default_radar_params(mmw_radar_params *rp);
/* Sp, Cp: the FFT lengths the detections were made with (mmw_info.Sp / .Cp) */
int mmw_to_physical(const mmw_radar_params *rp, int Sp, int Cp, const mmw_detection *dets, int n, mmw_target *out);

/* ---- clustering: each frame's detections grouped into objects, on the GPU (off by default) ----
 * One target under the Hann windows lights up a blob of neighbouring cells; MMW_FLAG_PEAK marks the blob's maximum but not
 * its members.  With clustering on, every batch also produces an ordered object list and a label per detection.
 * Definition (tests/cluster_ref.c: ref_cluster, a plain-C fp64 reference, is the specification; the GPU matches it bit for bit):
 *   signed Doppler d' = d < Cp/2 ? d : d - Cp, without wrap: a blob that straddles +-Cp/2 becomes two objects;
 *   detections i, j of one frame are neighbours iff |r_i - r_j| <= eps_range, |d'_i - d'_j| <= eps_doppler and
 *   |angle_bin_i - angle_bin_j| <= eps_angle (eps_angle >= n_theta ignores the angle);
 *   components of the neighbour graph (friends-of-friends: DBSCAN with min_points = 1, unique whatever the order) with at
 *   least min_points members are objects, ordered by (frame, lowest member index); at most max_objects_per_frame per frame
 *   are kept, the true count is always reported.
 * The kernels read the finished detection list and write their own buffers only: the detections are the same bytes with
 * clustering on or off.  They run at the end of every batch (mmw_process_device / _host, mmw_submit_host, capture-file
 * ingest, graph mode) and mmw_time_device counts them in stage 4.
 * Multi-GPU: mmw_group_* and mmw_exchange_* gather detections only; enable clustering on each mmw_group_context() and read
 * the objects of each shard from that context. */
typedef struct mmw_cluster_params {
    int eps_range;              /* 0..16 range bins */
    int eps_doppler;            /* 0..16 Doppler bins (signed, no wrap) */
    int eps_angle;              /* >= 0 angle bins; >= n_theta: angle ignored */
    int min_points;             /* >= 1 detections per object */
    int max_objects_per_frame;  /* 1..max_det_per_frame */
} mmw_cluster_params;

/* 48-byte object record.  Sums run over the members in ascending detection index, in fp64, rounded to fp32 once. */
typedef struct mmw_object {
    uint32_t frame;        /* the members' mmw_detection.frame (frame offset included) */
    uint32_t first_det;    /* index of the lowest-index member in the batch's detection list */
    uint32_t n_det;        /* members */
    uint32_t peak_det;     /* index of the strongest member (equal power: the lower index) */
    float range_bin;       /* power-weighted mean range bin */
    float doppler_bin;     /* power-weighted mean signed Doppler bin d' */
    float angle_rad;       /* power-weighted mean angle_rad */
    float power;           /* sum of the members' power */
    float peak_power;      /* power and noise of peak_det */
    float peak_noise;
    uint16_t range_min, range_max;
    int16_t doppler_min, doppler_max;   /* signed d' */
} mmw_object;

/* object header: {n_written, n_total, n_frames, flags} + 4 reserved words; flags bit 0: some frame had more than
 * max_objects_per_frame objects (those were cut), bit 1: the detection list itself was truncated (max_det_per_frame) */
#define MMW_OBJECT_HEADER_BYTES 32
#define MMW_OBJECTS_CUT 0x1u
#define MMW_OBJECTS_DETECTIONS_TRUNCATED 0x2u

/* (2, 2, 4, 1, 256) */
void mmw_default_cluster_params(mmw_cluster_params *cp);
/* cp = NULL turns clustering off (the default) and releases its buffers; otherwise checks the parameters, allocates the
 * buffers (all of them: nothing is allocated inside a batch, which may be under stream capture) and turns it on.
 * MMW_ERR_STATE while a submitted batch is pending.  Call between batches. */
int mmw_set_clustering(mmw_ctx *ctx, const mmw_cluster_params *cp);
/* After a batch with clustering on: synchronises, copies up to `capacity` objects.  Returns MMW_ERR_OVERFLOW (after
 * filling objs) if the header has a flag set or there were more than `capacity` objects. */
int mmw_read_objects(mmw_ctx *ctx, mmw_object *objs, int capacity, int *n_obj);
/* Per detection of the last batch (aligned with its detection list): the index of its object in the object list, or -1
 * (its component is smaller than min_points, or its object was cut).  MMW_ERR_OVERFLOW if capacity < detections. */
int mmw_read_labels(mmw_ctx *ctx, int32_t *labels, int capacity, int *n);
/* device views: *objs at the object records, *header at the MMW_OBJECT_HEADER_BYTES header right before them */
int mmw_device_objects(mmw_ctx *ctx, const mmw_object **objs, const uint32_t **header);
/* objects in physical units with mmw_to_physical's formulas applied to the fractional mean bins; snr_db is
 * 10 log10(peak_power / peak_noise), flags is 0 */
int mmw_objects_to_physical(const mmw_radar_params *rp, int Sp, int Cp, const mmw_object *objs, int n, mmw_target *out);

/* Intermediates of one frame of the last batch, copied to the host in canonical layouts
 * (synchronous, not on the hot path):
 *   range spectrum [A][Sp][C]  complex64 — NOTE: already multiplied by the Doppler window w_d[c]
 *   Doppler cube   [A][Sp][Cp] complex64 — needs keep_doppler_cube = 1
 *   power map      [Sp][Cp]    float32
 *   CFAR mask      [Sp][Cp]    uint8 */
int mmw_copy_range_spectrum(mmw_ctx *ctx, int frame, float *out);
int mmw_copy_doppler_cube(mmw_ctx *ctx, int frame, float *out);
int mmw_copy_power_map(mmw_ctx *ctx, int frame, float *out);
int mmw_copy_cfar_mask(mmw_ctx *ctx, int frame, uint8_t *out);

/* Device timing helper: runs mmw_process_device `iters` times back to back on the context
 * stream between two CUDA events and returns the elapsed milliseconds (total, not per run).
 * per_stage_ms (optional, 4 floats) receives the summed time of each stage
 * (range, doppler, cfar, detect+compact, plus the clustering kernels when clustering is on) measured with events between
 * the launches. */
int mmw_time_device(mmw_ctx *ctx, const int16_t *adc_dev, int n_frames, int iters,
                    float *total_ms, float *per_stage_ms);

/* Guard bands (a memcheck of our own; compute-sanitizer is not available on every pool): a context created with MMW_GUARD=1 in
 * the environment brackets every device buffer it owns (range spectrum, cube, power map, mask, noise, keys, counts, result
 * block, tables, staging, ...) with two 4 KB bands of a known byte.  mmw_check_guards synchronises the device, reads the bands
 * back and writes the number of overwritten guard bytes to *bad_bytes (0 = no kernel of the chain wrote out of bounds since
 * mmw_create; mmw_last_error() names the first buffer hit otherwise).  Returns MMW_ERR_STATE on a context created without
 * the switch.  The reference has no such check; its cudaDataExtension_kernel leaves element 12 800 uninitialised and its
 * reshape kernel reads out of bounds (acceleration.cu:152-166, 117-150; SURVEY.md §2.3). */
int mmw_check_guards(mmw_ctx *ctx, long long *bad_bytes);

/* ---- the exchange step of a frame-sharded job with ONE PROCESS PER GPU, without a kernel (SURVEY.md §8e) ----
 * The reference has no multi-GPU path (cudaBenchMarking.cpp:374-378 feeds one frame at a time to one GPU).  Every rank puts a
 * fixed-size prefix of its result block ([32-byte header | records_per_rank records], mmw_device_result_block) straight into
 * rank 0's memory over NVLink with the copy engine (a cudaIpc-mapped peer pointer) and raises an arrival counter there with a
 * stream memory operation; rank 0's side stream waits for the counters, runs the one merge kernel (as mmw_merge_gathered)
 * and writes a credit back so that a slot is not overwritten while it is being merged (`depth` steps may be in flight).
 * No NCCL kernel competes with the persistent FFT kernels for an SM.  Set-up: create on every rank, exchange the 64-byte
 * handles with any transport (bench.py: torch.distributed all_gather over NCCL), connect.  Per step, on every rank after
 * mmw_process_device: mmw_exchange_put; on rank 0 also mmw_exchange_merge.  All calls are asynchronous. */
typedef struct mmw_exchange mmw_exchange;
int mmw_exchange_create(mmw_ctx *ctx, int rank, int n_ranks, int records_per_rank, int depth, mmw_exchange **out);
void mmw_exchange_destroy(mmw_exchange *x);
int mmw_exchange_handle(mmw_exchange *x, void *handle64);                 /* 64 bytes out */
int mmw_exchange_connect(mmw_exchange *x, const void *all_handles);       /* n_ranks x 64 bytes, in rank order */
int mmw_exchange_put(mmw_exchange *x);                                    /* on the context's stream */
int mmw_exchange_merge(mmw_exchange *x, const void **merged_block);       /* rank 0: [32-byte header | ordered records], device */
int mmw_exchange_wait(mmw_exchange *x, void *cuda_stream, const void **merged_block);   /* rank 0: stream waits for the last merge */

#ifdef __cplusplus
}
#endif
#endif
