// mmw_common.cuh — shared declarations of the B200 radar pipeline (device side).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mmw_radar.h"

namespace mmw {

// ---------------------------------------------------------------------------
// device-side view of one plan (all pointers are device pointers)
// ---------------------------------------------------------------------------
struct PlanDev {
    int S, C, A;            // samples / chirps / antennas as captured
    int Sp, Cp;             // FFT lengths (nextPow2)
    int n_theta;            // angle FFT length
    int guard_r, guard_d, win_r_half, win_d_half;   // CFAR: guard and guard+train half widths
    float alpha;
    float lambda_over_d;
    int max_det;            // per-frame detection capacity
    int keep_cube;          // materialise the Doppler cube
    uint32_t frame_offset;  // added to mmw_detection.frame
    const float *win_r;     // [S]   range window
    const float *win_d;     // [C]   Doppler window
    const float2 *tw_d;     // [Cp]  exp(-2 pi i k / Cp), natural order (fused-mode Doppler bin evaluation)
    const float2 *tw1_r;    // [Sp]  pass-1 twiddles of the range FFT in consumption order (tw1_index)
    const float2 *tw1_d;    // [Cp]  pass-1 twiddles of the Doppler FFT in consumption order
    const float2 *tw_a;     // [n_theta]
    unsigned int *sched;    // [2] K1's tile counter {next tile, CTAs retired}; zero between launches
    const int16_t *base_adc; // one frame [C][A][S] IIQQ subtracted before the range window, or nullptr (static-clutter removal)
    int detect_path;        // host-side only: MMW_DETECT_AUTO / _PER_CELL / _REFFT (mmw_set_detect_path), read by launch_detect
    // Padding to a multiple of 16 bytes: the pointer arguments after the plan then keep their 16-byte pairing, which the
    // compiler loads with one 128-bit constant load (measure_wide_kernel).  alignas(16) would do the same but changes
    // the code of the kernels that read the plan's first fields.
    int pad_[3];
};
static_assert(sizeof(PlanDev) % 16 == 0, "PlanDev size");

// internal HBM layouts (DESIGN.md §3)
//   adc   [F][C][A][S]  int16 IIQQ   (the reference's capture format)
//   rs    [F][A][Sp][C] float2       range spectrum, already multiplied by win_d[c]
//   cube  [F][A][Cp][Sp] float2      Doppler cube (only if keep_cube)
//   pmap  [F][Cp][Sp]   float        integrated power, range fastest
//   mask  [F][Cp/32][Sp] uint32      CFAR hits, bit j of word (w, r) <-> doppler 32 w + j
//   keys  [F][max_det]  uint32 (range<<16 | doppler), counts [F], offsets [F+1]
//   dense [<= F*max_det] mmw_detection, ordered by (frame, range, doppler); header[4]

// ---------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D bulk tensor-memory-accelerator copies (UBLKCP)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// global -> shared bulk copy; completion is signalled on `bar` as transaction bytes.
// dst, src and bytes must be multiples of 16.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void st_global_f2(float2 *p, float2 v)
{
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

// ---------------------------------------------------------------------------
// host-side launchers (mmw_pipeline.cu) — return cudaError_t
// ---------------------------------------------------------------------------
cudaError_t launch_range_fft(const PlanDev &p, const int16_t *adc, float2 *rs, int n_frames, cudaStream_t st);
cudaError_t launch_doppler_fft(const PlanDev &p, const float2 *rs, float2 *cube, float *pmap, int n_frames, cudaStream_t st);
// small batches: K2 over F*A single-antenna frames into per-antenna maps, then the ordered sum (mmw_pipeline.cu)
bool doppler_prefers_split(const PlanDev &p, int n_frames);
cudaError_t launch_power_sum(const PlanDev &p, const float *per_antenna, float *pmap, int n_frames, cudaStream_t st);
// everything stages 3/4 read and write (device pointers)
struct DetectBuffers {
    const float2 *rs;
    const float2 *cube;
    const float *pmap;
    float *noise_map;       // [F][Cp][Sp], valid at hit cells only
    uint32_t *mask;         // [F][Cp/32][Sp]
    uint32_t *keys;         // [F][max_det]  (range << 16 | doppler), ordered
    uint32_t *counts;       // [F]    true hit count per frame
    uint32_t *offsets;      // [F+1]  exclusive scan of min(count, max_det)
    uint32_t *header;       // {n_written, n_total, n_frames, overflow}
    unsigned int *ticket;   // [0] last-CTA-done counter of list_kernel, [1] work cursor of measure_kernel, [2] hit-row count (all self-resetting)
    mmw_detection *dense;   // ordered detection list of the batch
    // buffers of the selective Doppler re-FFT path (detect_uses_refft; nullptr: a per-detection kernel instead)
    uint4 *rows;            // [F * Sp] {frame, range bin, dense index of the row's first hit, -}: every (frame, range bin) with hits
    float2 *snap;           // [dense capacity][A] antenna snapshots of the detected cells
};
cudaError_t launch_cfar(const PlanDev &p, const float *pmap, uint32_t *mask, float *noise_map, int n_frames, int sm_count, cudaStream_t st);
cudaError_t launch_detect(const PlanDev &p, const DetectBuffers &b, int n_frames, int dense_cap, int sm_count, cudaStream_t st);
// whether launch_detect takes the selective re-FFT path for this plan (mmw_detect.cu)
bool detect_uses_refft(const PlanDev &p, bool have_refft_buffers);
// the kernels that write mmw_detection records (the only readers of PlanDev.frame_offset, their argument 0): graph mode patches
// that argument in place instead of re-capturing when the frame offset changes (mmw_api.cu).  Returns the kernel's argument
// count, 0 if `func` is not one of them.
constexpr int kRecordKernelMaxArgs = 12;
int record_kernel_args(const void *func);
cudaError_t launch_doppler_extract(const PlanDev &p, const float2 *rs, const uint32_t *keys, const uint32_t *offsets, const uint4 *rows,
                                   const unsigned int *n_rows, float2 *snap, int dense_cap, int max_rows, cudaStream_t st);
cudaError_t launch_merge(const unsigned char *gathered, int n_ranks, size_t stride_bytes, unsigned char *merged, int merged_cap,
                         cudaStream_t st);
// clustering of the finished detection list into objects (mmw_cluster.cu); every buffer is [dense capacity] unless noted
struct ClusterBuffers {
    const mmw_detection *dense;     // the batch's detection list, its header {n_written, n_total, n_frames, overflow}
    const uint32_t *det_header;
    const uint32_t *keys;           // [F][max_det] (range << 16 | doppler) of list_kernel, offsets [F+1]
    const uint32_t *offsets;
    int *parent;                    // union-find forest; after the flatten pass the component root (its lowest index)
    uint32_t *size;                 // component size, at the root
    int *oid;                       // at a root: frame-local object number, -1 if the component is not an object
    uint32_t *cursor;               // at a kept root: next free slot of its members in `members`
    uint32_t *members;              // member indices grouped by object, ascending within each object
    int32_t *labels;                // object index per detection, -1 if none
    uint32_t *frame_objs;           // [2F] objects per frame: true count, kept count
    uint32_t *obj_offsets;          // [F+1] exclusive scan of the kept counts
    uint2 *slots;                   // [F][max_obj] {root, first member slot} of each kept object
    unsigned int *ticket;           // [1] last-CTA-done counter of the order kernel (self-resetting)
    uint32_t *obj_header;           // MMW_OBJECT_HEADER_BYTES
    mmw_object *objs;               // [F][max_obj] capacity
};
constexpr int kClusterKernels = 5;
cudaError_t launch_cluster(const mmw_cluster_params &cp, int Cp, int max_det, const ClusterBuffers &b, int n_frames, int dense_cap,
                           int sm_count, cudaStream_t st);
// export helpers (not on the hot path): internal layout -> the canonical layouts of mmw_radar.h
cudaError_t launch_export_cube(const PlanDev &p, const float2 *cube_frame, float2 *out, cudaStream_t st);
cudaError_t launch_export_pmap(const PlanDev &p, const float *pmap_frame, float *out, cudaStream_t st);
cudaError_t launch_export_mask(const PlanDev &p, const uint32_t *mask_frame, uint8_t *out, cudaStream_t st);
bool plan_supported(int Sp, int Cp, const char **why);
constexpr int kMaxDevices = 64;
int current_device();       // ordinal of the calling thread's current device, clamped to [0, kMaxDevices)
void plan_radices(int n, int *r1, int *r2);

// legacy single-frame path (mmw_legacy.cu)
struct LegacyDev {
    const float2 *tw;       // [16384]
    const double2 *base;    // [12800] base frame rx0 (as handed in by the caller)
    float2 *spectrum;       // [16384] optional export
    unsigned long long *best;  // packed (|X|^2 bits, ~index)
};

}  // namespace mmw
