// mmw_api.cu — host side of the C ABI declared in include/mmw_radar.h: context, plan tables,
// HBM workspace, stream, and the launch sequence of one batch.  No torch types, no CPU compute
// path: every processing call either launches the CUDA kernels or fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>       // types and prototypes only: the functions are resolved from libnccl.so.2 at run time (mmw_group_create)
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <tuple>
#include <vector>

#include "mmw_common.cuh"

namespace mmw {

static thread_local char g_err[512] = "";

void set_last_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int next_pow2(int n)
{
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}

}  // namespace mmw

using namespace mmw;

constexpr int kMaxChunks = 32;
constexpr int kResultHeaderBytes = MMW_RESULT_HEADER_BYTES;

struct mmw_ctx {
    mmw_config cfg;
    PlanDev plan;
    int device;
    int sm_count;
    cudaStream_t own_stream;
    cudaStream_t stream;
    // tables
    float *d_win_r, *d_win_d;
    float2 *d_tw_d, *d_tw_a, *d_tw1_r, *d_tw1_d;
    // workspace
    int16_t *d_adc;          // staging for host captures
    int16_t *d_base;         // base frame for static-clutter removal (lazy)
    int16_t *h_ring[2];      // pinned double buffer of the capture-file reader (lazy)
    float2 *d_rs;
    float2 *d_cube;
    float *d_pmap;
    float *d_psplit;         // per-antenna power maps of the antenna-split path for small batches (lazy)
    int psplit_frames;       // frames d_psplit holds
    uint32_t *d_mask;
    float *d_noise;
    uint32_t *d_keys;
    uint32_t *d_counts;
    uint32_t *d_offsets;
    unsigned int *d_ticket;
    unsigned int *d_sched;        // PlanDev.sched
    uint4 *d_rows;            // hit rows of the selective Doppler re-FFT (wide arrays, fused mode)
    float2 *d_snap;           // antenna snapshots of the detected cells (same path)
    unsigned char *d_result;  // [32-byte header | dense ordered detection list]: one D2H usually moves both
    mmw_detection *d_dense;
    uint32_t *d_header;
    void *d_scratch;         // export scratch
    size_t scratch_bytes;
    // MMW_GUARD=1 at mmw_create: every device buffer of the context sits between two kGuardBytes bands filled with kGuardByte;
    // mmw_check_guards reads them back (compute-sanitizer's memcheck is not available on every pool: this catches any
    // out-of-bounds WRITE of any kernel of the chain, at the granularity of one byte past either end)
    int guard_on;
    struct GuardedBuf { unsigned char *base; void *user; size_t bytes; const char *name; };
    std::vector<GuardedBuf> *guards;
    // pinned host
    unsigned char *h_result;  // pinned mirror of d_result
    uint32_t *h_header;
    mmw_detection *h_dense;
    uint32_t guess_det;       // records fetched speculatively with the header (adapts to the last batch)
    uint32_t fetched;         // records covered by the D2H queued by enqueue_fetch
    int submitted;            // a batch queued by mmw_submit_host is waiting for mmw_wait
    cudaStream_t copy_stream; // H2D of host captures, overlapped chunk-wise with the kernels
    cudaEvent_t chunk_ev[kMaxChunks];
    int dense_cap;
    int last_frames;
    size_t workspace_bytes;
    cudaEvent_t ev[6];
    // CUDA-graph mode (mmw_set_graph_mode): the launch sequence of one batch, captured once per distinct
    // (capture address, frame count, base frame, stream) and replayed with one cudaGraphLaunch.  The frame offset is NOT
    // part of the key: it lives in the kernel parameters of one node (the record writer) and is patched into the
    // instantiated graph when it changes (cudaGraphExecKernelNodeSetParams: host-side only), so a stream of frames with
    // advancing indices replays one graph.
    int graph_on;
    int graph_warm;           // the first batch runs eagerly: launchers set function attributes on first use
    struct GraphEntry {
        cudaGraph_t graph;            // kept: the parameter block the patch starts from lives in it
        cudaGraphExec_t exec;
        cudaGraphNode_t record_node;  // the kernel node whose PlanDev carries frame_offset (nullptr: none found)
        cudaKernelNodeParams record_kp;   // its launch parameters as captured (the argument pointers point into `graph`)
        int record_args;              // its argument count
        uint32_t frame_offset;        // value `exec` currently holds
    };
    std::map<std::tuple<const void *, int, const void *, void *>, GraphEntry> *graphs;
    // clustering (mmw_set_clustering): on when cluster_on; its buffers live from that call to the next one turning it off
    int cluster_on;
    mmw_cluster_params cluster;
    int last_clustered;       // the last batch ran the clustering kernels
    int *d_cl_parent, *d_cl_oid;
    uint32_t *d_cl_size, *d_cl_cursor, *d_cl_members, *d_cl_frame_objs, *d_cl_obj_offsets;
    int32_t *d_cl_labels;
    uint2 *d_cl_slots;
    unsigned int *d_cl_ticket;
    unsigned char *d_objects;   // [MMW_OBJECT_HEADER_BYTES header | max_frames * max_objects_per_frame records]
    size_t cluster_bytes;       // their share of workspace_bytes
};

static void destroy_graphs(mmw_ctx *c)
{
    if (!c->graphs) return;
    for (auto &kv : *c->graphs) {
        cudaGraphExecDestroy(kv.second.exec);
        cudaGraphDestroy(kv.second.graph);
    }
    c->graphs->clear();
}

static int env_int(const char *name)
{
    const char *v = getenv(name);
    return v ? atoi(v) : 0;
}

// A failed runtime call also parks its code in the runtime's per-thread "last error", where the launchers' cudaGetLastError()
// would find it after the NEXT (successful) kernel launch: it is cleared here, once it has been reported.
#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) {                                                                          \
            set_last_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);   \
            (void)cudaGetLastError();                                                                     \
            return MMW_ERR_CUDA;                                                                          \
        }                                                                                                 \
    } while (0)

constexpr size_t kGuardBytes = 4096;
constexpr int kGuardByte = 0xA5;

template <typename T>
static int dev_alloc_named(mmw_ctx *c, T **p, size_t count, const char *name)
{
    size_t bytes = count * sizeof(T);
    if (!bytes) bytes = 16;
    if (c->guard_on) {
        unsigned char *base = nullptr;
        CK(cudaMalloc((void **)&base, bytes + 2 * kGuardBytes));
        CK(cudaMemset(base, kGuardByte, kGuardBytes));
        CK(cudaMemset(base + kGuardBytes + bytes, kGuardByte, kGuardBytes));
        *p = reinterpret_cast<T *>(base + kGuardBytes);
        c->guards->push_back({base, (void *)*p, bytes, name});
    } else {
        CK(cudaMalloc((void **)p, bytes));
    }
    c->workspace_bytes += bytes;
    return MMW_OK;
}
#define dev_alloc(c, p, count) dev_alloc_named(c, p, count, #p)

// cudaFree of a buffer that came from dev_alloc (its guard bands go with it)
static void dev_free(mmw_ctx *c, void *user)
{
    if (!user) return;
    if (c->guard_on && c->guards) {
        for (size_t i = 0; i < c->guards->size(); ++i)
            if ((*c->guards)[i].user == user) {
                cudaFree((*c->guards)[i].base);
                c->guards->erase(c->guards->begin() + (long)i);
                return;
            }
    }
    cudaFree(user);
}

static void free_cluster_buffers(mmw_ctx *c)
{
    void *bufs[] = {c->d_cl_parent, c->d_cl_oid, c->d_cl_size, c->d_cl_cursor, c->d_cl_members, c->d_cl_frame_objs,
                    c->d_cl_obj_offsets, c->d_cl_labels, c->d_cl_slots, c->d_cl_ticket, c->d_objects};
    for (void *b : bufs) dev_free(c, b);
    c->d_cl_parent = c->d_cl_oid = nullptr;
    c->d_cl_size = c->d_cl_cursor = c->d_cl_members = c->d_cl_frame_objs = c->d_cl_obj_offsets = nullptr;
    c->d_cl_labels = nullptr;
    c->d_cl_slots = nullptr;
    c->d_cl_ticket = nullptr;
    c->d_objects = nullptr;
    c->workspace_bytes -= c->cluster_bytes;
    c->cluster_bytes = 0;
}

static std::vector<float2> make_twiddles(int n)
{
    std::vector<float2> t(n);
    for (int k = 0; k < n; ++k) {
        const double th = -2.0 * M_PI * (double)k / (double)n;
        t[k] = make_float2((float)cos(th), (float)sin(th));
    }
    return t;
}

// W_n^(n2*k1) for the two-pass plan of length n, laid out in the order pass 1 reads it (see tw1_index in mmw_pipeline.cu)
static std::vector<float2> make_pass1_twiddles(int n)
{
    int r1 = 0, r2 = 0;
    plan_radices(n, &r1, &r2);
    std::vector<float2> t(n);
    for (int n2 = 0; n2 < r2; ++n2)
        for (int k1 = 0; k1 < r1; ++k1) {
            const double th = -2.0 * M_PI * (double)((n2 * k1) % n) / (double)n;
            t[((n2 >> 1) * r1 + k1) * 2 + (n2 & 1)] = make_float2((float)cos(th), (float)sin(th));
        }
    return t;
}

static std::vector<float> make_hann(int n)
{
    std::vector<float> w(n);
    for (int i = 0; i < n; ++i) w[i] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * (double)i / (double)n));
    return w;
}

extern "C" {

const char *mmw_last_error(void) { return g_err; }

void mmw_default_config(mmw_config *cfg, int n_samples, int n_chirps, int n_antennas, int max_frames)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->n_samples = n_samples;
    cfg->n_chirps = n_chirps;
    cfg->n_antennas = n_antennas;
    cfg->max_frames = max_frames;
    cfg->cfar_guard_r = 2;
    cfg->cfar_guard_d = 2;
    cfg->cfar_train_r = 8;
    cfg->cfar_train_d = 4;
    cfg->cfar_alpha = 15.0f;
    cfg->max_det_per_frame = 1024;
    cfg->keep_doppler_cube = 0;
    cfg->lambda_over_d = 2.0f;
    cfg->device = -1;
}

void mmw_destroy(mmw_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    void *bufs[] = {c->d_win_r, c->d_win_d, c->d_tw1_r, c->d_tw1_d, c->d_tw_d, c->d_tw_a, c->d_adc, c->d_base, c->d_rs, c->d_cube, c->d_pmap,
                    c->d_psplit, c->d_mask, c->d_noise, c->d_keys, c->d_counts, c->d_offsets, c->d_ticket, c->d_sched,
                    c->d_rows, c->d_snap, c->d_result};
    for (void *b : bufs) dev_free(c, b);
    free_cluster_buffers(c);
    cudaFree(c->d_scratch);
    delete c->guards;
    if (c->h_result) cudaFreeHost(c->h_result);
    for (auto &h : c->h_ring) if (h) cudaFreeHost(h);
    for (auto &e : c->chunk_ev) if (e) cudaEventDestroy(e);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->graphs) {
        destroy_graphs(c);
        delete c->graphs;
    }
    for (auto &e : c->ev) if (e) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

// buffers of the selective Doppler re-FFT detection path (hit rows, antenna snapshots of the detected cells); no-op in cube
// mode, when they exist already, or when the snapshots would exceed 2 GB (the per-detection kernels are used then)
static int alloc_refft_buffers(mmw_ctx *c)
{
    const size_t A = (size_t)c->cfg.n_antennas;
    if (c->cfg.keep_doppler_cube || c->d_snap != nullptr) return MMW_OK;
    if ((size_t)c->dense_cap * A * sizeof(float2) > ((size_t)2 << 30)) return MMW_OK;
    int rc;
    if ((rc = dev_alloc(c, &c->d_rows, (size_t)c->cfg.max_frames * next_pow2(c->cfg.n_samples)))) return rc;
    if ((rc = dev_alloc(c, &c->d_snap, (size_t)c->dense_cap * A))) return rc;
    return MMW_OK;
}

int mmw_create(const mmw_config *cfg, mmw_ctx **out)
{
    if (!cfg || !out) { set_last_error("mmw_create: null argument"); return MMW_ERR_ARG; }
    *out = nullptr;
    const int S = cfg->n_samples, C = cfg->n_chirps, A = cfg->n_antennas;
    if (S < 4 || (S % 4) != 0) { set_last_error("n_samples must be a positive multiple of 4 (IIQQ packing + 16-byte rows), got %d", S); return MMW_ERR_ARG; }
    if (C < 2 || (C % 2) != 0) { set_last_error("n_chirps must be a positive multiple of 2, got %d", C); return MMW_ERR_ARG; }
    if (A < 1 || A > 256) { set_last_error("n_antennas must be 1..256, got %d", A); return MMW_ERR_ARG; }
    if (cfg->max_frames < 1) { set_last_error("max_frames must be >= 1"); return MMW_ERR_ARG; }
    const int Sp = next_pow2(S), Cp = next_pow2(C);
    const char *why = nullptr;
    if (!plan_supported(Sp, Cp, &why)) { set_last_error("unsupported shape: %s", why); return MMW_ERR_ARG; }
    const int Gr = cfg->cfar_guard_r, Gd = cfg->cfar_guard_d, Tr = cfg->cfar_train_r, Td = cfg->cfar_train_d;
    if (Gr < 0 || Gd < 0 || Tr < 0 || Td < 0 || Tr + Td == 0) { set_last_error("bad CFAR window"); return MMW_ERR_ARG; }
    if (2 * (Gd + Td) + 1 > Cp || Gr + Tr >= Sp || Gr + Tr > 64 || Gd + Td > 32) {
        set_last_error("CFAR window too large for a %dx%d map (limits: guard+train <= 64 range, <= 32 Doppler)", Sp, Cp);
        return MMW_ERR_ARG;
    }
    if (cfg->max_det_per_frame < 1 || cfg->max_det_per_frame > 65536) { set_last_error("max_det_per_frame must be 1..65536"); return MMW_ERR_ARG; }
    if ((long long)cfg->max_frames * cfg->max_det_per_frame > (1LL << 28)) { set_last_error("max_frames * max_det_per_frame must not exceed 2^28 records"); return MMW_ERR_ARG; }

    int dev = cfg->device;
    if (dev < 0) {
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) { set_last_error("no CUDA device: %s", cudaGetErrorString(e)); return MMW_ERR_CUDA; }
    }
    CK(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        set_last_error("this library is built for sm_100a (B200); device %d is sm_%d%d", dev, prop.major, prop.minor);
        return MMW_ERR_CUDA;
    }

    mmw_ctx *c = new mmw_ctx();
    memset(c, 0, sizeof(*c));
    c->cfg = *cfg;
    c->device = dev;
    c->sm_count = prop.multiProcessorCount;
    c->guard_on = env_int("MMW_GUARD") ? 1 : 0;
    c->guards = new std::vector<mmw_ctx::GuardedBuf>();
    int rc = MMW_OK;
    auto fail = [&](int code) { mmw_destroy(c); return code; };

    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { set_last_error("cudaStreamCreate failed"); return fail(MMW_ERR_CUDA); }
    c->stream = c->own_stream;
    for (auto &e : c->ev) if (cudaEventCreate(&e) != cudaSuccess) { set_last_error("cudaEventCreate failed"); return fail(MMW_ERR_CUDA); }

    const int F = cfg->max_frames;
    const int n_theta = A <= 64 ? 64 : next_pow2(A);
    const size_t N = (size_t)Sp * Cp * A, M = (size_t)Sp * Cp;

    if ((rc = dev_alloc(c, &c->d_win_r, (size_t)S))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_win_d, (size_t)C))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_tw1_r, (size_t)Sp))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_tw1_d, (size_t)Cp))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_tw_d, (size_t)Cp))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_tw_a, (size_t)n_theta))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_rs, (size_t)F * A * Sp * C))) return fail(rc);
    if (cfg->keep_doppler_cube && (rc = dev_alloc(c, &c->d_cube, (size_t)F * N))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_pmap, (size_t)F * M))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_mask, (size_t)F * M / 32))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_noise, (size_t)F * M))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_keys, (size_t)F * cfg->max_det_per_frame))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_counts, (size_t)F))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_offsets, (size_t)F + 1))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_ticket, (size_t)4))) return fail(rc);
    if ((rc = dev_alloc(c, &c->d_sched, (size_t)2))) return fail(rc);
    if (cudaMemset(c->d_sched, 0, 2 * sizeof(unsigned int)) != cudaSuccess) { set_last_error("cudaMemset failed"); return fail(MMW_ERR_CUDA); }
    if (cudaMemset(c->d_ticket, 0, 4 * sizeof(unsigned int)) != cudaSuccess) { set_last_error("cudaMemset failed"); return fail(MMW_ERR_CUDA); }
    c->dense_cap = F * cfg->max_det_per_frame;
    const size_t result_bytes = kResultHeaderBytes + (size_t)c->dense_cap * sizeof(mmw_detection);
    if ((rc = dev_alloc(c, &c->d_result, result_bytes))) return fail(rc);
    c->d_header = reinterpret_cast<uint32_t *>(c->d_result);
    c->d_dense = reinterpret_cast<mmw_detection *>(c->d_result + kResultHeaderBytes);
    c->guess_det = 4096;
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { set_last_error("cudaStreamCreate failed"); return fail(MMW_ERR_CUDA); }
    for (auto &e : c->chunk_ev) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { set_last_error("cudaEventCreate failed"); return fail(MMW_ERR_CUDA); }
    if (cudaMallocHost((void **)&c->h_result, result_bytes) == cudaSuccess) {
        c->h_header = reinterpret_cast<uint32_t *>(c->h_result);
        c->h_dense = reinterpret_cast<mmw_detection *>(c->h_result + kResultHeaderBytes);
    } else {
        set_last_error("cudaMallocHost failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(MMW_ERR_CUDA);
    }

    auto td = make_twiddles(Cp), ta = make_twiddles(n_theta);
    auto t1r = make_pass1_twiddles(Sp), t1d = make_pass1_twiddles(Cp);
    if (cudaMemcpy(c->d_tw1_r, t1r.data(), Sp * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(c->d_tw1_d, t1d.data(), Cp * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(c->d_tw_d, td.data(), Cp * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(c->d_tw_a, ta.data(), n_theta * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_last_error("twiddle upload failed");
        return fail(MMW_ERR_CUDA);
    }

    PlanDev &p = c->plan;
    p.S = S; p.C = C; p.A = A; p.Sp = Sp; p.Cp = Cp; p.n_theta = n_theta;
    p.guard_r = Gr; p.guard_d = Gd; p.win_r_half = Gr + Tr; p.win_d_half = Gd + Td;
    p.alpha = cfg->cfar_alpha; p.lambda_over_d = cfg->lambda_over_d;
    p.max_det = cfg->max_det_per_frame; p.keep_cube = cfg->keep_doppler_cube ? 1 : 0; p.frame_offset = 0;
    p.base_adc = nullptr;
    p.sched = c->d_sched;
    p.detect_path = MMW_DETECT_AUTO;
    p.win_r = c->d_win_r; p.win_d = c->d_win_d; p.tw_d = c->d_tw_d; p.tw_a = c->d_tw_a; p.tw1_r = c->d_tw1_r; p.tw1_d = c->d_tw1_d;

    // buffers of the selective re-FFT path if the plan takes it by default; they scale with the detection capacity — beyond
    // 2 GB the per-detection kernel is used instead.  Other plans get them when the caller picks that path (mmw_set_detect_path).
    if (detect_uses_refft(p, true) && (rc = alloc_refft_buffers(c))) return fail(rc);

    // antenna-split Doppler path of small batches (run_front): per-antenna power maps for the largest batch that still
    // prefers the split, if that stays modest.  Allocated here, never inside a batch: a batch may be under stream capture.
    if (A > 1 && !cfg->keep_doppler_cube && doppler_prefers_split(p, 1)) {
        int cap = 1;
        while (cap < F && doppler_prefers_split(p, cap + 1)) ++cap;
        if ((size_t)cap * A * M * sizeof(float) <= ((size_t)128 << 20)) {
            if ((rc = dev_alloc(c, &c->d_psplit, (size_t)cap * A * M))) return fail(rc);
            c->psplit_frames = cap;
        }
    }
    if ((rc = mmw_set_windows(c, nullptr, nullptr))) return fail(rc);
    *out = c;
    return MMW_OK;
}

int mmw_get_info(const mmw_ctx *c, mmw_info *info)
{
    if (!c || !info) { set_last_error("mmw_get_info: null argument"); return MMW_ERR_ARG; }
    const PlanDev &p = c->plan;
    info->Sp = p.Sp; info->Cp = p.Cp; info->n_theta = p.n_theta; info->sm_count = c->sm_count;
    info->adc_bytes_per_frame = 4LL * p.S * p.C * p.A;
    const long long N = (long long)p.Sp * p.Cp * p.A, M = (long long)p.Sp * p.Cp;
    info->algorithmic_bytes_per_frame = 28 * N + 8 * M;
    info->workspace_bytes = (long long)c->workspace_bytes;
    // K1, K2, K3, list, measure; the selective re-FFT path runs rows + extract + angle instead of measure
    info->kernels_per_batch = detect_uses_refft(p, c->d_rows != nullptr && c->d_snap != nullptr) ? 7 : 5;
    if (c->cluster_on) info->kernels_per_batch += kClusterKernels;
    return MMW_OK;
}

int mmw_set_windows(mmw_ctx *c, const float *win_range, const float *win_doppler)
{
    if (!c) { set_last_error("mmw_set_windows: null context"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    std::vector<float> wr = win_range ? std::vector<float>(win_range, win_range + c->plan.S) : make_hann(c->plan.S);
    std::vector<float> wd = win_doppler ? std::vector<float>(win_doppler, win_doppler + c->plan.C) : make_hann(c->plan.C);
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(c->d_win_r, wr.data(), wr.size() * sizeof(float), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_win_d, wd.data(), wd.size() * sizeof(float), cudaMemcpyHostToDevice));
    return MMW_OK;
}

int mmw_get_windows(const mmw_ctx *c, float *win_range, float *win_doppler)
{
    if (!c) { set_last_error("mmw_get_windows: null context"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    if (win_range) CK(cudaMemcpy(win_range, c->d_win_r, c->plan.S * sizeof(float), cudaMemcpyDeviceToHost));
    if (win_doppler) CK(cudaMemcpy(win_doppler, c->d_win_d, c->plan.C * sizeof(float), cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_set_frame_offset(mmw_ctx *c, uint32_t first_frame)
{
    if (!c) { set_last_error("mmw_set_frame_offset: null context"); return MMW_ERR_ARG; }
    c->plan.frame_offset = first_frame;
    return MMW_OK;
}

int mmw_set_base_frame(mmw_ctx *c, const int16_t *base_host)
{
    if (!c) { set_last_error("mmw_set_base_frame: null context"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    if (!base_host) { c->plan.base_adc = nullptr; return MMW_OK; }
    const size_t frame_shorts = (size_t)2 * c->plan.S * c->plan.C * c->plan.A;
    if (!c->d_base) {
        int rc = dev_alloc(c, &c->d_base, frame_shorts);
        if (rc) return rc;
    }
    CK(cudaMemcpy(c->d_base, base_host, frame_shorts * sizeof(int16_t), cudaMemcpyHostToDevice));
    c->plan.base_adc = c->d_base;
    return MMW_OK;
}

int mmw_set_graph_mode(mmw_ctx *c, int enable)
{
    if (!c) { set_last_error("mmw_set_graph_mode: null context"); return MMW_ERR_ARG; }
    c->graph_on = enable ? 1 : 0;
    return MMW_OK;
}

int mmw_set_detect_path(mmw_ctx *c, int path)
{
    if (!c) { set_last_error("mmw_set_detect_path: null context"); return MMW_ERR_ARG; }
    if (path != MMW_DETECT_AUTO && path != MMW_DETECT_PER_CELL && path != MMW_DETECT_REFFT) {
        set_last_error("mmw_set_detect_path: path must be MMW_DETECT_AUTO, _PER_CELL or _REFFT, got %d", path);
        return MMW_ERR_ARG;
    }
    if (c->submitted) { set_last_error("mmw_set_detect_path: a submitted batch is pending; collect it with mmw_wait"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    if (path == MMW_DETECT_REFFT) {
        CK(cudaStreamSynchronize(c->stream));
        int rc = alloc_refft_buffers(c);
        if (rc) return rc;
    }
    if (c->plan.detect_path != path && c->graphs) {     // the captured launch sequences belong to the old path
        CK(cudaStreamSynchronize(c->stream));
        destroy_graphs(c);
    }
    c->plan.detect_path = path;
    return MMW_OK;
}

void *mmw_stream(mmw_ctx *c) { return c ? (void *)c->stream : nullptr; }

int mmw_use_stream(mmw_ctx *c, void *cuda_stream)
{
    if (!c) { set_last_error("mmw_use_stream: null context"); return MMW_ERR_ARG; }
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return MMW_OK;
}

// stages 1-3 on frames [first, first + n) of the batch (they are per-frame independent)
static int run_front(mmw_ctx *c, const int16_t *adc_dev, int first, int n, cudaEvent_t *stage_ev)
{
    const PlanDev &p = c->plan;
    cudaStream_t st = c->stream;
    const size_t M = (size_t)p.Sp * p.Cp;
    const int16_t *adc = adc_dev + (size_t)first * 2 * p.S * p.C * p.A;
    float2 *rs = c->d_rs + (size_t)first * p.A * p.Sp * p.C;
    float2 *cube = p.keep_cube ? c->d_cube + (size_t)first * p.A * M : nullptr;
    if (stage_ev) CK(cudaEventRecord(stage_ev[0], st));
    const bool split = !cube && n <= c->psplit_frames && doppler_prefers_split(p, n);     // d_psplit: mmw_create
    CK(launch_range_fft(p, adc, rs, n, st));
    if (stage_ev) CK(cudaEventRecord(stage_ev[1], st));
    if (split) {
        PlanDev q = p;                                   // [F][A][Sp][C] read as F*A single-antenna frames
        q.A = 1;
        CK(launch_doppler_fft(q, rs, nullptr, c->d_psplit, n * p.A, st));
        CK(launch_power_sum(p, c->d_psplit, c->d_pmap + (size_t)first * M, n, st));
    } else {
        CK(launch_doppler_fft(p, rs, cube, c->d_pmap + (size_t)first * M, n, st));
    }
    if (stage_ev) CK(cudaEventRecord(stage_ev[2], st));
    CK(launch_cfar(p, c->d_pmap + (size_t)first * M, c->d_mask + (size_t)first * (M / 32), c->d_noise + (size_t)first * M, n, c->sm_count, st));
    if (stage_ev) CK(cudaEventRecord(stage_ev[3], st));
    return MMW_OK;
}

// stage 4 over the whole batch: ordered hit list, measurements, dense list + header
static int run_back(mmw_ctx *c, int n_frames, cudaEvent_t *stage_ev)
{
    const PlanDev &p = c->plan;
    DetectBuffers b;
    b.rs = c->d_rs; b.cube = c->d_cube; b.pmap = c->d_pmap; b.noise_map = c->d_noise; b.mask = c->d_mask;
    b.keys = c->d_keys; b.counts = c->d_counts; b.offsets = c->d_offsets; b.header = c->d_header;
    b.ticket = c->d_ticket; b.dense = c->d_dense; b.rows = c->d_rows; b.snap = c->d_snap;
    CK(launch_detect(p, b, n_frames, c->dense_cap, c->sm_count, c->stream));
    if (c->cluster_on) {
        ClusterBuffers cb;
        cb.dense = c->d_dense; cb.det_header = c->d_header; cb.keys = c->d_keys; cb.offsets = c->d_offsets;
        cb.parent = c->d_cl_parent; cb.size = c->d_cl_size; cb.oid = c->d_cl_oid; cb.cursor = c->d_cl_cursor;
        cb.members = c->d_cl_members; cb.labels = c->d_cl_labels; cb.frame_objs = c->d_cl_frame_objs;
        cb.obj_offsets = c->d_cl_obj_offsets; cb.slots = c->d_cl_slots; cb.ticket = c->d_cl_ticket;
        cb.obj_header = reinterpret_cast<uint32_t *>(c->d_objects);
        cb.objs = reinterpret_cast<mmw_object *>(c->d_objects + MMW_OBJECT_HEADER_BYTES);
        CK(launch_cluster(c->cluster, p.Cp, p.max_det, cb, n_frames, c->dense_cap, c->sm_count, c->stream));
    }
    if (stage_ev) CK(cudaEventRecord(stage_ev[4], c->stream));
    c->last_frames = n_frames;
    c->last_clustered = c->cluster_on;
    return MMW_OK;
}

static int run_batch(mmw_ctx *c, const int16_t *adc_dev, int n_frames, cudaEvent_t *stage_ev)
{
    int rc = run_front(c, adc_dev, 0, n_frames, stage_ev);
    if (rc) return rc;
    return run_back(c, n_frames, stage_ev);
}

// run_batch, or the replay of its captured graph when graph mode is on
static int run_batch_graphed(mmw_ctx *c, const int16_t *adc_dev, int n_frames)
{
    if (!c->graph_on) return run_batch(c, adc_dev, n_frames, nullptr);
    if (!c->graph_warm) {
        c->graph_warm = 1;
        return run_batch(c, adc_dev, n_frames, nullptr);
    }
    if (!c->graphs) c->graphs = new std::map<std::tuple<const void *, int, const void *, void *>, mmw_ctx::GraphEntry>();
    const auto key = std::make_tuple((const void *)adc_dev, n_frames, (const void *)c->plan.base_adc, (void *)c->stream);
    auto it = c->graphs->find(key);
    if (it == c->graphs->end()) {
        if (c->graphs->size() >= 256) destroy_graphs(c);      // bounded cache: start over rather than track recency
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = run_batch(c, adc_dev, n_frames, nullptr);
        const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        if (rc != MMW_OK || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            if (rc == MMW_OK) set_last_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
            return rc != MMW_OK ? rc : MMW_ERR_CUDA;
        }
        cudaGraphExec_t exec = nullptr;
        const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
        if (ei != cudaSuccess) {
            cudaGraphDestroy(graph);
            set_last_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ei));
            return MMW_ERR_CUDA;
        }
        mmw_ctx::GraphEntry ge{};
        ge.graph = graph; ge.exec = exec; ge.frame_offset = c->plan.frame_offset;
        // the node that writes mmw_detection.frame: the only consumer of PlanDev.frame_offset
        size_t n_nodes = 0;
        if (cudaGraphGetNodes(graph, nullptr, &n_nodes) == cudaSuccess && n_nodes > 0) {
            std::vector<cudaGraphNode_t> nodes(n_nodes);
            if (cudaGraphGetNodes(graph, nodes.data(), &n_nodes) == cudaSuccess)
                for (size_t i = 0; i < n_nodes; ++i) {
                    cudaGraphNodeType ty;
                    cudaKernelNodeParams kp;
                    if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
                    if (cudaGraphKernelNodeGetParams(nodes[i], &kp) != cudaSuccess) continue;
                    const int n_args = record_kernel_args(kp.func);
                    if (n_args > 0) { ge.record_node = nodes[i]; ge.record_kp = kp; ge.record_args = n_args; }
                }
        }
        cudaGetLastError();
        it = c->graphs->emplace(key, ge).first;
    }
    mmw_ctx::GraphEntry &ge = it->second;
    if (ge.frame_offset != c->plan.frame_offset) {
        if (!ge.record_node) { set_last_error("graph mode: record-writer node not found, cannot change the frame offset"); return MMW_ERR_STATE; }
        cudaKernelNodeParams kp = ge.record_kp;
        PlanDev patched = *reinterpret_cast<const PlanDev *>(kp.kernelParams[0]);       // argument 0 of both record kernels
        patched.frame_offset = c->plan.frame_offset;
        void *args[kRecordKernelMaxArgs];
        for (int i = 0; i < ge.record_args; ++i) args[i] = kp.kernelParams[i];
        args[0] = &patched;
        kp.kernelParams = args;
        CK(cudaGraphExecKernelNodeSetParams(ge.exec, ge.record_node, &kp));
        ge.frame_offset = c->plan.frame_offset;
    }
    CK(cudaGraphLaunch(ge.exec, c->stream));
    c->last_frames = n_frames;
    c->last_clustered = c->cluster_on;
    return MMW_OK;
}

static int check_batch_args(mmw_ctx *c, const void *adc, int n_frames, const char *who)
{
    if (!c || !adc) { set_last_error("%s: null argument", who); return MMW_ERR_ARG; }
    if (n_frames < 1 || n_frames > c->cfg.max_frames) {
        set_last_error("%s: n_frames %d outside 1..max_frames(%d)", who, n_frames, c->cfg.max_frames);
        return MMW_ERR_ARG;
    }
    if (c->submitted) {         // the context's buffers belong to the batch queued by mmw_submit_host until mmw_wait collects it
        set_last_error("%s: a batch submitted with mmw_submit_host has not been collected with mmw_wait", who);
        return MMW_ERR_STATE;
    }
    return MMW_OK;
}

// a misaligned or host pointer would fault inside the TMA copies of the first kernel and leave a sticky context error:
// refuse it up front
static int check_device_capture(const void *adc_dev, const char *who)
{
    if (((uintptr_t)adc_dev & 15u) != 0) { set_last_error("%s: adc_dev must be 16-byte aligned", who); return MMW_ERR_ARG; }
    cudaPointerAttributes at;
    const cudaError_t e = cudaPointerGetAttributes(&at, adc_dev);
    if (e != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        set_last_error("%s: adc_dev is not a device pointer (use mmw_process_host for host captures)", who);
        return MMW_ERR_ARG;
    }
    return MMW_OK;
}

int mmw_process_device(mmw_ctx *c, const int16_t *adc_dev, int n_frames)
{
    int rc = check_batch_args(c, adc_dev, n_frames, "mmw_process_device");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    if ((rc = check_device_capture(adc_dev, "mmw_process_device"))) return rc;
    return run_batch_graphed(c, adc_dev, n_frames);
}

// One D2H brings the header and the first `guess_det` records; a second copy is needed only when
// the batch produced more than that (the guess follows the previous batch).  Split in two so that a caller can
// queue a batch (enqueue_fetch) and collect it later (finish_fetch).
static int enqueue_fetch(mmw_ctx *c)
{
    const uint32_t guess = c->guess_det < (uint32_t)c->dense_cap ? c->guess_det : (uint32_t)c->dense_cap;
    c->fetched = guess;
    CK(cudaMemcpyAsync(c->h_result, c->d_result, kResultHeaderBytes + (size_t)guess * sizeof(mmw_detection), cudaMemcpyDeviceToHost, c->stream));
    return MMW_OK;
}

static int finish_fetch(mmw_ctx *c, mmw_detection *dets, int det_capacity, int *n_det)
{
    cudaStream_t st = c->stream;
    const uint32_t guess = c->fetched;
    CK(cudaStreamSynchronize(st));
    const uint32_t n_written = c->h_header[0];
    uint32_t n = n_written;
    int rc = c->h_header[3] ? MMW_ERR_OVERFLOW : MMW_OK;
    if ((int)n > det_capacity) { n = det_capacity > 0 ? (uint32_t)det_capacity : 0; rc = MMW_ERR_OVERFLOW; }
    if (n > guess) {
        CK(cudaMemcpyAsync(c->h_dense + guess, c->d_dense + guess, (size_t)(n - guess) * sizeof(mmw_detection), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    c->guess_det = n_written + n_written / 4 + 256;
    if (n > 0) {
        if (!dets) { set_last_error("detections pointer is null"); return MMW_ERR_ARG; }
        memcpy(dets, c->h_dense, (size_t)n * sizeof(mmw_detection));
    }
    if (n_det) *n_det = (int)n;
    if (rc == MMW_ERR_OVERFLOW)
        set_last_error("detection list truncated: %u of %u detections kept", n, c->h_header[1]);
    return rc;
}

static int fetch_results(mmw_ctx *c, mmw_detection *dets, int det_capacity, int *n_det)
{
    int rc = enqueue_fetch(c);
    if (rc) return rc;
    return finish_fetch(c, dets, det_capacity, n_det);
}

// Host capture -> device results, asynchronous.  The capture goes up in chunks on a copy stream; stages 1-3 of chunk k
// run while chunk k+1 is still on the bus (frames are independent), stage 4 runs once over the whole batch.
static int run_host_batch(mmw_ctx *c, const int16_t *adc_host, int n_frames)
{
    const size_t frame_shorts = (size_t)2 * c->plan.S * c->plan.C * c->plan.A;
    const size_t frame_bytes = frame_shorts * sizeof(int16_t);
    int rc;
    if (!c->d_adc) {            // staging for host captures, allocated on first use
        rc = dev_alloc(c, &c->d_adc, (size_t)c->cfg.max_frames * frame_shorts);
        if (rc) return rc;
    }
    int chunk = (int)((48u << 20) / frame_bytes);
    if (chunk < 1) chunk = 1;
    if (chunk * kMaxChunks < n_frames) chunk = (n_frames + kMaxChunks - 1) / kMaxChunks;
    if (c->graph_on && n_frames <= chunk) {
        // latency mode: one copy on the compute stream, then the whole launch sequence as one graph replay
        CK(cudaMemcpyAsync(c->d_adc, adc_host, (size_t)n_frames * frame_bytes, cudaMemcpyHostToDevice, c->stream));
        return run_batch_graphed(c, c->d_adc, n_frames);
    }
    int k = 0;
    for (int first = 0; first < n_frames; first += chunk, ++k) {
        const int n = n_frames - first < chunk ? n_frames - first : chunk;
        CK(cudaMemcpyAsync(c->d_adc + (size_t)first * frame_shorts, adc_host + (size_t)first * frame_shorts, (size_t)n * frame_bytes,
                           cudaMemcpyHostToDevice, c->copy_stream));
        CK(cudaEventRecord(c->chunk_ev[k], c->copy_stream));
        CK(cudaStreamWaitEvent(c->stream, c->chunk_ev[k], 0));
        rc = run_front(c, c->d_adc, first, n, nullptr);
        if (rc) return rc;
    }
    return run_back(c, n_frames, nullptr);
}

int mmw_process_host(mmw_ctx *c, const int16_t *adc_host, int n_frames, mmw_detection *dets, int det_capacity, int *n_det)
{
    int rc = mmw_submit_host(c, adc_host, n_frames);
    if (rc) return rc;
    return mmw_wait(c, dets, det_capacity, n_det);
}

int mmw_submit_host(mmw_ctx *c, const int16_t *adc_host, int n_frames)
{
    int rc = check_batch_args(c, adc_host, n_frames, "mmw_submit_host");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    rc = run_host_batch(c, adc_host, n_frames);
    if (rc) return rc;
    rc = enqueue_fetch(c);
    if (rc) return rc;
    c->submitted = 1;
    return MMW_OK;
}

int mmw_wait(mmw_ctx *c, mmw_detection *dets, int det_capacity, int *n_det)
{
    if (!c) { set_last_error("mmw_wait: null context"); return MMW_ERR_ARG; }
    if (!c->submitted) { set_last_error("mmw_wait: nothing submitted"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    c->submitted = 0;
    return finish_fetch(c, dets, det_capacity, n_det);
}

// ---------------------------------------------------------------------------
// capture-file ingest: fread into pinned double buffers, batch k+1 is read while batch k is on the GPU
// ---------------------------------------------------------------------------
int mmw_process_capture_file(mmw_ctx *c, const char *path, long long first_frame, int max_frames, int use_first_as_base,
                             mmw_detection *dets, int det_capacity, int *n_det, int *n_frames_done)
{
    if (n_det) *n_det = 0;
    if (n_frames_done) *n_frames_done = 0;
    if (!c || !path) { set_last_error("mmw_process_capture_file: null argument"); return MMW_ERR_ARG; }
    if (first_frame < 0 || det_capacity < 0 || (det_capacity > 0 && !dets)) { set_last_error("mmw_process_capture_file: bad argument"); return MMW_ERR_ARG; }
    if (c->submitted) { set_last_error("mmw_process_capture_file: a submitted batch is pending; collect it with mmw_wait"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    const size_t frame_shorts = (size_t)2 * c->plan.S * c->plan.C * c->plan.A;
    const size_t frame_bytes = frame_shorts * sizeof(int16_t);
    const int B = c->cfg.max_frames;
    FILE *fp = fopen(path, "rb");
    if (!fp) { set_last_error("unable to read the specified file: %s", path); return MMW_ERR_ARG; }    // the reference's message, cudaBenchMarking.cpp:346
    if (first_frame > 0 && fseeko(fp, (off_t)(first_frame * (long long)frame_bytes), SEEK_SET) != 0) {
        fclose(fp);
        set_last_error("mmw_process_capture_file: cannot seek to frame %lld", first_frame);
        return MMW_ERR_ARG;
    }
    for (auto &h : c->h_ring)
        if (!h && cudaMallocHost((void **)&h, (size_t)B * frame_bytes) != cudaSuccess) {
            fclose(fp);
            set_last_error("cudaMallocHost failed: %s", cudaGetErrorString(cudaGetLastError()));
            return MMW_ERR_CUDA;
        }
    // reads up to `want` frames into `dst`; a trailing partial frame is zero-filled and counted
    auto read_frames = [&](int16_t *dst, int want) -> int {
        if (want <= 0) return 0;
        const size_t got = fread(dst, sizeof(int16_t), (size_t)want * frame_shorts, fp);
        const size_t whole = got / frame_shorts, rest = got % frame_shorts;
        if (rest) {
            memset(dst + got, 0, (frame_shorts - rest) * sizeof(int16_t));
            return (int)whole + 1;
        }
        return (int)whole;
    };
    const uint32_t saved_offset = c->plan.frame_offset;
    long long frame_no = first_frame;           // file index of the next frame to be read
    long long budget = max_frames > 0 ? (long long)max_frames : -1;
    int rc = MMW_OK, total_det = 0, total_frames = 0, overflow = 0;
    if (use_first_as_base) {
        if (read_frames(c->h_ring[0], 1) == 1) {
            rc = mmw_set_base_frame(c, c->h_ring[0]);
            ++frame_no;
        }
    }
    int cur = 0;
    int n_cur = rc ? 0 : read_frames(c->h_ring[0 + cur], (int)(budget < 0 || budget > B ? B : budget));
    while (rc == MMW_OK && n_cur > 0) {
        if (budget > 0) budget -= n_cur;
        // queue batch `cur` (H2D chunks + kernels are asynchronous until fetch_results), then read the next batch
        // from the file while the GPU works
        c->plan.frame_offset = (uint32_t)frame_no;
        rc = run_host_batch(c, c->h_ring[cur], n_cur);
        const int want_next = budget == 0 ? 0 : (int)(budget < 0 || budget > B ? B : budget);
        const int n_next = rc == MMW_OK ? read_frames(c->h_ring[cur ^ 1], want_next) : 0;      // overlaps the GPU work above
        if (rc == MMW_OK) {
            int got = 0;
            rc = fetch_results(c, dets ? dets + total_det : nullptr, det_capacity - total_det, &got);
            if (rc == MMW_ERR_OVERFLOW) { overflow = 1; rc = MMW_OK; }
            total_det += got;
            total_frames += n_cur;
            frame_no += n_cur;
        }
        cur ^= 1;
        n_cur = n_next;
    }
    fclose(fp);
    c->plan.frame_offset = saved_offset;
    if (n_det) *n_det = total_det;
    if (n_frames_done) *n_frames_done = total_frames;
    if (rc == MMW_OK && overflow) {
        set_last_error("detection list truncated while reading %s", path);
        return MMW_ERR_OVERFLOW;
    }
    return rc;
}

// ---------------------------------------------------------------------------
// detections -> physical units (host arithmetic, mirrors cudaBenchMarking.cpp:10-19 and :301-303)
// ---------------------------------------------------------------------------
void mmw_default_radar_params(mmw_radar_params *rp)
{
    if (!rp) return;
    rp->f0_hz = 77e9;
    rp->slope_hz_per_s = 5.987e12;
    rp->fs_hz = 2.0e6;
    rp->chirp_period_s = 64e-6;
    rp->light_speed = 3.0e8;
}

// the bin -> metre and bin -> m/s formulas of mmw_to_physical and mmw_objects_to_physical (a fractional bin takes the same
// expression; an integer bin converts to double exactly)
static float range_bin_to_m(const mmw_radar_params *rp, int Sp, double range_bin)
{
    const double f_beat = range_bin / (double)Sp * rp->fs_hz;
    return (float)(rp->light_speed * f_beat / (2.0 * rp->slope_hz_per_s));
}

static float doppler_bin_to_mps(const mmw_radar_params *rp, int Cp, double signed_doppler_bin)
{
    const double lambda = rp->light_speed / rp->f0_hz;
    const double f_dop = signed_doppler_bin / ((double)Cp * rp->chirp_period_s);
    return (float)(0.5 * lambda * f_dop);
}

static int check_radar_params(const mmw_radar_params *rp, int Sp, int Cp, int n, const void *in, const void *out, const char *who)
{
    if (!rp || Sp < 1 || Cp < 1 || n < 0 || (n > 0 && (!in || !out))) { set_last_error("%s: bad argument", who); return MMW_ERR_ARG; }
    if (rp->f0_hz <= 0 || rp->slope_hz_per_s <= 0 || rp->fs_hz <= 0 || rp->chirp_period_s <= 0 || rp->light_speed <= 0) {
        set_last_error("%s: radar parameters must be positive", who);
        return MMW_ERR_ARG;
    }
    return MMW_OK;
}

int mmw_to_physical(const mmw_radar_params *rp, int Sp, int Cp, const mmw_detection *dets, int n, mmw_target *out)
{
    const int rc = check_radar_params(rp, Sp, Cp, n, dets, out, "mmw_to_physical");
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        const mmw_detection &d = dets[i];
        const int dw = d.doppler_bin < Cp / 2 ? (int)d.doppler_bin : (int)d.doppler_bin - Cp;
        mmw_target &t = out[i];
        t.frame = d.frame;
        t.range_m = range_bin_to_m(rp, Sp, (double)d.range_bin);
        t.velocity_mps = doppler_bin_to_mps(rp, Cp, (double)dw);
        t.angle_deg = (float)((double)d.angle_rad * (180.0 / M_PI));
        t.snr_db = (d.noise > 0.f && d.power > 0.f) ? (float)(10.0 * log10((double)d.power / (double)d.noise)) : 0.f;
        t.flags = d.flags;
    }
    return MMW_OK;
}

int mmw_objects_to_physical(const mmw_radar_params *rp, int Sp, int Cp, const mmw_object *objs, int n, mmw_target *out)
{
    const int rc = check_radar_params(rp, Sp, Cp, n, objs, out, "mmw_objects_to_physical");
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        const mmw_object &o = objs[i];
        mmw_target &t = out[i];
        t.frame = o.frame;
        t.range_m = range_bin_to_m(rp, Sp, (double)o.range_bin);
        t.velocity_mps = doppler_bin_to_mps(rp, Cp, (double)o.doppler_bin);
        t.angle_deg = (float)((double)o.angle_rad * (180.0 / M_PI));
        t.snr_db = (o.peak_noise > 0.f && o.peak_power > 0.f) ? (float)(10.0 * log10((double)o.peak_power / (double)o.peak_noise)) : 0.f;
        t.flags = 0;
    }
    return MMW_OK;
}

// ---------------------------------------------------------------------------
// clustering of each frame's detections into objects (kernels: mmw_cluster.cu)
// ---------------------------------------------------------------------------
void mmw_default_cluster_params(mmw_cluster_params *cp)
{
    if (!cp) return;
    cp->eps_range = 2;
    cp->eps_doppler = 2;
    cp->eps_angle = 4;
    cp->min_points = 1;
    cp->max_objects_per_frame = 256;
}

int mmw_set_clustering(mmw_ctx *c, const mmw_cluster_params *cp)
{
    if (!c) { set_last_error("mmw_set_clustering: null context"); return MMW_ERR_ARG; }
    if (cp) {
        if (cp->eps_range < 0 || cp->eps_range > 16) { set_last_error("mmw_set_clustering: eps_range must be 0..16, got %d", cp->eps_range); return MMW_ERR_ARG; }
        if (cp->eps_doppler < 0 || cp->eps_doppler > 16) { set_last_error("mmw_set_clustering: eps_doppler must be 0..16, got %d", cp->eps_doppler); return MMW_ERR_ARG; }
        if (cp->eps_angle < 0) { set_last_error("mmw_set_clustering: eps_angle must be >= 0, got %d", cp->eps_angle); return MMW_ERR_ARG; }
        if (cp->min_points < 1) { set_last_error("mmw_set_clustering: min_points must be >= 1, got %d", cp->min_points); return MMW_ERR_ARG; }
        if (cp->max_objects_per_frame < 1 || cp->max_objects_per_frame > c->cfg.max_det_per_frame) {
            set_last_error("mmw_set_clustering: max_objects_per_frame must be 1..max_det_per_frame (%d), got %d", c->cfg.max_det_per_frame,
                           cp->max_objects_per_frame);
            return MMW_ERR_ARG;
        }
    }
    if (c->submitted) { set_last_error("mmw_set_clustering: a submitted batch is pending; collect it with mmw_wait"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));               // a batch in flight may still use the buffers
    if (c->graphs) destroy_graphs(c);                  // the captured launch sequences belong to the old setting
    const bool same_capacity = cp && c->cluster_on && c->cluster.max_objects_per_frame == cp->max_objects_per_frame;
    if (!same_capacity) {
        free_cluster_buffers(c);
        c->cluster_on = 0;
        c->last_clustered = 0;
    }
    if (!cp) return MMW_OK;
    if (!same_capacity) {
        const size_t D = (size_t)c->dense_cap, F = (size_t)c->cfg.max_frames;
        const size_t obj_cap = F * (size_t)cp->max_objects_per_frame;
        const size_t before = c->workspace_bytes;
        int rc;
        if ((rc = dev_alloc(c, &c->d_cl_parent, D)) || (rc = dev_alloc(c, &c->d_cl_size, D)) || (rc = dev_alloc(c, &c->d_cl_oid, D)) ||
            (rc = dev_alloc(c, &c->d_cl_cursor, D)) || (rc = dev_alloc(c, &c->d_cl_members, D)) || (rc = dev_alloc(c, &c->d_cl_labels, D)) ||
            (rc = dev_alloc(c, &c->d_cl_frame_objs, 2 * F)) || (rc = dev_alloc(c, &c->d_cl_obj_offsets, F + 1)) ||
            (rc = dev_alloc(c, &c->d_cl_slots, obj_cap)) || (rc = dev_alloc(c, &c->d_cl_ticket, (size_t)1)) ||
            (rc = dev_alloc(c, &c->d_objects, (size_t)MMW_OBJECT_HEADER_BYTES + obj_cap * sizeof(mmw_object)))) {
            c->cluster_bytes = c->workspace_bytes - before;
            free_cluster_buffers(c);
            return rc;
        }
        c->cluster_bytes = c->workspace_bytes - before;
        // the ticket self-resets after every batch; the header reads "no objects" until the first clustered batch
        CK(cudaMemset(c->d_cl_ticket, 0, sizeof(unsigned int)));
        CK(cudaMemset(c->d_objects, 0, MMW_OBJECT_HEADER_BYTES));
    }
    c->cluster = *cp;
    c->cluster_on = 1;
    return MMW_OK;
}

static int check_clustered(mmw_ctx *c, const char *who)
{
    if (!c) { set_last_error("%s: null context", who); return MMW_ERR_ARG; }
    if (c->submitted) { set_last_error("%s: a submitted batch is pending; collect it with mmw_wait", who); return MMW_ERR_STATE; }
    if (!c->cluster_on || !c->last_clustered || c->last_frames <= 0) {
        set_last_error("%s: the last batch was not clustered (mmw_set_clustering)", who);
        return MMW_ERR_STATE;
    }
    return MMW_OK;
}

int mmw_read_objects(mmw_ctx *c, mmw_object *objs, int capacity, int *n_obj)
{
    int rc = check_clustered(c, "mmw_read_objects");
    if (rc) return rc;
    if (capacity < 0 || (capacity > 0 && !objs)) { set_last_error("mmw_read_objects: bad capacity / null output"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    uint32_t hdr[MMW_OBJECT_HEADER_BYTES / 4];
    CK(cudaMemcpyAsync(hdr, c->d_objects, sizeof(hdr), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    uint32_t n = hdr[0];
    rc = hdr[3] ? MMW_ERR_OVERFLOW : MMW_OK;
    if ((long long)n > (long long)capacity) { n = (uint32_t)capacity; rc = MMW_ERR_OVERFLOW; }
    if (n > 0) {
        CK(cudaMemcpyAsync(objs, c->d_objects + MMW_OBJECT_HEADER_BYTES, (size_t)n * sizeof(mmw_object), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    if (n_obj) *n_obj = (int)n;
    if (rc == MMW_ERR_OVERFLOW)
        set_last_error("object list incomplete: %u of %u objects kept (flags 0x%x)", n, hdr[1], hdr[3]);
    return rc;
}

int mmw_read_labels(mmw_ctx *c, int32_t *labels, int capacity, int *n)
{
    int rc = check_clustered(c, "mmw_read_labels");
    if (rc) return rc;
    if (capacity < 0 || (capacity > 0 && !labels)) { set_last_error("mmw_read_labels: bad capacity / null output"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    uint32_t n_written = 0;
    CK(cudaMemcpyAsync(&n_written, c->d_header, sizeof(n_written), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    uint32_t k = n_written;
    rc = MMW_OK;
    if ((long long)k > (long long)capacity) { k = (uint32_t)capacity; rc = MMW_ERR_OVERFLOW; }
    if (k > 0) {
        CK(cudaMemcpyAsync(labels, c->d_cl_labels, (size_t)k * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    if (n) *n = (int)k;
    if (rc == MMW_ERR_OVERFLOW) set_last_error("mmw_read_labels: %u labels, capacity %d", n_written, capacity);
    return rc;
}

int mmw_device_objects(mmw_ctx *c, const mmw_object **objs, const uint32_t **header)
{
    if (!c) { set_last_error("mmw_device_objects: null context"); return MMW_ERR_ARG; }
    if (!c->cluster_on) { set_last_error("mmw_device_objects: clustering is off (mmw_set_clustering)"); return MMW_ERR_STATE; }
    if (objs) *objs = reinterpret_cast<const mmw_object *>(c->d_objects + MMW_OBJECT_HEADER_BYTES);
    if (header) *header = reinterpret_cast<const uint32_t *>(c->d_objects);
    return MMW_OK;
}

int mmw_read_detections(mmw_ctx *c, mmw_detection *dets, int det_capacity, int *n_det)
{
    if (!c) { set_last_error("mmw_read_detections: null context"); return MMW_ERR_ARG; }
    if (c->last_frames <= 0) { set_last_error("mmw_read_detections: no batch processed"); return MMW_ERR_STATE; }
    if (c->submitted) { set_last_error("mmw_read_detections: a submitted batch is pending; collect it with mmw_wait"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    return fetch_results(c, dets, det_capacity, n_det);
}

int mmw_read_counts(mmw_ctx *c, uint32_t *counts, int n_frames)
{
    if (!c || !counts) { set_last_error("mmw_read_counts: null argument"); return MMW_ERR_ARG; }
    if (n_frames < 1 || n_frames > c->last_frames) { set_last_error("mmw_read_counts: n_frames outside the last batch"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(counts, c->d_counts, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return MMW_OK;
}

int mmw_device_results(mmw_ctx *c, const mmw_detection **dense_dets, const uint32_t **header)
{
    if (!c) { set_last_error("mmw_device_results: null context"); return MMW_ERR_ARG; }
    if (dense_dets) *dense_dets = c->d_dense;
    if (header) *header = c->d_header;
    return MMW_OK;
}

int mmw_device_result_block(mmw_ctx *c, const void **block, long long *capacity_bytes)
{
    if (!c) { set_last_error("mmw_device_result_block: null context"); return MMW_ERR_ARG; }
    if (block) *block = c->d_result;
    if (capacity_bytes) *capacity_bytes = kResultHeaderBytes + (long long)c->dense_cap * (long long)sizeof(mmw_detection);
    return MMW_OK;
}

int mmw_merge_gathered(mmw_ctx *c, const void *gathered_dev, int n_ranks, long long stride_bytes, void *merged_dev, int merged_capacity)
{
    if (!c || !gathered_dev || !merged_dev) { set_last_error("mmw_merge_gathered: null argument"); return MMW_ERR_ARG; }
    if (n_ranks < 1 || stride_bytes < kResultHeaderBytes || (stride_bytes % 8) != 0 || merged_capacity < 0) {
        set_last_error("mmw_merge_gathered: bad rank count / stride / capacity");
        return MMW_ERR_ARG;
    }
    CK(cudaSetDevice(c->device));
    CK(launch_merge((const unsigned char *)gathered_dev, n_ranks, (size_t)stride_bytes, (unsigned char *)merged_dev, merged_capacity, c->stream));
    return MMW_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// Peer exchange: the gather of the detection lists of a frame-sharded job (one process per GPU) WITHOUT a kernel.
// ---------------------------------------------------------------------------------------------------------------
// The FFT kernels are persistent and fill every SM's register file, so any kernel of another stream — NCCL's send/recv
// kernel included — waits for an FFT CTA to retire, then holds that slot while it waits for its peers, and the next FFT
// kernel starts short of CTAs: measured +11 us per 0.40 ms step at 2 GPUs and +33 us at 8 for the NCCL gather
// (profiles/r2/exchange.md).  Here every rank PUTS its result block straight into rank 0's memory with the copy engine
// (cudaMemcpyAsync to a cudaIpc-mapped peer pointer: NVLink, no SM) and raises a flag in rank 0's memory with a stream
// memory operation (cuStreamWriteValue32); rank 0's side stream waits for the flags (cuStreamWaitValue32) and runs the one
// merge kernel; a credit written back the same way keeps a rank from overwriting a slot that is still being merged.
// Set-up (exchange of the IPC handles) goes through whatever the launcher has — torch.distributed / NCCL in bench.py.
typedef unsigned int (*StreamValueFn)(cudaStream_t, unsigned long long, unsigned int, unsigned int);   // CUresult f(CUstream, CUdeviceptr, value, flags)

struct mmw_exchange {
    mmw_ctx *ctx;
    int device;
    int rank, n_ranks, depth;
    long long stride;                 // bytes one rank contributes per step: header + records_per_rank records
    int merged_cap;
    // rank 0 owns: [depth][n_ranks][stride] gathered blocks, then n_ranks arrival counters (one allocation = one IPC handle)
    unsigned char *gathered;          // rank 0: own allocation; others: mapped
    unsigned int *arrival;            // inside the same allocation
    unsigned char *merged[2];         // rank 0
    unsigned int *credit;             // this rank's credit word (own allocation; rank 0 maps every rank's)
    unsigned int *peer_credit[kMaxDevices];   // rank 0: mapped credit words of the other ranks
    void *mapped_root;                // non-root: base of the mapped rank-0 allocation
    cudaStream_t side;                // rank 0: wait + merge + credits
    cudaEvent_t merged_ev[2];
    unsigned int step;                // puts issued
    unsigned int merges;              // merges issued (rank 0)
    StreamValueFn wait_value, write_value;
    int connected;
};

static size_t exchange_root_bytes(const mmw_exchange *x)
{
    return (size_t)x->depth * x->n_ranks * (size_t)x->stride + (size_t)kMaxDevices * sizeof(unsigned int);
}

extern "C" {

void mmw_exchange_destroy(mmw_exchange *x)
{
    if (!x) return;
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();                                          // (the context may already be gone: nothing of it is touched here)
    if (x->rank == 0) {
        for (int r = 1; r < x->n_ranks; ++r) if (x->peer_credit[r]) cudaIpcCloseMemHandle(x->peer_credit[r]);
        cudaFree(x->gathered);
        cudaFree(x->merged[0]); cudaFree(x->merged[1]);
    } else if (x->mapped_root) {
        cudaIpcCloseMemHandle(x->mapped_root);
    }
    cudaFree(x->credit);
    for (auto &e : x->merged_ev) if (e) cudaEventDestroy(e);
    if (x->side) cudaStreamDestroy(x->side);
    delete x;
}

int mmw_exchange_create(mmw_ctx *c, int rank, int n_ranks, int records_per_rank, int depth, mmw_exchange **out)
{
    if (!c || !out) { set_last_error("mmw_exchange_create: null argument"); return MMW_ERR_ARG; }
    *out = nullptr;
    if (n_ranks < 1 || n_ranks > kMaxDevices || rank < 0 || rank >= n_ranks || depth < 2 || depth > 64 || records_per_rank < 1 ||
        records_per_rank > c->dense_cap) {
        set_last_error("mmw_exchange_create: bad rank / rank count / depth / records_per_rank");
        return MMW_ERR_ARG;
    }
    CK(cudaSetDevice(c->device));
    mmw_exchange *x = new mmw_exchange();
    memset(x, 0, sizeof(*x));
    x->ctx = c; x->device = c->device; x->rank = rank; x->n_ranks = n_ranks; x->depth = depth;
    x->stride = kResultHeaderBytes + (long long)records_per_rank * (long long)sizeof(mmw_detection);
    x->merged_cap = n_ranks * records_per_rank;
    auto fail = [&](const char *what) { set_last_error("mmw_exchange_create: %s: %s", what, cudaGetErrorString(cudaGetLastError())); mmw_exchange_destroy(x); return MMW_ERR_CUDA; };
    cudaDriverEntryPointQueryResult q;
    void *fw = nullptr, *fs = nullptr;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fw, cudaEnableDefault, &q) != cudaSuccess || !fw ||
        cudaGetDriverEntryPoint("cuStreamWriteValue32", &fs, cudaEnableDefault, &q) != cudaSuccess || !fs)
        return fail("stream memory operations are not available");
    x->wait_value = (StreamValueFn)fw; x->write_value = (StreamValueFn)fs;
    if (cudaMalloc((void **)&x->credit, 256) != cudaSuccess || cudaMemset(x->credit, 0, 256) != cudaSuccess) return fail("cudaMalloc");
    if (rank == 0) {
        const size_t bytes = exchange_root_bytes(x);
        if (cudaMalloc((void **)&x->gathered, bytes) != cudaSuccess || cudaMemset(x->gathered, 0, bytes) != cudaSuccess) return fail("cudaMalloc");
        x->arrival = reinterpret_cast<unsigned int *>(x->gathered + (size_t)depth * n_ranks * (size_t)x->stride);
        const size_t mbytes = kResultHeaderBytes + (size_t)x->merged_cap * sizeof(mmw_detection);
        for (auto &m : x->merged) if (cudaMalloc((void **)&m, mbytes) != cudaSuccess || cudaMemset(m, 0, mbytes) != cudaSuccess) return fail("cudaMalloc");
        if (cudaStreamCreateWithFlags(&x->side, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate");
        for (auto &e : x->merged_ev) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return fail("cudaEventCreate");
    }
    CK(cudaDeviceSynchronize());
    *out = x;
    return MMW_OK;
}

/* 64 bytes: rank 0 -> the IPC handle of its gathered block; every other rank -> the IPC handle of its credit word */
int mmw_exchange_handle(mmw_exchange *x, void *handle64)
{
    if (!x || !handle64) { set_last_error("mmw_exchange_handle: null argument"); return MMW_ERR_ARG; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, x->rank == 0 ? (void *)x->gathered : (void *)x->credit));
    memcpy(handle64, &h, sizeof(h));
    return MMW_OK;
}

/* all_handles: n_ranks x 64 bytes, entry r = what rank r's mmw_exchange_handle returned */
int mmw_exchange_connect(mmw_exchange *x, const void *all_handles)
{
    if (!x || !all_handles) { set_last_error("mmw_exchange_connect: null argument"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(x->ctx->device));
    const cudaIpcMemHandle_t *h = static_cast<const cudaIpcMemHandle_t *>(all_handles);
    if (x->rank == 0) {
        for (int r = 1; r < x->n_ranks; ++r) {
            void *p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, h[r], cudaIpcMemLazyEnablePeerAccess));
            x->peer_credit[r] = static_cast<unsigned int *>(p);
        }
    } else {
        CK(cudaIpcOpenMemHandle(&x->mapped_root, h[0], cudaIpcMemLazyEnablePeerAccess));
        x->gathered = static_cast<unsigned char *>(x->mapped_root);
        x->arrival = reinterpret_cast<unsigned int *>(x->gathered + (size_t)x->depth * x->n_ranks * (size_t)x->stride);
    }
    x->connected = 1;
    return MMW_OK;
}

/* After mmw_process_device, on the context's stream: this rank's result block goes to its slot of step `step` in rank 0's
 * memory, then the arrival flag.  No kernel.  Blocks (on the stream, not the host) only if rank 0 is `depth` steps behind. */
int mmw_exchange_put(mmw_exchange *x)
{
    if (!x || !x->connected) { set_last_error("mmw_exchange_put: not connected"); return MMW_ERR_STATE; }
    mmw_ctx *c = x->ctx;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const unsigned int s = x->step++;
    const int slot = (int)(s % (unsigned int)x->depth);
    if (s >= (unsigned int)x->depth) {
        // the slot was last used by step s - depth: rank 0 has merged it once the credit reads s - depth + 1
        if (x->wait_value(st, (unsigned long long)(uintptr_t)x->credit, s - (unsigned int)x->depth + 1u, 0u /* GEQ */) != 0) {
            set_last_error("mmw_exchange_put: cuStreamWaitValue32 failed");
            return MMW_ERR_CUDA;
        }
    }
    unsigned char *dst = x->gathered + ((size_t)slot * x->n_ranks + x->rank) * (size_t)x->stride;
    CK(cudaMemcpyAsync(dst, c->d_result, (size_t)x->stride, cudaMemcpyDeviceToDevice, st));
    if (x->write_value(st, (unsigned long long)(uintptr_t)(x->arrival + x->rank), s + 1u, 0u) != 0) {
        set_last_error("mmw_exchange_put: cuStreamWriteValue32 failed");
        return MMW_ERR_CUDA;
    }
    return MMW_OK;
}

/* Rank 0, once per step after its own put: the side stream waits for every rank's flag of that step, merges the blocks
 * into one ordered list (one kernel), and hands the slot back.  Returns the merged block (device pointer; complete when the
 * side stream gets there: mmw_exchange_wait makes a stream wait for it). */
int mmw_exchange_merge(mmw_exchange *x, const void **merged_block)
{
    if (!x || !x->connected || x->rank != 0) { set_last_error("mmw_exchange_merge: rank 0 only, after connect"); return MMW_ERR_STATE; }
    mmw_ctx *c = x->ctx;
    CK(cudaSetDevice(c->device));
    const unsigned int m = x->merges++;
    if (m >= x->step) { x->merges--; set_last_error("mmw_exchange_merge: no put for this step yet"); return MMW_ERR_STATE; }
    const int slot = (int)(m % (unsigned int)x->depth), k = (int)(m & 1u);
    for (int r = 0; r < x->n_ranks; ++r)
        if (x->wait_value(x->side, (unsigned long long)(uintptr_t)(x->arrival + r), m + 1u, 0u) != 0) { set_last_error("cuStreamWaitValue32 failed"); return MMW_ERR_CUDA; }
    CK(launch_merge(x->gathered + (size_t)slot * x->n_ranks * (size_t)x->stride, x->n_ranks, (size_t)x->stride, x->merged[k], x->merged_cap, x->side));
    CK(cudaEventRecord(x->merged_ev[k], x->side));
    for (int r = 0; r < x->n_ranks; ++r) {
        unsigned int *cr = r == 0 ? x->credit : x->peer_credit[r];
        if (x->write_value(x->side, (unsigned long long)(uintptr_t)cr, m + 1u, 0u) != 0) { set_last_error("cuStreamWriteValue32 failed"); return MMW_ERR_CUDA; }
    }
    if (merged_block) *merged_block = x->merged[k];
    return MMW_OK;
}

/* Rank 0: `cuda_stream` (nullptr: the context's stream) waits for the last merge issued; *merged_block is that block. */
int mmw_exchange_wait(mmw_exchange *x, void *cuda_stream, const void **merged_block)
{
    if (!x || x->rank != 0 || x->merges == 0) { set_last_error("mmw_exchange_wait: rank 0 only, after a merge"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(x->ctx->device));
    const int k = (int)((x->merges - 1u) & 1u);
    CK(cudaStreamWaitEvent(cuda_stream ? (cudaStream_t)cuda_stream : x->ctx->stream, x->merged_ev[k], 0));
    if (merged_block) *merged_block = x->merged[k];
    return MMW_OK;
}

}  // extern "C"

extern "C" {

static int ensure_scratch(mmw_ctx *c, size_t bytes)
{
    if (bytes <= c->scratch_bytes) return MMW_OK;
    if (c->d_scratch) cudaFree(c->d_scratch);
    c->d_scratch = nullptr;
    c->scratch_bytes = 0;
    CK(cudaMalloc(&c->d_scratch, bytes));
    c->scratch_bytes = bytes;
    return MMW_OK;
}

static int check_frame(mmw_ctx *c, int frame, const void *out, const char *who)
{
    if (!c || !out) { set_last_error("%s: null argument", who); return MMW_ERR_ARG; }
    if (frame < 0 || frame >= c->last_frames) { set_last_error("%s: frame %d not in the last batch (%d frames)", who, frame, c->last_frames); return MMW_ERR_STATE; }
    return MMW_OK;
}

int mmw_copy_range_spectrum(mmw_ctx *c, int frame, float *out)
{
    int rc = check_frame(c, frame, out, "mmw_copy_range_spectrum");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    const PlanDev &p = c->plan;
    const size_t n = (size_t)p.A * p.Sp * p.C;
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(out, c->d_rs + (size_t)frame * n, n * sizeof(float2), cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_copy_doppler_cube(mmw_ctx *c, int frame, float *out)
{
    int rc = check_frame(c, frame, out, "mmw_copy_doppler_cube");
    if (rc) return rc;
    if (!c->plan.keep_cube) { set_last_error("mmw_copy_doppler_cube: context was created with keep_doppler_cube = 0"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    const PlanDev &p = c->plan;
    const size_t n = (size_t)p.A * p.Sp * p.Cp;
    if ((rc = ensure_scratch(c, n * sizeof(float2)))) return rc;
    CK(launch_export_cube(p, c->d_cube + (size_t)frame * n, (float2 *)c->d_scratch, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(out, c->d_scratch, n * sizeof(float2), cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_copy_power_map(mmw_ctx *c, int frame, float *out)
{
    int rc = check_frame(c, frame, out, "mmw_copy_power_map");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    const PlanDev &p = c->plan;
    const size_t n = (size_t)p.Sp * p.Cp;
    if ((rc = ensure_scratch(c, n * sizeof(float)))) return rc;
    CK(launch_export_pmap(p, c->d_pmap + (size_t)frame * n, (float *)c->d_scratch, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(out, c->d_scratch, n * sizeof(float), cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_copy_cfar_mask(mmw_ctx *c, int frame, uint8_t *out)
{
    int rc = check_frame(c, frame, out, "mmw_copy_cfar_mask");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    const PlanDev &p = c->plan;
    const size_t n = (size_t)p.Sp * p.Cp;
    if ((rc = ensure_scratch(c, n))) return rc;
    CK(launch_export_mask(p, c->d_mask + (size_t)frame * (n / 32), (uint8_t *)c->d_scratch, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(out, c->d_scratch, n, cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_check_guards(mmw_ctx *c, long long *bad_bytes)
{
    if (!c || !bad_bytes) { set_last_error("mmw_check_guards: null argument"); return MMW_ERR_ARG; }
    *bad_bytes = 0;
    if (!c->guard_on) { set_last_error("mmw_check_guards: the context was not created with MMW_GUARD=1"); return MMW_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    std::vector<unsigned char> h(2 * kGuardBytes);
    long long bad = 0;
    char first[160] = "";
    for (const auto &g : *c->guards) {
        CK(cudaMemcpy(h.data(), g.base, kGuardBytes, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(h.data() + kGuardBytes, g.base + kGuardBytes + g.bytes, kGuardBytes, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < 2 * kGuardBytes; ++i)
            if (h[i] != (unsigned char)kGuardByte) {
                if (!bad)
                    snprintf(first, sizeof first, "%s (%zu bytes): byte %lld %s", g.name, g.bytes,
                             i < kGuardBytes ? (long long)kGuardBytes - (long long)i : (long long)(i - kGuardBytes),
                             i < kGuardBytes ? "before its start" : "past its end");
                ++bad;
            }
    }
    *bad_bytes = bad;
    if (bad) set_last_error("mmw_check_guards: %lld guard bytes overwritten; first: %s", bad, first);
    return MMW_OK;
}

int mmw_time_device(mmw_ctx *c, const int16_t *adc_dev, int n_frames, int iters, float *total_ms, float *per_stage_ms)
{
    int rc = check_batch_args(c, adc_dev, n_frames, "mmw_time_device");
    if (rc) return rc;
    if (iters < 1 || !total_ms) { set_last_error("mmw_time_device: bad iters / null output"); return MMW_ERR_ARG; }
    CK(cudaSetDevice(c->device));
    if ((rc = check_device_capture(adc_dev, "mmw_time_device"))) return rc;
    cudaStream_t st = c->stream;
    if (per_stage_ms) {
        // separate instrumented pass: events between launches serialise the stages
        float acc[4] = {0, 0, 0, 0};
        for (int i = 0; i < iters; ++i) {
            rc = run_batch(c, adc_dev, n_frames, c->ev);
            if (rc) return rc;
            CK(cudaStreamSynchronize(st));
            for (int s = 0; s < 4; ++s) {
                float ms = 0;
                CK(cudaEventElapsedTime(&ms, c->ev[s], c->ev[s + 1]));
                acc[s] += ms;
            }
        }
        for (int s = 0; s < 4; ++s) per_stage_ms[s] = acc[s];
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaEventRecord(c->ev[0], st));
    for (int i = 0; i < iters; ++i) {
        rc = run_batch(c, adc_dev, n_frames, nullptr);
        if (rc) return rc;
    }
    CK(cudaEventRecord(c->ev[5], st));
    CK(cudaEventSynchronize(c->ev[5]));
    CK(cudaEventElapsedTime(total_ms, c->ev[0], c->ev[5]));
    return MMW_OK;
}

// ---------------------------------------------------------------------------
// multi-GPU group: frame shards on the GPUs of one process, detection lists gathered to GPU 0 over NCCL
// ---------------------------------------------------------------------------
struct NcclApi {
    void *handle;
    decltype(&ncclGetUniqueId) GetUniqueId;
    decltype(&ncclCommInitRankConfig) CommInitRankConfig;
    decltype(&ncclCommInitAll) CommInitAll;
    decltype(&ncclCommDestroy) CommDestroy;
    decltype(&ncclGroupStart) GroupStart;
    decltype(&ncclGroupEnd) GroupEnd;
    decltype(&ncclSend) Send;
    decltype(&ncclRecv) Recv;
    decltype(&ncclGetErrorString) GetErrorString;
};

struct mmw_group {
    int n;
    std::vector<mmw_ctx *> ctx;
    std::vector<int> dev;
    std::vector<ncclComm_t> comm;
    NcclApi nccl;
    unsigned char *d_merged;          // on dev[0]: [32-byte header | records of all ranks, ordered]
    long long merged_cap;             // records d_merged can hold
    uint32_t *h_headers;              // pinned: 8 words per rank
    uint32_t *h_merged_header;        // pinned: 8 words
    uint32_t frame_offset;
    int gathered;                     // a merged block is queued / ready on GPU 0
};

#define NCCLCK(g, call)                                                                                   \
    do {                                                                                                  \
        ncclResult_t r_ = (call);                                                                         \
        if (r_ != ncclSuccess) {                                                                          \
            set_last_error("%s failed: %s", #call, (g)->nccl.GetErrorString ? (g)->nccl.GetErrorString(r_) : "?"); \
            return MMW_ERR_CUDA;                                                                          \
        }                                                                                                 \
    } while (0)

static int load_nccl(NcclApi *api)
{
    memset(api, 0, sizeof(*api));
    // the soname torch's bundled NCCL and the system NCCL share: if one is already in the process, this is it
    api->handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!api->handle) { set_last_error("mmw_group_create: cannot load libnccl.so.2 (%s)", dlerror()); return MMW_ERR_STATE; }
#define NCCL_SYM(field, name) api->field = reinterpret_cast<decltype(api->field)>(dlsym(api->handle, name))
    NCCL_SYM(GetUniqueId, "ncclGetUniqueId");
    NCCL_SYM(CommInitRankConfig, "ncclCommInitRankConfig");
    NCCL_SYM(CommInitAll, "ncclCommInitAll");
    NCCL_SYM(CommDestroy, "ncclCommDestroy");
    NCCL_SYM(GroupStart, "ncclGroupStart");
    NCCL_SYM(GroupEnd, "ncclGroupEnd");
    NCCL_SYM(Send, "ncclSend");
    NCCL_SYM(Recv, "ncclRecv");
    NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef NCCL_SYM
    if (!api->CommInitAll || !api->CommDestroy || !api->GroupStart || !api->GroupEnd || !api->Send || !api->Recv) {
        set_last_error("mmw_group_create: libnccl.so.2 lacks a required symbol");
        return MMW_ERR_STATE;
    }
    return MMW_OK;
}

void mmw_shard_frames(int n_frames, int n_ranks, int rank, int *first, int *count)
{
    if (n_ranks < 1) n_ranks = 1;
    const int base = n_frames / n_ranks, rem = n_frames % n_ranks;
    if (count) *count = base + (rank < rem ? 1 : 0);
    if (first) *first = rank * base + (rank < rem ? rank : rem);
}

void mmw_group_destroy(mmw_group *g)
{
    if (!g) return;
    for (size_t i = 0; i < g->comm.size(); ++i)
        if (g->comm[i] && g->nccl.CommDestroy) {
            cudaSetDevice(g->dev[i]);
            g->nccl.CommDestroy(g->comm[i]);
        }
    if (!g->dev.empty()) cudaSetDevice(g->dev[0]);
    if (g->d_merged) cudaFree(g->d_merged);
    if (g->h_headers) cudaFreeHost(g->h_headers);
    if (g->h_merged_header) cudaFreeHost(g->h_merged_header);
    for (mmw_ctx *c : g->ctx) mmw_destroy(c);
    delete g;
}

int mmw_group_create(const mmw_config *cfg, const int *devices, int n_devices, mmw_group **out)
{
    if (!cfg || !devices || !out || n_devices < 1 || n_devices > kMaxDevices) { set_last_error("mmw_group_create: bad argument"); return MMW_ERR_ARG; }
    *out = nullptr;
    for (int i = 0; i < n_devices; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) { set_last_error("mmw_group_create: device %d listed twice", devices[i]); return MMW_ERR_ARG; }
    mmw_group *g = new mmw_group();
    g->n = n_devices;
    g->d_merged = nullptr; g->h_headers = nullptr; g->h_merged_header = nullptr; g->frame_offset = 0; g->gathered = 0; g->merged_cap = 0;
    memset(&g->nccl, 0, sizeof(g->nccl));
    auto fail = [&](int code) { mmw_group_destroy(g); return code; };
    for (int i = 0; i < n_devices; ++i) {
        mmw_config c = *cfg;
        c.device = devices[i];
        mmw_ctx *ctx = nullptr;
        const int rc = mmw_create(&c, &ctx);
        if (rc) return fail(rc);
        g->ctx.push_back(ctx);
        g->dev.push_back(ctx->device);
        g->merged_cap += ctx->dense_cap;
    }
    if (cudaSetDevice(g->dev[0]) != cudaSuccess ||
        cudaMalloc((void **)&g->d_merged, kResultHeaderBytes + (size_t)g->merged_cap * sizeof(mmw_detection)) != cudaSuccess ||
        cudaMallocHost((void **)&g->h_headers, (size_t)n_devices * 32) != cudaSuccess ||
        cudaMallocHost((void **)&g->h_merged_header, 32) != cudaSuccess) {
        set_last_error("mmw_group_create: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(MMW_ERR_CUDA);
    }
    if (n_devices > 1) {
        int rc = load_nccl(&g->nccl);
        if (rc) return fail(rc);
        g->comm.assign(n_devices, nullptr);
        if (g->nccl.CommInitRankConfig && g->nccl.GetUniqueId) {
            // one CTA per peer: the gather moves KBs, and a wider NCCL kernel would evict the persistent CTAs of the FFT kernels
            ncclConfig_t conf = NCCL_CONFIG_INITIALIZER;
            conf.minCTAs = 1;
            conf.maxCTAs = 1;
            ncclUniqueId id;
            ncclResult_t r = g->nccl.GetUniqueId(&id);
            if (r == ncclSuccess) r = g->nccl.GroupStart();
            for (int i = 0; r == ncclSuccess && i < n_devices; ++i) {
                cudaSetDevice(g->dev[i]);
                r = g->nccl.CommInitRankConfig(&g->comm[i], n_devices, id, i, &conf);
            }
            if (r == ncclSuccess) r = g->nccl.GroupEnd();
            if (r != ncclSuccess) {
                set_last_error("mmw_group_create: NCCL communicator init failed: %s", g->nccl.GetErrorString ? g->nccl.GetErrorString(r) : "?");
                return fail(MMW_ERR_CUDA);
            }
        } else {
            const ncclResult_t r = g->nccl.CommInitAll(g->comm.data(), n_devices, g->dev.data());
            if (r != ncclSuccess) {
                set_last_error("mmw_group_create: ncclCommInitAll failed: %s", g->nccl.GetErrorString ? g->nccl.GetErrorString(r) : "?");
                return fail(MMW_ERR_CUDA);
            }
        }
    }
    *out = g;
    return MMW_OK;
}

int mmw_group_size(const mmw_group *g) { return g ? g->n : 0; }

mmw_ctx *mmw_group_context(mmw_group *g, int i) { return (g && i >= 0 && i < g->n) ? g->ctx[i] : nullptr; }

int mmw_group_set_frame_offset(mmw_group *g, uint32_t first_frame)
{
    if (!g) { set_last_error("mmw_group_set_frame_offset: null group"); return MMW_ERR_ARG; }
    g->frame_offset = first_frame;
    return MMW_OK;
}

// the exchange step: headers to the host, then exactly count_r records from every rank to their final offsets on GPU 0
static int group_gather(mmw_group *g, const int *n_frames)
{
    const int n = g->n;
    for (int i = 0; i < n; ++i) {
        mmw_ctx *c = g->ctx[i];
        CK(cudaSetDevice(c->device));
        if (n_frames[i] > 0)
            CK(cudaMemcpyAsync(g->h_headers + 8 * i, c->d_header, 32, cudaMemcpyDeviceToHost, c->stream));
        else
            memset(g->h_headers + 8 * i, 0, 32);
    }
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(g->ctx[i]->device));
        CK(cudaStreamSynchronize(g->ctx[i]->stream));
    }
    uint64_t off = 0, true_total = 0, frames = 0;
    uint32_t overflow = 0;
    std::vector<uint64_t> offs(n), cnt(n);
    for (int i = 0; i < n; ++i) {
        const uint32_t *h = g->h_headers + 8 * i;
        offs[i] = off;
        cnt[i] = h[0];
        if (off + cnt[i] > (uint64_t)g->merged_cap) { cnt[i] = (uint64_t)g->merged_cap > off ? (uint64_t)g->merged_cap - off : 0; overflow = 1; }
        off += cnt[i];
        true_total += h[1];
        frames += h[2];
        overflow |= h[3];
    }
    mmw_ctx *c0 = g->ctx[0];
    unsigned char *rec0 = g->d_merged + kResultHeaderBytes;
    CK(cudaSetDevice(c0->device));
    if (cnt[0] > 0)
        CK(cudaMemcpyAsync(rec0, c0->d_dense, cnt[0] * sizeof(mmw_detection), cudaMemcpyDeviceToDevice, c0->stream));
    bool any = false;
    for (int r = 1; r < n; ++r) any |= cnt[r] > 0;
    if (any) {
        NCCLCK(g, g->nccl.GroupStart());
        for (int r = 1; r < n; ++r) {
            if (cnt[r] == 0) continue;
            const size_t bytes = (size_t)cnt[r] * sizeof(mmw_detection);
            CK(cudaSetDevice(g->ctx[r]->device));
            NCCLCK(g, g->nccl.Send(g->ctx[r]->d_dense, bytes, ncclUint8, 0, g->comm[r], g->ctx[r]->stream));
            CK(cudaSetDevice(c0->device));
            NCCLCK(g, g->nccl.Recv(rec0 + offs[r] * sizeof(mmw_detection), bytes, ncclUint8, r, g->comm[0], c0->stream));
        }
        NCCLCK(g, g->nccl.GroupEnd());
    }
    uint32_t *mh = g->h_merged_header;
    memset(mh, 0, 32);
    mh[0] = (uint32_t)off;
    mh[1] = (uint32_t)true_total;
    mh[2] = (uint32_t)frames;
    mh[3] = overflow ? 1u : 0u;
    CK(cudaSetDevice(c0->device));
    CK(cudaMemcpyAsync(g->d_merged, mh, 32, cudaMemcpyHostToDevice, c0->stream));
    g->gathered = 1;
    return MMW_OK;
}

int mmw_group_process_device(mmw_group *g, const int16_t *const *adc_dev, const int *n_frames)
{
    if (!g || !adc_dev || !n_frames) { set_last_error("mmw_group_process_device: null argument"); return MMW_ERR_ARG; }
    g->gathered = 0;
    uint32_t first = g->frame_offset;
    for (int i = 0; i < g->n; ++i) {
        mmw_ctx *c = g->ctx[i];
        if (n_frames[i] < 0 || n_frames[i] > c->cfg.max_frames) { set_last_error("mmw_group_process_device: n_frames[%d] = %d outside 0..max_frames", i, n_frames[i]); return MMW_ERR_ARG; }
        if (n_frames[i] == 0) continue;
        int rc = check_batch_args(c, adc_dev[i], n_frames[i], "mmw_group_process_device");
        if (rc) return rc;
        CK(cudaSetDevice(c->device));
        if ((rc = check_device_capture(adc_dev[i], "mmw_group_process_device"))) return rc;
        c->plan.frame_offset = first;
        if ((rc = run_batch_graphed(c, adc_dev[i], n_frames[i]))) return rc;
        first += (uint32_t)n_frames[i];
    }
    return group_gather(g, n_frames);
}

int mmw_group_merged_block(mmw_group *g, const void **block_dev0, long long *capacity_bytes)
{
    if (!g) { set_last_error("mmw_group_merged_block: null group"); return MMW_ERR_ARG; }
    if (block_dev0) *block_dev0 = g->d_merged;
    if (capacity_bytes) *capacity_bytes = kResultHeaderBytes + g->merged_cap * (long long)sizeof(mmw_detection);
    return MMW_OK;
}

int mmw_group_read_detections(mmw_group *g, mmw_detection *dets, int det_capacity, int *n_det)
{
    if (n_det) *n_det = 0;
    if (!g) { set_last_error("mmw_group_read_detections: null group"); return MMW_ERR_ARG; }
    if (!g->gathered) { set_last_error("mmw_group_read_detections: no batch gathered"); return MMW_ERR_STATE; }
    mmw_ctx *c0 = g->ctx[0];
    CK(cudaSetDevice(c0->device));
    CK(cudaStreamSynchronize(c0->stream));
    uint32_t n = g->h_merged_header[0];
    int rc = g->h_merged_header[3] ? MMW_ERR_OVERFLOW : MMW_OK;
    if ((int)n > det_capacity) { n = det_capacity > 0 ? (uint32_t)det_capacity : 0; rc = MMW_ERR_OVERFLOW; }
    if (n > 0) {
        if (!dets) { set_last_error("detections pointer is null"); return MMW_ERR_ARG; }
        CK(cudaMemcpy(dets, g->d_merged + kResultHeaderBytes, (size_t)n * sizeof(mmw_detection), cudaMemcpyDeviceToHost));
    }
    if (n_det) *n_det = (int)n;
    if (rc == MMW_ERR_OVERFLOW) set_last_error("detection list truncated: %u of %u detections kept", n, g->h_merged_header[1]);
    return rc;
}

int mmw_group_process_host(mmw_group *g, const int16_t *adc_host, int n_frames, mmw_detection *dets, int det_capacity, int *n_det)
{
    if (n_det) *n_det = 0;
    if (!g || !adc_host) { set_last_error("mmw_group_process_host: null argument"); return MMW_ERR_ARG; }
    if (n_frames < 1 || n_frames > g->n * g->ctx[0]->cfg.max_frames) {
        set_last_error("mmw_group_process_host: n_frames %d outside 1..%d (n_devices * max_frames)", n_frames, g->n * g->ctx[0]->cfg.max_frames);
        return MMW_ERR_ARG;
    }
    g->gathered = 0;
    std::vector<int> cnt(g->n);
    const size_t frame_shorts = (size_t)2 * g->ctx[0]->plan.S * g->ctx[0]->plan.C * g->ctx[0]->plan.A;
    // every GPU's upload and chain are queued before any is waited for: the shards run side by side
    for (int i = 0; i < g->n; ++i) {
        int first = 0;
        mmw_shard_frames(n_frames, g->n, i, &first, &cnt[i]);
        if (cnt[i] == 0) continue;
        mmw_ctx *c = g->ctx[i];
        int rc = check_batch_args(c, adc_host, cnt[i], "mmw_group_process_host");
        if (rc) return rc;
        CK(cudaSetDevice(c->device));
        c->plan.frame_offset = g->frame_offset + (uint32_t)first;
        if ((rc = run_host_batch(c, adc_host + (size_t)first * frame_shorts, cnt[i]))) return rc;
    }
    const int rc = group_gather(g, cnt.data());
    if (rc) return rc;
    return mmw_group_read_detections(g, dets, det_capacity, n_det);
}

}  // extern "C"
