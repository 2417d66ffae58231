// mmw_cluster.cu — the batch's detection list grouped into objects (include/mmw_radar.h: mmw_set_clustering).
//
// Five launches after the detection stage, all sized on the host from capacities; the counts they work on (n_written, the
// frame offsets) are read on the device, so the sequence needs no host sync and can be captured in a graph:
//   init     parent[i] = i, size[i] = 0, labels[i] = -1
//   link     lock-free union-find (ECL-CC style): every detection looks up its neighbour candidates in the eps_range + 1
//            range rows at or below its own by binary search on the frame's sorted keys, and links each one by hooking
//            the larger root onto the smaller with atomicCAS.  Parents only decrease and parent[x] <= x, so every walk
//            ends, and the final root of a component is its lowest index whatever the schedule.
//   flatten  parent[i] = root(i); component sizes by integer atomicAdd (order-free)
//   order    one warp per frame walks the frame in index order: new qualifying roots get frame-local object numbers
//            (ballot + popc), members get their rank inside their object (match_any + popc) and are scattered to the
//            object's slots; the last CTA to finish scans the per-frame counts into object offsets and the header
//   objects  one warp per object loads its members 32 at a time and sums them in ascending index order (fp64, products
//            exact, the order kept through shuffles), then writes the record
// No kernel waits on another CTA: the only cross-CTA step is the last-CTA-done scan list_kernel also uses.  The kernels do
// not take PlanDev: frame_offset reaches the objects through the records' own frame field.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mmw_common.cuh"

namespace mmw {

constexpr int kClusterNT = 256;
constexpr int kOrderWarps = kClusterNT / 32;

// the frame f with offsets[f] <= i < offsets[f + 1], for i < offsets[n_frames]
__device__ __forceinline__ int cluster_frame_of(const uint32_t *__restrict__ offsets, int n_frames, uint32_t i)
{
    int lo = 0, hi = n_frames;                                   // offsets[lo] <= i < offsets[hi]
    while (hi - lo > 1) {                                        // <= log2(max_frames) + 1 steps
        const int mid = (lo + hi) >> 1;
        if (offsets[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ int ld_parent(const int *parent, int x)
{
    return *(const volatile int *)(parent + x);
}

// root of x with pointer jumping: every store writes an ancestor (smaller index) into a non-root, so roots are never
// overwritten here and the atomicCAS hooks below stay valid.  Each step lowers `cur`: at most max_det steps.
__device__ __forceinline__ int cluster_find(int *parent, int x)
{
    int cur = ld_parent(parent, x);
    if (cur != x) {
        int prev = x, next;
        while (cur > (next = ld_parent(parent, cur))) {
            parent[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

// hook the larger of the two roots onto the smaller; a failed CAS returns the (smaller) parent the root got meanwhile.
// Every pass lowers a or b, both stay inside the frame: at most 2 * max_det passes.
__device__ __forceinline__ void cluster_unite(int *parent, int a, int b)
{
    a = cluster_find(parent, a);
    b = cluster_find(parent, b);
    while (a != b) {
        if (a < b) { const int t = a; a = b; b = t; }           // a > b: hook a onto b
        const int old = atomicCAS(parent + a, a, b);
        if (old == a) break;
        a = old;
    }
}

__global__ void __launch_bounds__(kClusterNT) cluster_init_kernel(const uint32_t *__restrict__ det_header, int *__restrict__ parent,
                                                                  uint32_t *__restrict__ size, int32_t *__restrict__ labels, int dense_cap)
{
    const uint32_t n = min(det_header[0], (uint32_t)dense_cap);
    for (uint32_t i = blockIdx.x * kClusterNT + threadIdx.x; i < n; i += gridDim.x * kClusterNT) {
        parent[i] = (int)i;
        size[i] = 0u;
        labels[i] = -1;
    }
}

__global__ void __launch_bounds__(kClusterNT) cluster_link_kernel(mmw_cluster_params cp, int Cp, int max_det, const mmw_detection *__restrict__ dense,
                                                                  const uint32_t *__restrict__ det_header, const uint32_t *__restrict__ keys,
                                                                  const uint32_t *__restrict__ offsets, int *parent, int n_frames, int dense_cap)
{
    const uint32_t n = min(det_header[0], (uint32_t)dense_cap);
    const int half = Cp / 2;
    for (uint32_t i = blockIdx.x * kClusterNT + threadIdx.x; i < n; i += gridDim.x * kClusterNT) {
        const int f = cluster_frame_of(offsets, n_frames, i);
        const uint32_t s = offsets[f];
        const uint32_t k = i - s;                                // < min(count, max_det): list_kernel's clip
        if (k >= (uint32_t)max_det) continue;
        const uint32_t nf = min(offsets[f + 1] - s, (uint32_t)max_det);
        const uint32_t *kf = keys + (size_t)f * max_det;
        const uint32_t key = kf[k];
        const int r = (int)(key >> 16), d = (int)(key & 0xffffu);
        const int ds = d < half ? d : d - Cp;
        const int a = dense[i].angle_bin;
        const int lo_s = max(ds - cp.eps_doppler, -half), hi_s = min(ds + cp.eps_doppler, half - 1);
        for (int rr = max(0, r - cp.eps_range); rr <= r; ++rr) {
            const uint32_t limit = rr == r ? k : nf;              // same row: only the lower-index candidates (j < i)
            // the signed window [lo_s, hi_s] as at most two contiguous bin intervals: d' >= 0 and d' < 0 (bins + Cp)
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                const int u0 = part == 0 ? max(lo_s, 0) : lo_s + Cp;
                const int u1 = part == 0 ? hi_s : min(hi_s, -1) + Cp;
                if ((part == 0 && hi_s < 0) || (part == 1 && lo_s >= 0) || u0 > u1) continue;
                const uint32_t q0 = ((uint32_t)rr << 16) | (uint32_t)u0, q1 = ((uint32_t)rr << 16) | (uint32_t)u1;
                uint32_t lo = 0, hi = limit;                     // lower bound of q0 in kf[0, limit)
                while (lo < hi) {                                // <= log2(max_det) + 1 steps
                    const uint32_t mid = (lo + hi) >> 1;
                    if (kf[mid] < q0) lo = mid + 1;
                    else hi = mid;
                }
                for (uint32_t j = lo; j < limit && kf[j] <= q1; ++j) {   // distinct keys: <= 2 eps_doppler + 1 candidates
                    const int aj = dense[s + j].angle_bin;
                    if (abs(a - aj) <= cp.eps_angle) cluster_unite(parent, (int)i, (int)(s + j));
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kClusterNT) cluster_flatten_kernel(const uint32_t *__restrict__ det_header, int *parent, uint32_t *__restrict__ size,
                                                                     int dense_cap)
{
    const uint32_t n = min(det_header[0], (uint32_t)dense_cap);
    for (uint32_t i = blockIdx.x * kClusterNT + threadIdx.x; i < n; i += gridDim.x * kClusterNT) {
        // the forest is final: walk without shortcuts (the only stores of this kernel write the final roots)
        int x = (int)i, p = ld_parent(parent, x);
        while (p != x) {                                         // each step lowers x: <= max_det steps
            x = p;
            p = ld_parent(parent, x);
        }
        parent[i] = x;
        atomicAdd(size + x, 1u);
    }
}

__global__ void __launch_bounds__(kClusterNT) cluster_order_kernel(mmw_cluster_params cp, int max_det, const uint32_t *__restrict__ det_header,
                                                                   const uint32_t *__restrict__ offsets, const int *__restrict__ parent,
                                                                   const uint32_t *__restrict__ size, int *__restrict__ oid,
                                                                   uint32_t *__restrict__ cursor, uint32_t *__restrict__ members,
                                                                   uint32_t *__restrict__ frame_objs, uint32_t *__restrict__ obj_offsets,
                                                                   uint2 *__restrict__ slots, unsigned int *__restrict__ ticket,
                                                                   uint32_t *__restrict__ obj_header, int n_frames, int dense_cap)
{
    __shared__ uint32_t scan_s[kOrderWarps], tsum_s[kOrderWarps];
    __shared__ bool is_last;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t n = min(det_header[0], (uint32_t)dense_cap);
    const int f = blockIdx.x * kOrderWarps + warp;
    if (f < n_frames) {
        const uint32_t s = min(offsets[f], n), e = min(min(offsets[f + 1], n), s + (uint32_t)max_det);
        uint32_t n_obj = 0, n_slots = 0;                         // objects numbered so far, member slots handed out
        int r_next = s + lane < e ? parent[s + lane] : -1;      // the walk is latency-bound: the next chunk's loads are
        uint32_t sz_next = s + lane < e ? size[s + lane] : 0u;  // issued one chunk ahead
        for (uint32_t base = s; base < e; base += 32) {           // <= max_det / 32 chunks
            const uint32_t i = base + lane;
            const bool valid = i < e;
            const int r = r_next;
            const uint32_t sz = sz_next;
            r_next = i + 32 < e ? parent[i + 32] : -1;
            sz_next = i + 32 < e ? size[i + 32] : 0u;
            const bool is_root = valid && r == (int)i;
            const bool qual = is_root && sz >= (uint32_t)cp.min_points;
            const uint32_t bal = __ballot_sync(0xffffffffu, qual);
            const uint32_t local = n_obj + __popc(bal & lt);
            const bool kept = qual && local < (uint32_t)cp.max_objects_per_frame;
            // member slots of the objects kept in this chunk: exclusive scan of their sizes
            const uint32_t want = kept ? sz : 0u;
            uint32_t incl = want;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            if (is_root) {
                oid[i] = qual ? (int)local : -1;
                if (kept) {
                    const uint32_t first = s + n_slots + incl - want;
                    cursor[i] = first;
                    slots[(size_t)f * cp.max_objects_per_frame + local] = make_uint2(i, first);
                }
            }
            n_obj += __popc(bal);
            n_slots += __shfl_sync(0xffffffffu, incl, 31);
            __syncwarp();                                        // oid / cursor of this chunk's roots visible to the warp
            // rank of each member inside its object: members of one root in this chunk are one match group
            const uint32_t grp = __match_any_sync(0xffffffffu, r);
            const int o = valid ? oid[r] : -1;
            const uint32_t cur = valid ? cursor[r] : 0u;             // meaningful for members of kept objects only
            const bool member = o >= 0 && o < cp.max_objects_per_frame;
            uint32_t slot = 0;
            if (member) slot = cur + __popc(grp & lt);
            __syncwarp();                                        // every lane has read cursor[r] before the leader moves it
            if (member) {
                members[slot] = i;
                if (lane == 31 - __clz(grp)) cursor[r] = slot + 1;
            }
            __syncwarp();
        }
        if (lane == 0) {
            frame_objs[2 * f] = n_obj;
            frame_objs[2 * f + 1] = min(n_obj, (uint32_t)cp.max_objects_per_frame);
            __threadfence();
        }
    }
    __syncthreads();
    if (tid == 0) {
        const unsigned int done = atomicAdd(ticket, 1u);
        is_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;

    // ---- last CTA: exclusive scan of the kept counts -> obj_offsets[f], header ----
    __threadfence();
    uint32_t carry = 0, true_total = 0, cut = 0;
    for (int b0 = 0; b0 < n_frames; b0 += kClusterNT) {          // <= max_frames / 256 rounds
        const int i = b0 + tid;
        const uint32_t t = i < n_frames ? __ldcg(frame_objs + 2 * i) : 0u;
        const uint32_t kc = i < n_frames ? __ldcg(frame_objs + 2 * i + 1) : 0u;
        uint32_t inc = kc, ts = t;
        cut |= t != kc ? 1u : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ts += __shfl_xor_sync(0xffffffffu, ts, o);
        __syncthreads();
        if (lane == 31) { scan_s[warp] = inc; tsum_s[warp] = ts; }
        __syncthreads();
        uint32_t wbase = 0, chunk = 0, tchunk = 0;
        for (int w = 0; w < kOrderWarps; ++w) {
            if (w < warp) wbase += scan_s[w];
            chunk += scan_s[w];
            tchunk += tsum_s[w];
        }
        if (i < n_frames) obj_offsets[i] = carry + wbase + inc - kc;
        carry += chunk;
        true_total += tchunk;
    }
    cut = __syncthreads_or(cut);
    if (tid == 0) {
        obj_offsets[n_frames] = carry;
        obj_header[0] = carry;
        obj_header[1] = true_total;
        obj_header[2] = (uint32_t)n_frames;
        obj_header[3] = (cut ? MMW_OBJECTS_CUT : 0u) | (det_header[3] ? MMW_OBJECTS_DETECTIONS_TRUNCATED : 0u);
        obj_header[4] = obj_header[5] = obj_header[6] = obj_header[7] = 0u;
        ticket[0] = 0u;                                          // self-cleaning for the next batch
    }
}

// one warp per object: the lanes load 32 members at a time (independent loads, labels written in parallel); the fp64 sums
// then take the members one by one in index order through shuffles, so the rounding sequence is the CPU reference's (tests/cluster_ref.c)
__global__ void __launch_bounds__(kClusterNT) cluster_object_kernel(int Cp, int max_obj, const mmw_detection *__restrict__ dense,
                                                                    const uint32_t *__restrict__ obj_offsets, const uint2 *__restrict__ slots,
                                                                    const uint32_t *__restrict__ size, const uint32_t *__restrict__ members,
                                                                    const uint32_t *__restrict__ obj_header, int32_t *__restrict__ labels,
                                                                    mmw_object *__restrict__ objs, int n_frames, int dense_cap)
{
    const uint32_t n_obj = min(obj_header[0], (uint32_t)n_frames * (uint32_t)max_obj);
    const int half = Cp / 2;
    const int lane = threadIdx.x & 31;
    const uint32_t n_warps = gridDim.x * (kClusterNT / 32);
    for (uint32_t o = (blockIdx.x * kClusterNT + threadIdx.x) >> 5; o < n_obj; o += n_warps) {     // warp-uniform
        const int f = cluster_frame_of(obj_offsets, n_frames, o);
        const uint32_t local = o - obj_offsets[f];
        if (local >= (uint32_t)max_obj) continue;
        const uint2 sl = slots[(size_t)f * max_obj + local];
        const uint32_t root = sl.x, first = sl.y;
        if (root >= (uint32_t)dense_cap) continue;
        const uint32_t cnt = size[root];
        if (cnt == 0 || first + cnt > (uint32_t)dense_cap) continue;
        double sp = 0.0, sr = 0.0, sd = 0.0, sa = 0.0;
        float pp = -INFINITY;
        uint32_t peak = root;
        int rmin = 0xffff, rmax = 0, dmin = half, dmax = -half;
        for (uint32_t t0 = 0; t0 < cnt; t0 += 32) {                // <= max_det / 32 chunks
            const uint32_t t = t0 + lane;
            const bool valid = t < cnt;
            uint32_t j = valid ? members[first + t] : 0u;
            const bool ok = valid && j < (uint32_t)dense_cap;
            float pw = -INFINITY;
            double p = 0.0, pr = 0.0, pd = 0.0, pa = 0.0;
            int r = 0xffff, rx = 0, ds = half, dx = -half;
            if (ok) {
                const mmw_detection rec = dense[j];
                const int d = rec.doppler_bin < half ? (int)rec.doppler_bin : (int)rec.doppler_bin - Cp;
                pw = rec.power;
                p = (double)rec.power;                           // p * x is exact in fp64: contraction cannot change a sum
                pr = p * (double)rec.range_bin;
                pd = p * (double)d;
                pa = p * (double)rec.angle_rad;
                r = rx = rec.range_bin;
                ds = dx = d;
                labels[j] = (int32_t)o;
            } else {
                j = 0xffffffffu;
            }
            const int m = cnt - t0 < 32u ? (int)(cnt - t0) : 32;
            for (int l = 0; l < m; ++l) {                        // ascending member index
                sp += __shfl_sync(0xffffffffu, p, l);
                sr += __shfl_sync(0xffffffffu, pr, l);
                sd += __shfl_sync(0xffffffffu, pd, l);
                sa += __shfl_sync(0xffffffffu, pa, l);
            }
            // strongest member of the chunk, the lower index on equal power; an earlier chunk wins ties (lower indices)
            float bp = pw;
            uint32_t bj = j;
#pragma unroll
            for (int x = 16; x > 0; x >>= 1) {
                const float op = __shfl_xor_sync(0xffffffffu, bp, x);
                const uint32_t oj = __shfl_xor_sync(0xffffffffu, bj, x);
                if (op > bp || (op == bp && oj < bj)) { bp = op; bj = oj; }
            }
            if (bp > pp) { pp = bp; peak = bj; }
            rmin = min(rmin, __reduce_min_sync(0xffffffffu, r));
            rmax = max(rmax, __reduce_max_sync(0xffffffffu, rx));
            dmin = min(dmin, __reduce_min_sync(0xffffffffu, ds));
            dmax = max(dmax, __reduce_max_sync(0xffffffffu, dx));
        }
        if (lane == 0 && peak < (uint32_t)dense_cap) {
            mmw_object ob;
            ob.frame = dense[root].frame;
            ob.first_det = root;
            ob.n_det = cnt;
            ob.peak_det = peak;
            ob.range_bin = sp > 0.0 ? (float)(sr / sp) : 0.f;
            ob.doppler_bin = sp > 0.0 ? (float)(sd / sp) : 0.f;
            ob.angle_rad = sp > 0.0 ? (float)(sa / sp) : 0.f;
            ob.power = (float)sp;
            ob.peak_power = pp;
            ob.peak_noise = dense[peak].noise;
            ob.range_min = (uint16_t)rmin;
            ob.range_max = (uint16_t)rmax;
            ob.doppler_min = (int16_t)dmin;
            ob.doppler_max = (int16_t)dmax;
            objs[o] = ob;
        }
    }
}

cudaError_t launch_cluster(const mmw_cluster_params &cp, int Cp, int max_det, const ClusterBuffers &b, int n_frames, int dense_cap,
                           int sm_count, cudaStream_t st)
{
    // grid-stride grids sized from the capacities (the counts are only known on the device)
    const int by_cap = (dense_cap + kClusterNT - 1) / kClusterNT;
    const int grid = by_cap < sm_count * 8 ? (by_cap < 1 ? 1 : by_cap) : sm_count * 8;
    const int obj_cap = n_frames * cp.max_objects_per_frame;
    const int by_obj = (obj_cap + kOrderWarps - 1) / kOrderWarps;          // one warp per object
    const int grid_obj = by_obj < sm_count * 8 ? (by_obj < 1 ? 1 : by_obj) : sm_count * 8;
    cluster_init_kernel<<<grid, kClusterNT, 0, st>>>(b.det_header, b.parent, b.size, b.labels, dense_cap);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    cluster_link_kernel<<<grid, kClusterNT, 0, st>>>(cp, Cp, max_det, b.dense, b.det_header, b.keys, b.offsets, b.parent, n_frames, dense_cap);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    cluster_flatten_kernel<<<grid, kClusterNT, 0, st>>>(b.det_header, b.parent, b.size, dense_cap);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    cluster_order_kernel<<<(n_frames + kOrderWarps - 1) / kOrderWarps, kClusterNT, 0, st>>>(
        cp, max_det, b.det_header, b.offsets, b.parent, b.size, b.oid, b.cursor, b.members, b.frame_objs, b.obj_offsets, b.slots,
        b.ticket, b.obj_header, n_frames, dense_cap);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    cluster_object_kernel<<<grid_obj, kClusterNT, 0, st>>>(Cp, cp.max_objects_per_frame, b.dense, b.obj_offsets, b.slots, b.size, b.members,
                                                            b.obj_header, b.labels, b.objs, n_frames, dense_cap);
    return cudaGetLastError();
}

}  // namespace mmw
