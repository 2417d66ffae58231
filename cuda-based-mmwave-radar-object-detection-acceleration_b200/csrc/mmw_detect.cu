// mmw_detect.cu — stages 3 and 4 of the chain: power map -> detection records.
//
//   K3  cfar_walk_kernel / cfar_kernel
//                       2-D cell-averaging CFAR on the integrated power map.  Range axis clamps
//                       (training count recounted), Doppler axis wraps.  Emits a bit mask and, for
//                       hit cells only, the noise estimate.  Default geometry: the "walk" form (Doppler
//                       sums in registers down each range column, range sums on packed pairs out of
//                       shared memory); any other guard / training window: the tiled kernel.
//   K4a list_kernel     per frame: ordered compaction of the mask bits into (range, doppler) keys and
//                       the per-frame count; the last CTA to finish scans the counts into offsets of
//                       the dense list and writes the header (no extra launch, no host round trip).
//   K4b measure_kernel  one warp per detection over the whole batch: 3x3 peak grouping, antenna
//                       snapshot (from the Doppler cube, or re-derived from the range spectrum in fused
//                       mode), angle spectrum arg-max; records go straight into the dense ordered list.
//
// The reference has no counterpart for any of this (SURVEY.md §8a n4-n8); its only "detector" is the
// host arg-max of acceleration.cu:391-407.
//
// Numerical note on the CFAR sums.  A target cell is up to ~1e9 x the noise floor after the 2-D FFT
// gain, so running sums with subtraction, prefix-sum differences and "outer box minus inner box" are
// all unusable in fp32: they leave an error of tens of noise floors behind every strong cell.  Every
// sum below therefore only ever ADDS training cells.  Tiled kernel: per row a `full` window sum and a
// `ring` sum (full minus the guard span, computed as left + right), then a column sum that takes `ring`
// rows inside the Doppler guard and `full` rows outside it; the walk kernel splits the window the other
// way round (see its header).
#include <stdlib.h>

#include "fft_regs.cuh"
#include "mmw_common.cuh"

namespace mmw {

constexpr int kCfarRT = 64;      // range bins per tile
constexpr int kCfarDT = 32;      // Doppler bins per tile (one mask word per range bin)
constexpr int kCfarNT = 256;
constexpr int kCfarRS = kCfarRT + 4;   // row stride of the row-sum arrays (16-byte aligned rows)

// Tiled CFAR for any guard / training window other than the default one (that one takes cfar_walk_kernel below):
// one CTA per 64 x 32 tile plus its halo, run-time window bounds, one cell at a time.
__global__ void __launch_bounds__(kCfarNT) cfar_kernel(PlanDev p, const float *__restrict__ pmap, uint32_t *__restrict__ mask,
                                                       float *__restrict__ noise_map)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int Gr = p.guard_r, Gd = p.guard_d;
    const int Wr = p.win_r_half, Wd = p.win_d_half;
    const int Sp = p.Sp, Cp = p.Cp;
    const int Lp = (Wr + 3) & ~3;                        // halo rounded up to whole float4 chunks
    const int tw_ = kCfarRT + 2 * Lp;                    // tile width (range, fastest)
    const int th_ = kCfarDT + 2 * Wd;                    // tile height (Doppler)
    constexpr int RS = kCfarRS;
    float *tile = reinterpret_cast<float *>(smem);       // [th_][tw_]
    float *fullS = tile + th_ * tw_;                     // [th_][RS]
    float *ringS = fullS + th_ * RS;                     // [th_][RS]
    uint32_t *words = reinterpret_cast<uint32_t *>(ringS + th_ * RS);   // [RT]

    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * kCfarRT;
    const int dblk = blockIdx.y;
    const int f = blockIdx.z;
    const int d0 = dblk * kCfarDT;
    const float *pf = pmap + (size_t)f * Cp * Sp;

    // ---- tile + halo, staged with 16-byte cp.async (all copies in flight at once; zero-fill outside
    //      [0, Sp) -- adding +0 is exact); Doppler wraps.  Tile column 0 is range bin r0 - Lp. ----
    if (tid < kCfarRT) words[tid] = 0u;
    {
        const int qpr = tw_ / 4;                             // float4 chunks per tile row
        for (int i = tid; i < th_ * qpr; i += kCfarNT) {
            const int j = i / qpr, x4 = (i - j * qpr) * 4;
            const int d = (d0 - Wd + j + Cp) & (Cp - 1);
            const int r = r0 - Lp + x4;
            const bool in = (r >= 0 && r < Sp);
            const float *src = pf + (size_t)d * Sp + (in ? r : 0);
            const uint32_t dst = smem_u32(tile + j * tw_ + x4);
            const int nbytes = in ? 16 : 0;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
        }
        asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();

    for (int t = tid; t < th_ * kCfarRT; t += kCfarNT) {
        const int j = t / kCfarRT, x = t % kCfarRT;
        const float *c = tile + j * tw_ + x + (Lp - Wr);   // c[i] = offset (i - Wr)
        float left = 0.f, right = 0.f, mid = 0.f;
        for (int i = 0; i < Wr - Gr; ++i) left += c[i];
        for (int i = Wr + Gr + 1; i <= 2 * Wr; ++i) right += c[i];
        for (int i = Wr - Gr; i <= Wr + Gr; ++i) mid += c[i];
        ringS[j * RS + x] = left + right;
        fullS[j * RS + x] = (left + right) + mid;
    }
    __syncthreads();
    for (int t = tid; t < kCfarDT * kCfarRT; t += kCfarNT) {
        const int x = t % kCfarRT, dl = t / kCfarRT;
        const int r = r0 + x;
        float T = 0.f;
        for (int jj = 0; jj <= 2 * Wd; ++jj) {
            const float *src = (jj >= Wd - Gd && jj <= Wd + Gd) ? ringS : fullS;
            T += src[(dl + jj) * RS + x];
        }
        const int n_full = min(r + Wr, Sp - 1) - max(r - Wr, 0) + 1;
        const int n_guard = min(r + Gr, Sp - 1) - max(r - Gr, 0) + 1;
        const int n = (2 * Wd + 1) * n_full - (2 * Gd + 1) * n_guard;
        const float noise = T * (1.0f / (float)max(n, 1));
        const float cut = tile[(dl + Wd) * tw_ + x + Lp];
        if ((r < Sp) && (n > 0) && (cut > p.alpha * noise)) {
            atomicOr(&words[x], 1u << dl);
            noise_map[((size_t)f * Cp + d0 + dl) * Sp + r] = noise;
        }
    }
    __syncthreads();
    if (tid < kCfarRT && r0 + tid < Sp) mask[((size_t)f * (Cp / 32) + dblk) * Sp + r0 + tid] = words[tid];
}

// ---------------------------------------------------------------------------
// K3, default geometry (guard 2x2, train 8x4), Sp % 64 == 0, Cp % 32 == 0: "walk" form.
//
// A tiled kernel like cfar_kernel above is instruction-bound (ncu, on its fully unrolled form for this window, which the
// walk form replaced: ~74 thread instructions per cell): independent 64 x 32 tiles re-stage
// 1.9x their cells as halo, and the column pass reads 22 scalar shared-memory words per 4 cells.  Here the window is
// split the other way round.  With F13 / R8 = the 13-row Doppler sum of one range column and its 8-row ring (13 minus
// the 5 guard rows),
//     noise_sum(r, d) = sum_{3 <= |dr| <= 10} F13[r + dr][d]  +  sum_{|dr| <= 2} R8[r + dr][d]
// (the same training cells, still only ever added).  A CTA owns a strip of RT range bins x (16 * nchunk) Doppler bins of
// one frame.  Everything is computed on float2 pairs = (strip column c, strip column c + RT/2) with packed fp32x2 adds,
// so the two halves of the strip ride in the two halves of every instruction and no value is ever moved between them.
//   phase A  one thread = one pair-column (lanes along range: plain coalesced global loads, no staging), walking down
//            the Doppler axis 16 rows at a time with the last 12 input rows carried in registers; sliding 4- and
//            5-sums by doubling: 100 FADD2 per 32 cells.
//   phase B  one thread = SW pair-cells of one row: F13 / R8 / the cells come back as LDS.128 (two pair-columns each),
//            sliding 8- and 5-sums by doubling, threshold test by sign (109 FADD2 per 16 cells at SW = 8).
// Doppler wraps, range zero-fills (adding +0 is exact) and the training count is recounted near the range edges
// exactly as above.  Every cell's sum is one fixed expression of the power map, independent of RT, nchunk and the
// batch size.
// ---------------------------------------------------------------------------
template <int RT>
struct WalkShape {
    static constexpr int H = RT / 2;             // pair-cells per row
    static constexpr int NP = H + 24;            // pair-columns incl. the 12-bin halo on either side (10 needed; 12 keeps 16-byte alignment)
    static constexpr int CS = H + 34;            // row stride in float2; CS % 16 == 2 makes phase B's LDS.128 conflict-free
    static constexpr int SW = 8;                 // pair-cells per phase-B task
    static constexpr int NTASK = 16 * (H / SW);
    static constexpr int NT = NTASK > ((NP + 31) & ~31) ? NTASK : ((NP + 31) & ~31);
    static constexpr int SMEM = 3 * 16 * CS * 8 + H * 8 + RT * 4;
    static_assert(CS % 16 == 2 && CS >= NP + 2, "row stride");
};

template <int RT, int MINB, int SPT>
__global__ void __launch_bounds__(WalkShape<RT>::NT, MINB) cfar_walk_kernel(PlanDev p, const float *__restrict__ pmap, uint32_t *__restrict__ mask,
                                                                            float *__restrict__ noise_map, int nchunk)
{
    using Sh = WalkShape<RT>;
    constexpr int H = Sh::H, NP = Sh::NP, CS = Sh::CS, SW = Sh::SW;
    extern __shared__ __align__(16) unsigned char smem[];
    float2 *sF = reinterpret_cast<float2 *>(smem);      // [16][CS]  F13 of (column c, column c + H)
    float2 *sR = sF + 16 * CS;                          // ring sums, same layout
    float2 *sC = sR + 16 * CS;                          // the cells themselves; phase B leaves each cell's noise estimate in its place
    float2 *sInv = sC + 16 * CS;                        // [H]  1 / training-cell count of range bins (r0 + q, r0 + H + q)
    uint32_t *words = reinterpret_cast<uint32_t *>(sInv + H);   // [RT]

    const int tid = threadIdx.x;
    const uint32_t Sp = SPT ? SPT : p.Sp, Cp = p.Cp;    // SPT: the row offsets of phase A's loads become immediates
    const int r0 = blockIdx.x * RT;
    const uint32_t dseg0 = blockIdx.y * 16 * nchunk;
    const uint32_t f = blockIdx.z;
    const float *pf = pmap + (size_t)f * Cp * Sp;

    // phase A identity: pair-column tid = range bins (rX, rX + H)
    const int rX = r0 - 12 + tid;
    const bool colA = tid < NP;
    const bool liveX = colA && rX >= 0 && rX < (int)Sp;
    const bool liveY = colA && rX + H >= 0 && rX + H < (int)Sp;
    const float *cx = pf + (liveX ? rX : 0), *cy = pf + (liveY ? rX + H : 0);
    // phase B identity: row j of the chunk, pair-cells x0 .. x0 + SW - 1
    const int j = tid & 15, x0 = (tid >> 4) * SW;
    const bool taskB = tid < Sh::NTASK;

    if (tid < H) {
        float inv[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int r = r0 + tid + u * H;
            const int n_full = min(r + 10, (int)Sp - 1) - max(r - 10, 0) + 1;
            const int n_guard = min(r + 2, (int)Sp - 1) - max(r - 2, 0) + 1;
            inv[u] = 1.0f / (float)(13 * n_full - 5 * n_guard);            // 1/248 away from the range edges
        }
        sInv[tid] = make_float2(inv[0], inv[1]);
    }
    if (tid < RT) words[tid] = 0u;

    float2 P[28];                            // P[i] = row dseg0 + 16 k - 6 + i of this pair-column
#pragma unroll
    for (int i = 0; i < 28; ++i) P[i] = make_float2(0.f, 0.f);
    if (colA) {                              // run-in: the 12 rows before the segment's first new row
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            const uint32_t o = ((dseg0 + Cp - 6 + i) & (Cp - 1)) * Sp;
            if (liveX) P[16 + i].x = __ldg(cx + o);
            if (liveY) P[16 + i].y = __ldg(cy + o);
        }
    }

    for (int k = 0; k < nchunk; ++k) {
        const uint32_t dk = dseg0 + 16 * k;
        if (colA) {
#pragma unroll
            for (int i = 0; i < 12; ++i) P[i] = P[i + 16];
            if (liveX && liveY && dk + 22 <= Cp) {       // the usual case: both columns inside the map, rows dk + 6 .. dk + 21 do not wrap
                const float *px = cx + (dk + 6) * Sp, *py = cy + (dk + 6) * Sp;
#pragma unroll
                for (int i = 0; i < 16; ++i) P[12 + i] = make_float2(__ldg(px + i * Sp), __ldg(py + i * Sp));
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const uint32_t o = ((dk + 6 + i) & (Cp - 1)) * Sp;
                    P[12 + i] = make_float2(liveX ? __ldg(cx + o) : 0.f, liveY ? __ldg(cy + o) : 0.f);
                }
            }
            float2 s2[27], s4[25];
#pragma unroll
            for (int i = 0; i < 27; ++i) s2[i] = __fadd2_rn(P[i], P[i + 1]);
#pragma unroll
            for (int i = 0; i < 25; ++i) s4[i] = __fadd2_rn(s2[i], s2[i + 2]);      // rows i .. i+3
#pragma unroll
            for (int q = 0; q < 16; ++q) {                                           // output row q; its centre is input row q + 6
                const float2 ring = __fadd2_rn(s4[q], s4[q + 9]);                    // Doppler offsets -6..-3 and +3..+6
                const float2 mid = __fadd2_rn(s4[q + 4], P[q + 8]);                  // offsets -2..+2
                sR[q * CS + tid] = ring;
                sF[q * CS + tid] = __fadd2_rn(ring, mid);
                sC[q * CS + tid] = P[q + 6];
            }
        }
        __syncthreads();
        if (taskB) {
            const float4 *f4 = reinterpret_cast<const float4 *>(sF + j * CS + x0);
            const float4 *r4 = reinterpret_cast<const float4 *>(sR + j * CS + x0 + 8);
            float4 *c4 = reinterpret_cast<float4 *>(sC + j * CS + x0 + 12);
            const float4 *i4 = reinterpret_cast<const float4 *>(sInv + x0);
            constexpr int NV = SW + 24;      // V[i] = F13 at pair-column x0 + i; pair-cell q sits at pair-column x0 + 12 + q
            float2 V[NV], LR[SW];
#pragma unroll
            for (int i = 1; i < NV / 2 - 1; ++i) {
                const float4 t = f4[i];
                V[2 * i] = make_float2(t.x, t.y); V[2 * i + 1] = make_float2(t.z, t.w);
            }
            {
                float2 a2[NV - 3], a4[NV - 5];
#pragma unroll
                for (int i = 2; i < NV - 3; ++i) a2[i] = __fadd2_rn(V[i], V[i + 1]);
#pragma unroll
                for (int i = 2; i < NV - 5; ++i) a4[i] = __fadd2_rn(a2[i], a2[i + 2]);   // columns i .. i+3
#pragma unroll
                for (int q = 0; q < SW; ++q)                                         // range offsets -10..-3 and +3..+10
                    LR[q] = __fadd2_rn(__fadd2_rn(a4[q + 2], a4[q + 6]), __fadd2_rn(a4[q + 15], a4[q + 19]));
            }
            float2 W[SW + 8];                // W[i] = ring sum at pair-column x0 + 8 + i; pair-cell q uses W[q+2 .. q+6]
#pragma unroll
            for (int i = 1; i < SW / 2 + 4; ++i) {
                const float4 t = r4[i];
                W[2 * i] = make_float2(t.x, t.y); W[2 * i + 1] = make_float2(t.z, t.w);
            }
            float2 b2[SW + 5], b4[SW + 2];
#pragma unroll
            for (int i = 2; i < SW + 5; ++i) b2[i] = __fadd2_rn(W[i], W[i + 1]);
#pragma unroll
            for (int i = 2; i < SW + 2; ++i) b4[i] = __fadd2_rn(b2[i], b2[i + 2]);
            const float2 alpha2 = make_float2(p.alpha, p.alpha);
            // hit <=> cut > alpha * noise <=> alpha * noise - cut < 0 (the rounded difference of two floats has the sign of the
            // exact one); the sign bits are shifted into hx / hy: after the loop bit (SW - 1 - q) = pair-cell q, x / y half
            uint32_t hx = 0, hy = 0;
#pragma unroll
            for (int q2 = 0; q2 < SW / 2; ++q2) {
                const float4 inv = i4[q2];
                const float4 cc = c4[q2];
                float2 nz[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int q = 2 * q2 + u;
                    const float2 mid = __fadd2_rn(b4[q + 2], W[q + 6]);              // -2..+2 of the ring sums
                    const float2 T = __fadd2_rn(LR[q], mid);
                    nz[u] = __fmul2_rn(T, u ? make_float2(inv.z, inv.w) : make_float2(inv.x, inv.y));
                    const float2 thr = __fmul2_rn(nz[u], alpha2);
                    const float2 dlt = __ffma2_rn(u ? make_float2(cc.z, cc.w) : make_float2(cc.x, cc.y), make_float2(-1.f, -1.f), thr);
                    hx = __funnelshift_l(__float_as_uint(dlt.x), hx, 1);
                    hy = __funnelshift_l(__float_as_uint(dlt.y), hy, 1);
                }
                c4[q2] = make_float4(nz[0].x, nz[0].y, nz[1].x, nz[1].y);           // these cells belong to this task alone
            }
            // rare: record the hits
            uint32_t h = hx | (hy << 16);
            while (h) {
                const int b = __ffs(h) - 1;
                h &= h - 1;
                const int q = SW - 1 - (b & 15), hi = b >> 4;
                const float noise = reinterpret_cast<const float *>(c4)[2 * q + hi];
                const int x = x0 + q + hi * H;                                       // range bin within the strip
                const uint32_t d = dk + j;
                atomicOr(&words[x], 1u << (d & 31));
                noise_map[((size_t)f * Cp + d) * Sp + r0 + x] = noise;              // sparse: hit cells only
            }
        }
        __syncthreads();
        if ((k & 1) && tid < RT) {           // 32 Doppler rows done: one mask word per range bin
            mask[((size_t)f * (Cp / 32) + ((dk - 16) >> 5)) * Sp + r0 + tid] = words[tid];
            words[tid] = 0u;
        }
    }
}

template <int RT, int MINB, int SPT>
static cudaError_t run_cfar_walk_t(const PlanDev &p, const float *pmap, uint32_t *mask, float *noise_map, int nchunk, int n_frames, cudaStream_t st)
{
    using Sh = WalkShape<RT>;
    if (Sh::SMEM > 48 * 1024) {
        static bool configured_dev[kMaxDevices] = {false};
        bool &configured = configured_dev[current_device()];
        if (!configured) {
            cudaError_t e = cudaFuncSetAttribute(cfar_walk_kernel<RT, MINB, SPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Sh::SMEM);
            if (e != cudaSuccess) return e;
            configured = true;
        }
    }
    dim3 grid(p.Sp / RT, p.Cp / (16 * nchunk), n_frames);
    cfar_walk_kernel<RT, MINB, SPT><<<grid, Sh::NT, Sh::SMEM, st>>>(p, pmap, mask, noise_map, nchunk);
    return cudaGetLastError();
}

template <int RT, int MINB>
static cudaError_t run_cfar_walk(const PlanDev &p, const float *pmap, uint32_t *mask, float *noise_map, int nchunk, int n_frames, cudaStream_t st)
{
    switch (p.Sp) {
    case 256:  return run_cfar_walk_t<RT, MINB, 256>(p, pmap, mask, noise_map, nchunk, n_frames, st);
    case 512:  return run_cfar_walk_t<RT, MINB, 512>(p, pmap, mask, noise_map, nchunk, n_frames, st);
    case 1024: return run_cfar_walk_t<RT, MINB, 1024>(p, pmap, mask, noise_map, nchunk, n_frames, st);
    default:
        // 256-bin strips need Sp % 256 == 0, and every such Sp has its own specialisation above: no run-time-Sp form
        if constexpr (RT == 256) return cudaErrorInvalidValue;
        else return run_cfar_walk_t<RT, MINB, 0>(p, pmap, mask, noise_map, nchunk, n_frames, st);
    }
}

// ---------------------------------------------------------------------------
// K4a: ordered hit list per frame + batch-wide offsets (last CTA scans)
// ---------------------------------------------------------------------------
constexpr int kListNT = 256;

__global__ void __launch_bounds__(kListNT) list_kernel(PlanDev p, const uint32_t *__restrict__ mask, uint32_t *__restrict__ keys,
                                                       uint32_t *__restrict__ counts, uint32_t *__restrict__ offsets,
                                                       uint32_t *__restrict__ header, unsigned int *__restrict__ ticket,
                                                       int n_frames, int dense_cap)
{
    __shared__ uint32_t scan[kListNT / 32], tsum[kListNT / 32];
    __shared__ uint32_t total_s;
    __shared__ bool is_last;
    extern __shared__ uint32_t ordered[];                     // the frame's mask words in (range, doppler-word) order

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int f = blockIdx.x;
    const int Sp = p.Sp, Cp = p.Cp;
    const int wpr = Cp / 32;                                  // mask words per range bin
    const int nwords = wpr * Sp;
    const uint32_t *mf = mask + (size_t)f * nwords;
    uint32_t *kf = keys + (size_t)f * p.max_det;

    // the mask is stored [doppler word][range]; read it coalesced and transpose on the way into shared memory (one pad
    // word per 32 keeps the strided writes off a single bank) so that the ordered walk below is local
    for (int i = tid; i < nwords; i += kListNT) {
        const int w = i / Sp, r = i - w * Sp;
        const int o = r * wpr + w;
        ordered[o + (o >> 5)] = mf[i];
    }
    __syncthreads();

    // thread t owns the contiguous run [i0, i1) of the (range, doppler-word) ordered word sequence
    const int wpt = (nwords + kListNT - 1) / kListNT;
    const int i0 = tid * wpt, i1 = min(nwords, i0 + wpt);
    uint32_t cnt = 0;
#pragma unroll 8
    for (int i = i0; i < i1; ++i) cnt += __popc(ordered[i + (i >> 5)]);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) scan[warp] = incl;
    __syncthreads();
    if (tid == 0) {
        uint32_t s = 0;
        for (int w = 0; w < kListNT / 32; ++w) {
            const uint32_t v = scan[w];
            scan[w] = s;
            s += v;
        }
        total_s = s;
    }
    __syncthreads();
    uint32_t pos = scan[warp] + incl - cnt;
    if (cnt) {
        for (int i = i0; i < i1 && pos < (uint32_t)p.max_det; ++i) {
            uint32_t w = ordered[i + (i >> 5)];
            const uint32_t r = i / wpr, dbase = (i % wpr) * 32;
            while (w && pos < (uint32_t)p.max_det) {
                const int b = __ffs(w) - 1;
                w &= w - 1;
                kf[pos++] = (r << 16) | (dbase + b);
            }
        }
    }
    if (tid == 0) {
        counts[f] = total_s;
        __threadfence();
        const unsigned int done = atomicAdd(ticket, 1u);
        is_last = (done == (unsigned)n_frames - 1);
    }
    __syncthreads();
    if (!is_last) return;

    // ---- last CTA: exclusive scan of the clipped counts -> offsets[f], header ----
    __threadfence();
    uint32_t carry = 0, true_total = 0;                        // uniform across the block
    for (int base = 0; base < n_frames; base += kListNT) {
        const int i = base + tid;
        const uint32_t c = i < n_frames ? __ldcg(counts + i) : 0u;
        const uint32_t cc = min(c, (uint32_t)p.max_det);
        uint32_t inc = cc, ts = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ts += __shfl_xor_sync(0xffffffffu, ts, o);
        __syncthreads();                                       // scan[] / tsum[] free for reuse
        if (lane == 31) { scan[warp] = inc; tsum[warp] = ts; }
        __syncthreads();
        uint32_t wbase = 0, chunk = 0, tchunk = 0;
        for (int w = 0; w < kListNT / 32; ++w) {
            if (w < warp) wbase += scan[w];
            chunk += scan[w];
            tchunk += tsum[w];
        }
        if (i < n_frames) offsets[i] = carry + wbase + inc - cc;
        carry += chunk;
        true_total += tchunk;
    }
    if (tid == 0) {
        offsets[n_frames] = carry;
        header[0] = min(carry, (uint32_t)dense_cap);
        header[1] = true_total;
        header[2] = (uint32_t)n_frames;
        header[3] = (true_total != carry || carry > (uint32_t)dense_cap) ? 1u : 0u;
        ticket[0] = 0u;                                         // self-cleaning for the next batch
        ticket[1] = 0u;                                         // work cursor of measure_kernel
        ticket[2] = 0u;                                         // hit-row count of rows_kernel
    }
}

// ---------------------------------------------------------------------------
// K4b: detection records.  Chunks of up to kMeasG detections that share (frame, range bin) are measured together.
// ---------------------------------------------------------------------------
constexpr int kMeasNT = 256;
constexpr int kMeasWarps = kMeasNT / 32;
constexpr int kMeasG = 4;            // detections measured together (they share every range-spectrum row they read)
constexpr int kMeasQ = 2;            // antennas whose rows are in flight together
// Wide arrays, from this many antennas on: fused mode takes the selective re-FFT path (detect_uses_refft); otherwise a whole
// CTA (not one warp) measures a chunk ...
constexpr int kMeasWideA = 32;
constexpr int kMeasWideG = 32;       // ... of up to this many detections (kMeasG at a time in registers, rows re-read from L1)

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// The list is ordered by (frame, range, doppler), so the hits a target leaves in neighbouring Doppler cells of one
// range bin are consecutive.  In fused mode each of them needs one Doppler bin of the SAME A x C block of the range
// spectrum; a run of equal range bin is cut into chunks of kMeasG detections, and whoever measures a chunk reads every
// row once for all its detections.
struct MeasFrame {                   // cached frame lookup: list positions [fbeg, fend_raw) belong to frame f
    int f;
    uint32_t fbeg, fend_raw;
};
struct MeasChunk {
    int f, r, ng;
    uint32_t mykey;                  // lane j: key of the chunk's j-th detection (lanes >= ng: don't care)
    __device__ __forceinline__ int doppler(int j) const { return (int)(__shfl_sync(0xffffffffu, mykey, min(j, ng - 1)) & 0xffffu); }
};

__device__ __forceinline__ void lookup_frame(const uint32_t *__restrict__ offsets, int n_frames, uint32_t g, MeasFrame &fc)
{
    if (g >= fc.fbeg && g < fc.fend_raw) return;
    int lo = 0, hi = n_frames - 1;                                // largest f with offsets[f] <= g
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (offsets[mid] <= g) lo = mid; else hi = mid - 1;
    }
    fc.f = lo;
    fc.fbeg = offsets[lo];
    fc.fend_raw = offsets[lo + 1];
}

// Warp-collective: how many list positions directly before g (down to the frame's first, fbeg) have range bin r, i.e. the
// position of g inside its run of equal range bin.  kf[q] = key of list position q.  The predecessors are read 32 at a
// time, one per lane, so that finding the run costs one memory round trip instead of one per element.
__device__ __forceinline__ uint32_t run_back(const uint32_t *__restrict__ kf, uint32_t fbeg, uint32_t g, int r, int lane)
{
    uint32_t back = 0;
    for (uint32_t base = g;;) {
        const bool same = base >= fbeg + 1 + lane && (int)(kf[base - 1 - lane] >> 16) == r;
        const uint32_t m = __ballot_sync(0xffffffffu, same);
        const uint32_t n = m == 0xffffffffu ? 32u : (uint32_t)(__ffs(~m) - 1);
        back += n;
        if (n < 32u) return back;
        base -= 32u;
    }
}

// Warp-collective.  Returns false if list position g0 is not the head of a chunk.
template <int G>
__device__ __forceinline__ bool locate_chunk(const PlanDev &p, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ offsets,
                                             int n_frames, uint32_t total, uint32_t g0, int lane, MeasFrame &fc, MeasChunk &ch)
{
    lookup_frame(offsets, n_frames, g0, fc);
    const uint32_t fbeg = fc.fbeg, fend = min(fc.fend_raw, total);
    const uint32_t *kf = keys + (size_t)fc.f * p.max_det - fbeg;  // kf[g] = key of list position g
    const int r = (int)(kf[g0] >> 16);
    if (run_back(kf, fbeg, g0, r, lane) % G != 0) return false;   // every G-th detection of a run heads a chunk
    const uint32_t mykey = g0 + lane < fend ? kf[g0 + lane] : 0xffffffffu;      // lane j: key of list position g0 + j
    const uint32_t fm = __ballot_sync(0xffffffffu, g0 + lane < fend && (int)(mykey >> 16) == r);
    ch.f = fc.f;
    ch.r = r;
    static_assert(G <= 32, "a chunk's keys live one per lane");
    ch.ng = min(G, fm == 0xffffffffu ? 32 : __ffs(~fm) - 1);
    ch.mykey = mykey;
    return true;
}

// Warp-collective: antenna snapshots X[a] = Doppler bin d_j of antenna a at range bin r, for every detection j of the
// chunk and the antennas a_first, a_first + kMeasQ, ... in steps of a_step, written to xw[j * A + a].
// Cube mode copies them; fused mode re-derives them from the (already windowed) range spectrum: kMeasQ antennas x 256
// chirps (kMeasQ * 8 independent 8-byte loads per lane) are pulled into registers before anything is consumed — this is
// bound by memory latency, not by arithmetic — and every value then feeds kMeasG detections at a time; a longer chunk
// re-reads the same few KB from L1.  The summation order per (antenna, detection) is fixed: lane-strided partial sums
// in ascending chirp order, then the xor-butterfly.
__device__ __forceinline__ void snapshot_antennas(const PlanDev &p, const float2 *__restrict__ rs, const float2 *__restrict__ cube,
                                                  const MeasChunk &ch, int lane, int a_first, int a_step, float2 *xw)
{
    const int Sp = p.Sp, Cp = p.Cp, A = p.A, C = p.C;
    const int f = ch.f, r = ch.r, ng = ch.ng;
    if (cube != nullptr) {
        for (int j = 0; j < ng; ++j) {
            const int d = ch.doppler(j);
            for (int e = lane;; e += 32) {                        // e-th antenna of this caller's share, one per lane
                const int a0 = a_first + (e / kMeasQ) * a_step, a = a0 + e % kMeasQ;
                if (a0 >= A) break;
                if (a < A) xw[j * A + a] = cube[(((size_t)f * A + a) * Cp + d) * Sp + r];
            }
        }
        return;
    }
    const float2 *src0 = rs + (((size_t)f * A) * Sp + r) * (size_t)C;
    const size_t astride = (size_t)Sp * C;
    for (int a0 = a_first; a0 < A; a0 += a_step) {
        for (int jb = 0; jb < ng; jb += kMeasG) {
            int dj[kMeasG];
#pragma unroll
            for (int j = 0; j < kMeasG; ++j) dj[j] = ch.doppler(jb + j);
            const int nj = min(kMeasG, ng - jb);
            float sx[kMeasG][kMeasQ], sy[kMeasG][kMeasQ];
#pragma unroll
            for (int j = 0; j < kMeasG; ++j)
#pragma unroll
                for (int q = 0; q < kMeasQ; ++q) sx[j][q] = sy[j][q] = 0.f;
            for (int cc0 = 0; cc0 < C; cc0 += 256) {
                float2 v[kMeasQ][8];
#pragma unroll
                for (int q = 0; q < kMeasQ; ++q) {
                    const float2 *sa = src0 + (size_t)min(a0 + q, A - 1) * astride;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int c = cc0 + lane + 32 * i;
                        v[q][i] = c < C ? sa[c] : make_float2(0.f, 0.f);
                    }
                }
#pragma unroll
                for (int j = 0; j < kMeasG; ++j) {
                    if (j < nj) {
                        const int d = dj[j];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int c = cc0 + lane + 32 * i;
                            const float2 w = p.tw_d[(c * d) & (Cp - 1)];
#pragma unroll
                            for (int q = 0; q < kMeasQ; ++q) {
                                sx[j][q] += v[q][i].x * w.x - v[q][i].y * w.y;
                                sy[j][q] += v[q][i].x * w.y + v[q][i].y * w.x;
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < kMeasG; ++j)
#pragma unroll
                for (int q = 0; q < kMeasQ; ++q)
                    if (j < nj) {                                 // warp-uniform
                        const float tx = warp_sum(sx[j][q]), ty = warp_sum(sy[j][q]);
                        if (lane == 0 && a0 + q < A) xw[(jb + j) * A + a0 + q] = make_float2(tx, ty);
                    }
        }
    }
}

// The 3x3 grouping test of every detection path: is neighbour `cell` (0..8, row-major over range offsets -1..1 x Doppler
// offsets -1..1; 4 is the detection itself) of detection (r, d) with power pw a detected cell that outranks it?  Doppler
// wraps, range clamps; larger power outranks, equal power -> the lower (r, d).  A detection is a peak (strict 3x3 maximum)
// when none of its eight neighbours outranks it.  pf / mf: the frame's power map and CFAR mask.
__device__ __forceinline__ bool neighbour_outranks(const PlanDev &p, const float *__restrict__ pf, const uint32_t *__restrict__ mf,
                                                   int r, int d, float pw, int cell)
{
    const int Sp = p.Sp, Cp = p.Cp;
    const int rr = r + cell / 3 - 1;
    const int dd = (d + cell % 3 - 1 + Cp) & (Cp - 1);
    if (rr < 0 || rr >= Sp) return false;
    const uint32_t w = mf[(size_t)(dd >> 5) * Sp + rr];
    if (!((w >> (dd & 31)) & 1u)) return false;
    const float pn = pf[(size_t)dd * Sp + rr];
    const uint32_t key = ((uint32_t)r << 16) | (uint32_t)d, kn = ((uint32_t)rr << 16) | (uint32_t)dd;
    return (pn > pw) || (pn == pw && kn < key);
}

// The arg-max tie rule of the angle spectrum: larger power wins, equal power -> lower bin (strict >, first wins).
__device__ __forceinline__ void argmax_update(float m, int k, float &best, int &bestk)
{
    if (m > best || (m == best && k < bestk)) { best = m; bestk = k; }
}

// Arg-max over aligned groups of WIDTH lanes (xor butterfly); every lane of a group ends with the group's result.
template <int WIDTH = 32>
__device__ __forceinline__ void warp_argmax(float &best, int &bestk)
{
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int ok = __shfl_xor_sync(0xffffffffu, bestk, o);
        argmax_update(ob, ok, best, bestk);
    }
}

__device__ __forceinline__ void angle_bin_power(const float2 *xj, const float2 *twa, int A, int n_theta, int k, float &best, int &bestk)
{
    float yx = 0.f, yy = 0.f;
    for (int a = 0; a < A; ++a) {
        const float2 v = xj[a];
        const float2 w = twa[(k * a) & (n_theta - 1)];
        yx += v.x * w.x - v.y * w.y;
        yy += v.x * w.y + v.y * w.x;
    }
    argmax_update(yx * yx + yy * yy, k, best, bestk);
}

__device__ __forceinline__ void write_record(const PlanDev &p, mmw_detection *__restrict__ dense, uint32_t g, int f, int r, int d, float pw,
                                             float noise, int bestk, bool is_peak)
{
    const int kw = bestk < p.n_theta / 2 ? bestk : bestk - p.n_theta;
    float sn = (float)kw * p.lambda_over_d / (float)p.n_theta;
    sn = fminf(1.f, fmaxf(-1.f, sn));
    mmw_detection o;
    o.frame = (uint32_t)f + p.frame_offset;
    o.range_bin = (uint16_t)r;
    o.doppler_bin = (uint16_t)d;
    o.power = pw;
    o.noise = noise;
    o.angle_bin = (int16_t)kw;
    o.flags = is_peak ? MMW_FLAG_PEAK : 0;
    o.angle_rad = asinf(sn);
    dense[g] = o;
}

// Warp-collective: records of all (<= kMeasG <= 4) detections of a chunk.  Lane l looks at neighbour l % 8 of detection
// l / 8, so the grouping test of the whole chunk costs two memory round trips (mask words, then the neighbours' powers)
// instead of two per detection; the angle spectra come from the snapshots in shared memory.
__device__ __forceinline__ void emit_chunk(const PlanDev &p, const float *__restrict__ pf, const uint32_t *__restrict__ mf,
                                           const float *__restrict__ noise_map, const MeasChunk &ch, int lane, const float2 *xw,
                                           const float2 *twa, mmw_detection *__restrict__ dense, uint32_t g0)
{
    static_assert(kMeasG * 8 <= 32, "one lane per (detection, neighbour)");
    const int Sp = p.Sp, Cp = p.Cp, A = p.A;
    const int j = lane >> 3, nb = lane & 7;
    const bool active = j < ch.ng;
    const int r = ch.r;
    const int d = (int)(__shfl_sync(0xffffffffu, ch.mykey, min(j, ch.ng - 1)) & 0xffffu);
    const float pw = active ? pf[(size_t)d * Sp + r] : 0.f;
    const float noise = (active && nb == 0) ? noise_map[((size_t)ch.f * Cp + d) * Sp + r] : 0.f;
    const bool worse = active && neighbour_outranks(p, pf, mf, r, d, pw, nb < 4 ? nb : nb + 1);     // nb skips the centre
    const uint32_t wm = __ballot_sync(0xffffffffu, worse);
    const bool is_peak = ((wm >> (8 * j)) & 0xffu) == 0u;
    int my_bestk = 0;
    for (int jj = 0; jj < ch.ng; ++jj) {
        float best = -1.f;
        int bestk = 0;
        for (int k = lane; k < p.n_theta; k += 32) angle_bin_power(xw + jj * A, twa, A, p.n_theta, k, best, bestk);
        warp_argmax(best, bestk);
        if (j == jj) my_bestk = bestk;
    }
    if (active && nb == 0) write_record(p, dense, g0 + j, ch.f, r, d, pw, noise, my_bestk, is_peak);
}

// narrow form (A < kMeasWideA): one warp per chunk.
// List positions are handed out from a global cursor (reset by list_kernel) in blocks of up to kMeasBlk consecutive
// positions: chunk heads are scattered irregularly through the list, so a static assignment leaves most warps of an SM
// without one, and the kernel is bound by memory round trips, so everything that can be is done for a whole block at
// once — one lane-parallel read brings the block's keys, shuffles find every chunk head in it, and only the per-chunk
// measurements remain serial.
constexpr int kMeasBlk = 32 - kMeasG;                             // + kMeasG - 1 keys of look-ahead fit the 32 lanes

__global__ void __launch_bounds__(kMeasNT) measure_kernel(PlanDev p, const float2 *__restrict__ rs, const float2 *__restrict__ cube,
                                                          const float *__restrict__ pmap, const float *__restrict__ noise_map,
                                                          const uint32_t *__restrict__ mask, const uint32_t *__restrict__ keys,
                                                          const uint32_t *__restrict__ offsets, mmw_detection *__restrict__ dense,
                                                          unsigned int *__restrict__ cursor, int n_frames, int dense_cap)
{
    extern __shared__ __align__(16) unsigned char smem[];
    float2 *twa = reinterpret_cast<float2 *>(smem);                 // [n_theta]
    float2 *xs = twa + p.n_theta;                                   // [warps][kMeasG][A]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Sp = p.Sp, Cp = p.Cp, A = p.A;
    for (int i = tid; i < p.n_theta; i += kMeasNT) twa[i] = p.tw_a[i];
    __syncthreads();

    const uint32_t total = min(offsets[n_frames], (uint32_t)dense_cap);
    float2 *xw = xs + warp * (kMeasG * A);
    const uint32_t blk = min((uint32_t)kMeasBlk, max(1u, total / (uint32_t)(gridDim.x * kMeasWarps)));
    MeasFrame fc = {0, 0u, 0u};
    for (;;) {
        uint32_t gblk = 0;
        if (lane == 0) gblk = atomicAdd(cursor, blk);
        gblk = __shfl_sync(0xffffffffu, gblk, 0);
        if (gblk >= total) break;
        const uint32_t gblk_end = min(gblk + blk, total);
        for (uint32_t g = gblk; g < gblk_end;) {                     // one segment per frame the block touches
            lookup_frame(offsets, n_frames, g, fc);
            const uint32_t fbeg = fc.fbeg, fend = min(fc.fend_raw, total);
            const uint32_t seg_end = min(gblk_end, fend);
            const uint32_t *kf = keys + (size_t)fc.f * p.max_det - fbeg;      // kf[q] = key of list position q
            // keys of positions g .. g+31 (the segment and its look-ahead), and the predecessors of g, in one round trip
            const bool valid = g + lane < fend;
            const uint32_t mykey = valid ? kf[g + lane] : 0xffffffffu;
            const int myr = (int)(mykey >> 16);
            const uint32_t back = run_back(kf, fbeg, g, __shfl_sync(0xffffffffu, myr, 0), lane);   // how far the run of g reaches back
            // index of every position inside its run of equal range bin -> chunk heads (every kMeasG-th)
            const int prev_r = __shfl_up_sync(0xffffffffu, myr, 1);
            const uint32_t starts = __ballot_sync(0xffffffffu, lane > 0 && valid && myr != prev_r);
            const uint32_t below = starts & (0xffffffffu >> (31 - lane));         // run starts at lanes <= mine
            const uint32_t idx = below ? (uint32_t)(lane - (31 - __clz(below))) : back + lane;
            uint32_t heads = __ballot_sync(0xffffffffu, g + lane < seg_end && idx % kMeasG == 0);
            const float *pf = pmap + (size_t)fc.f * Cp * Sp;
            const uint32_t *mf = mask + (size_t)fc.f * (Cp / 32) * Sp;
            while (heads) {
                const int h = __ffs(heads) - 1;
                heads &= heads - 1;
                MeasChunk ch;
                ch.f = fc.f;
                ch.r = __shfl_sync(0xffffffffu, myr, h);
                const uint32_t same = __ballot_sync(0xffffffffu, valid && myr == ch.r) >> h;      // bit j: position h + j
                ch.ng = min(kMeasG, same == 0xffffffffu ? 32 : __ffs(~same) - 1);
                ch.mykey = __shfl_sync(0xffffffffu, mykey, (h + lane) & 31);                       // lane j: position h + j
                snapshot_antennas(p, rs, cube, ch, lane, 0, kMeasQ, xw);
                __syncwarp();
                emit_chunk(p, pf, mf, noise_map, ch, lane, xw, twa, dense, g + h);
                __syncwarp();
            }
            g = seg_end;
        }
    }
}

// wide form (A >= kMeasWideA, e.g. the 192-antenna imaging cube: 786 KB of range spectrum per range bin): a whole CTA
// measures a chunk of up to kMeasWideG detections — the warps split the antennas of the snapshot and the bins of the
// angle spectrum — so the serial chain of memory round trips per chunk is eight times shorter and a long run of hits in
// one range bin pulls its rows from HBM once.
__global__ void __launch_bounds__(kMeasNT) measure_wide_kernel(PlanDev p, const float2 *__restrict__ rs, const float2 *__restrict__ cube,
                                                               const float *__restrict__ pmap, const float *__restrict__ noise_map,
                                                               const uint32_t *__restrict__ mask, const uint32_t *__restrict__ keys,
                                                               const uint32_t *__restrict__ offsets, mmw_detection *__restrict__ dense,
                                                               unsigned int *__restrict__ cursor, int n_frames, int dense_cap)
{
    extern __shared__ __align__(16) unsigned char smem[];
    float2 *twa = reinterpret_cast<float2 *>(smem);                 // [n_theta]
    float2 *xs = twa + p.n_theta;                                   // [kMeasWideG][A], shared by the CTA
    __shared__ uint32_t s_g0;
    __shared__ float s_best[kMeasWarps];
    __shared__ int s_bestk[kMeasWarps];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Sp = p.Sp, Cp = p.Cp, A = p.A;
    for (int i = tid; i < p.n_theta; i += kMeasNT) twa[i] = p.tw_a[i];
    const uint32_t total = min(offsets[n_frames], (uint32_t)dense_cap);
    MeasFrame fc = {0, 0u, 0u};
    for (;;) {
        __syncthreads();                                             // s_g0 / xs / s_best free again (and twa loaded)
        if (tid == 0) s_g0 = atomicAdd(cursor, 1u);
        __syncthreads();
        const uint32_t g0 = s_g0;
        if (g0 >= total) break;
        MeasChunk ch;                                                // every warp derives the same chunk (uniform control flow)
        if (!locate_chunk<kMeasWideG>(p, keys, offsets, n_frames, total, g0, lane, fc, ch)) continue;
        const float *pf = pmap + (size_t)ch.f * Cp * Sp;
        const uint32_t *mf = mask + (size_t)ch.f * (Cp / 32) * Sp;
        snapshot_antennas(p, rs, cube, ch, lane, warp * kMeasQ, kMeasWarps * kMeasQ, xs);
        __syncthreads();
        for (int j = 0; j < ch.ng; ++j) {
            float best = -1.f;
            int bestk = 0;
            for (int k = tid; k < p.n_theta; k += kMeasNT) angle_bin_power(xs + j * A, twa, A, p.n_theta, k, best, bestk);
            warp_argmax(best, bestk);
            if (lane == 0) { s_best[warp] = best; s_bestk[warp] = bestk; }
            __syncthreads();
            if (warp == 0) {
                best = lane < kMeasWarps ? s_best[lane] : -1.f;
                bestk = lane < kMeasWarps ? s_bestk[lane] : 0x7fffffff;
                warp_argmax(best, bestk);
                const int d = ch.doppler(j);
                const float pw = pf[(size_t)d * Sp + ch.r];
                const float noise = noise_map[((size_t)ch.f * Cp + d) * Sp + ch.r];
                const bool worse = lane < 9 && lane != 4 && neighbour_outranks(p, pf, mf, ch.r, d, pw, lane);
                const bool is_peak = __ballot_sync(0xffffffffu, worse) == 0u;
                if (lane == 0) write_record(p, dense, g0 + j, ch.f, ch.r, d, pw, noise, bestk, is_peak);
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// wide arrays, fused mode: hit rows -> (K2x doppler_extract_kernel, mmw_pipeline.cu) -> angle FFT + records
// ---------------------------------------------------------------------------
// rows_kernel: every (frame, range bin) that has at least one detection, found as the heads of the runs of equal range bin
// in the ordered key list.  The order of `rows` is whatever the atomics give; nothing downstream depends on it (each row is
// transformed on its own, and a detection's slot in `snap` is its position in the dense list).
__global__ void __launch_bounds__(256) rows_kernel(PlanDev p, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ offsets,
                                                   uint4 *__restrict__ rows, unsigned int *__restrict__ n_rows, int n_frames, int dense_cap)
{
    const uint32_t total = min(offsets[n_frames], (uint32_t)dense_cap);
    MeasFrame fc = {0, 0u, 0u};
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
        lookup_frame(offsets, n_frames, g, fc);
        const uint32_t *kf = keys + (size_t)fc.f * p.max_det - fc.fbeg;
        const uint32_t r = kf[g] >> 16;
        if (g == fc.fbeg || (kf[g - 1] >> 16) != r) rows[atomicAdd(n_rows, 1u)] = make_uint4((uint32_t)fc.f, r, g, 0u);
    }
}

// angle_fft_kernel: the NTH-point angle spectrum of every detection as a real FFT (the per-detection kernels evaluate it as a
// DFT, NTH * A complex MACs per detection: 0.4 MFLOP at A = 192, more than the rest of the record put together), its arg-max
// (strict >, first wins), the 3x3 grouping flag and the 24-byte record.  Same scheme as the Doppler kernels: a warp owns its
// rows outright — lanes = ROWS detections x SUBS butterflies of one detection — the two passes meet in a warp-private
// shared-memory row, no CTA barrier after the twiddle table is loaded.
template <int NTH, int R1, int R2>
struct AngleWarp {
    static constexpr int kMinR = R1 < R2 ? R1 : R2;
    static constexpr int kSubs = kMinR > 16 ? 16 : kMinR;
    static constexpr int kRows = 32 / kSubs;
    static constexpr int kU1 = R2 / kSubs;
    static constexpr int kU2 = R1 / kSubs;
    static constexpr int kRowStride = NTH + R1;                      // float2: NTH points + one pad per run of R2
    static constexpr int kWarps = 8;
    static constexpr int kBytes = NTH * 8 + kWarps * kRows * kRowStride * 8;
    static_assert(kSubs >= 8, "the eight 3x3 neighbours of a detection are tested by eight lanes of its group");
};

template <int NTH, int R1, int R2>
__global__ void __launch_bounds__(256) angle_fft_kernel(PlanDev p, const float2 *__restrict__ snap, const float *__restrict__ pmap,
                                                        const float *__restrict__ noise_map, const uint32_t *__restrict__ mask,
                                                        const uint32_t *__restrict__ keys, const uint32_t *__restrict__ offsets,
                                                        mmw_detection *__restrict__ dense, int n_frames, int dense_cap)
{
    static_assert(R1 * R2 == NTH, "plan");
    using L = AngleWarp<NTH, R1, R2>;
    constexpr int SUBS = L::kSubs, ROWS = L::kRows, U1 = L::kU1, U2 = L::kU2;
    constexpr int LR1 = ilog2(R1), LR2 = ilog2(R2);
    extern __shared__ __align__(16) unsigned char smem[];
    float2 *tw = reinterpret_cast<float2 *>(smem);                   // exp(-2 pi i k / NTH), natural order
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float2 *ring = tw + NTH + (size_t)warp * ROWS * L::kRowStride;
    const int row = lane / SUBS, sub = lane % SUBS;
    const int Sp = p.Sp, Cp = p.Cp, A = p.A;
    for (int i = tid; i < NTH; i += 256) tw[i] = p.tw_a[i];
    __syncthreads();                                                 // the only CTA-wide barrier

    const uint32_t total = min(offsets[n_frames], (uint32_t)dense_cap);
    const uint32_t gw = (blockIdx.x * L::kWarps + warp) * ROWS, gstep = gridDim.x * L::kWarps * ROWS;
    float2 *r = ring + row * L::kRowStride;
    MeasFrame fc = {0, 0u, 0u};
#pragma unroll 1
    for (uint32_t g0 = gw; g0 < total; g0 += gstep) {
        const uint32_t g = g0 + row;
        const bool live = g < total;
        // the snapshot, zero-padded to NTH (coalesced: the SUBS lanes of a group read neighbouring antennas)
        const float2 *src = snap + (size_t)(live ? g : 0) * A;
#pragma unroll 4
        for (int i = sub; i < NTH; i += SUBS) r[i] = (live && i < A) ? src[i] : make_float2(0.f, 0.f);
        __syncwarp();
        // pass 1: every input into registers first (the outputs overwrite other threads' inputs)
        float2 x[U1][R1];
#pragma unroll
        for (int u = 0; u < U1; ++u) {
            const int n2 = sub + u * SUBS;
#pragma unroll
            for (int m = 0; m < R1; ++m) x[u][m] = r[n2 + m * R2];
        }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < U1; ++u) {
            const int n2 = sub + u * SUBS;
            dft_regs<R1>(x[u]);
            r[n2] = x[u][0];
#pragma unroll
            for (int k1 = 1; k1 < R1; ++k1) r[k1 * (R2 + 1) + n2] = cmul(x[u][bitrev(k1, LR1)], tw[(n2 * k1) & (NTH - 1)]);
        }
        __syncwarp();
        // pass 2 + arg-max of |Y|^2: larger power wins, equal power -> lower bin
        float best = -1.f;
        int bestk = 0;
#pragma unroll
        for (int u = 0; u < U2; ++u) {
            const int k1 = sub + u * SUBS;
            float2 y[R2];
            const float2 *wi = r + k1 * (R2 + 1);
#pragma unroll
            for (int n2 = 0; n2 < R2; ++n2) y[n2] = wi[n2];
            dft_regs<R2>(y);
#pragma unroll
            for (int k2 = 0; k2 < R2; ++k2) {
                const float2 v = y[bitrev(k2, LR2)];
                argmax_update(v.x * v.x + v.y * v.y, k1 + R1 * k2, best, bestk);
            }
        }
        warp_argmax<SUBS>(best, bestk);
        __syncwarp();                                                // the row is free for the next detection
        // record: lanes 0..7 of the group look at the eight 3x3 neighbours
        bool worse = false;
        int f = 0, rb = 0, d = 0;
        float pw = 0.f, noise = 0.f;
        if (live) {
            lookup_frame(offsets, n_frames, g, fc);
            f = fc.f;
            const uint32_t key = keys[(size_t)f * p.max_det + (g - fc.fbeg)];
            rb = (int)(key >> 16);
            d = (int)(key & 0xffffu);
            const float *pf = pmap + (size_t)f * Cp * Sp;
            pw = pf[(size_t)d * Sp + rb];
            if (sub == 0) noise = noise_map[((size_t)f * Cp + d) * Sp + rb];
            if (sub < 8) worse = neighbour_outranks(p, pf, mask + (size_t)f * (Cp / 32) * Sp, rb, d, pw, sub < 4 ? sub : sub + 1);
        }
        const uint32_t wm = __ballot_sync(0xffffffffu, worse);
        const bool is_peak = ((wm >> (row * SUBS)) & 0xffu) == 0u;
        if (live && sub == 0) write_record(p, dense, g, f, rb, d, pw, noise, bestk, is_peak);
    }
}

template <int NTH, int R1, int R2>
static cudaError_t run_angle_fft(const PlanDev &p, const DetectBuffers &b, int n_frames, int dense_cap, int sm_count, cudaStream_t st)
{
    using L = AngleWarp<NTH, R1, R2>;
    const long long want = ((long long)dense_cap + L::kWarps * L::kRows - 1) / (L::kWarps * L::kRows);
    const int grid = (int)(want < (long long)sm_count * 4 ? (want < 1 ? 1 : want) : (long long)sm_count * 4);
    angle_fft_kernel<NTH, R1, R2><<<grid, 256, L::kBytes, st>>>(p, b.snap, b.pmap, b.noise_map, b.mask, b.keys, b.offsets, b.dense, n_frames, dense_cap);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// merge of gathered per-rank result blocks (rank 0, after the NCCL gather)
// ---------------------------------------------------------------------------
constexpr int kMergeSplit = 8;       // CTAs per rank

__global__ void __launch_bounds__(256) merge_kernel(const unsigned char *__restrict__ gathered, int n_ranks, size_t stride_bytes,
                                                    unsigned char *__restrict__ merged, int merged_cap)
{
    const int r = blockIdx.x, part = blockIdx.y;
    uint32_t off = 0, tot_written = 0, tot_true = 0, tot_frames = 0, ovf = 0;
    for (int i = 0; i < n_ranks; ++i) {
        const uint32_t *hd = reinterpret_cast<const uint32_t *>(gathered + (size_t)i * stride_bytes);
        const uint32_t cap_i = (uint32_t)((stride_bytes - MMW_RESULT_HEADER_BYTES) / sizeof(mmw_detection));
        const uint32_t n = min(hd[0], cap_i);
        if (i < r) off += n;
        tot_written += n;
        tot_true += hd[1];
        tot_frames += hd[2];
        ovf |= hd[3] | (hd[0] > cap_i ? 1u : 0u);
    }
    const uint32_t *hd = reinterpret_cast<const uint32_t *>(gathered + (size_t)r * stride_bytes);
    const uint32_t cap_r = (uint32_t)((stride_bytes - MMW_RESULT_HEADER_BYTES) / sizeof(mmw_detection));
    const uint32_t n = min(hd[0], cap_r);
    // 24-byte records as three 8-byte words
    const uint2 *src = reinterpret_cast<const uint2 *>(gathered + (size_t)r * stride_bytes + MMW_RESULT_HEADER_BYTES);
    uint2 *dst = reinterpret_cast<uint2 *>(merged + MMW_RESULT_HEADER_BYTES);
    for (uint32_t i = part * 256 + threadIdx.x; i < 3 * n; i += kMergeSplit * 256) {
        const uint32_t rec = off + i / 3;
        if (rec < (uint32_t)merged_cap) dst[(size_t)off * 3 + i] = src[i];
    }
    if (r == 0 && part == 0 && threadIdx.x == 0) {
        uint32_t *out = reinterpret_cast<uint32_t *>(merged);
        out[0] = min(tot_written, (uint32_t)merged_cap);
        out[1] = tot_true;
        out[2] = tot_frames;
        out[3] = (ovf || tot_written > (uint32_t)merged_cap) ? 1u : 0u;
    }
}

cudaError_t launch_merge(const unsigned char *gathered, int n_ranks, size_t stride_bytes, unsigned char *merged, int merged_cap,
                         cudaStream_t st)
{
    merge_kernel<<<dim3(n_ranks, kMergeSplit), 256, 0, st>>>(gathered, n_ranks, stride_bytes, merged, merged_cap);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
static int cfar_smem_bytes(const PlanDev &p)
{
    const int tw_ = kCfarRT + 2 * ((p.win_r_half + 3) & ~3), th_ = kCfarDT + 2 * p.win_d_half;
    return (th_ * tw_ + 2 * th_ * kCfarRS) * 4 + kCfarRT * 4;
}

// The default window takes the walk form (every plan_supported shape has Sp % 64 == 0 and Cp % 32 == 0); the tiled
// cfar_kernel serves every other window.
cudaError_t launch_cfar(const PlanDev &p, const float *pmap, uint32_t *mask, float *noise_map, int n_frames, int sm_count, cudaStream_t st)
{
    const bool fixed = p.guard_r == 2 && p.guard_d == 2 && p.win_r_half == 10 && p.win_d_half == 6;
    if (fixed && p.Sp % 64 == 0 && p.Cp % 32 == 0) {
        // walk form.  Longer Doppler segments amortise the 12-row run-in (28 input rows for the first 16 outputs, 16
        // after that), wider strips the 24-column halo; both are traded against having enough CTAs for every SM.
        const long long cells = (long long)n_frames * p.Sp * p.Cp;
        const long long want = (long long)sm_count * 8;
        int rt = 64;
        if (p.Sp % 128 == 0 && cells / (128 * 32) >= want) rt = 128;
        if (p.Sp % 256 == 0 && cells / (256 * 32) >= want) rt = 256;
        int nchunk = 2;
        while (nchunk < 8 && p.Cp % (32 * nchunk) == 0 && cells / ((long long)rt * 32 * nchunk) >= want) nchunk *= 2;
        switch (rt) {
        case 256: return run_cfar_walk<256, 3>(p, pmap, mask, noise_map, nchunk, n_frames, st);
        case 128: return run_cfar_walk<128, 5>(p, pmap, mask, noise_map, nchunk, n_frames, st);
        default:  return run_cfar_walk<64, 8>(p, pmap, mask, noise_map, nchunk, n_frames, st);
        }
    }
    const int bytes = cfar_smem_bytes(p);
    static int configured_dev[kMaxDevices] = {0};
    int &configured = configured_dev[current_device()];
    if (bytes > configured) {
        cudaError_t e = cudaFuncSetAttribute(cfar_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        configured = bytes;
    }
    dim3 grid((p.Sp + kCfarRT - 1) / kCfarRT, p.Cp / kCfarDT, n_frames);
    cfar_kernel<<<grid, kCfarNT, bytes, st>>>(p, pmap, mask, noise_map);
    return cudaGetLastError();
}

int record_kernel_args(const void *func)
{
    if (func == (const void *)measure_kernel || func == (const void *)measure_wide_kernel) return 12;
    if (func == (const void *)angle_fft_kernel<64, 8, 8> || func == (const void *)angle_fft_kernel<128, 8, 16> ||
        func == (const void *)angle_fft_kernel<256, 16, 16>)
        return 10;
    return 0;
}

// Wide arrays in fused mode take the selective re-FFT path (rows_kernel -> doppler_extract_kernel -> angle_fft_kernel);
// everything else takes a per-detection kernel.  PlanDev.detect_path (mmw_set_detect_path) forces either path.  Cube mode
// has no range spectrum to re-transform and always measures per detection, and so does a context without the re-FFT
// buffers (have_refft_buffers: rows and snap allocated).
bool detect_uses_refft(const PlanDev &p, bool have_refft_buffers)
{
    if (p.keep_cube || !have_refft_buffers || p.detect_path == MMW_DETECT_PER_CELL) return false;
    return p.A >= kMeasWideA || p.detect_path == MMW_DETECT_REFFT;
}

cudaError_t launch_detect(const PlanDev &p, const DetectBuffers &b, int n_frames, int dense_cap, int sm_count, cudaStream_t st)
{
    const int nwords = p.Sp * p.Cp / 32;
    const int list_bytes = (nwords + nwords / 32 + 1) * 4;
    static int list_configured_dev[kMaxDevices] = {0};
    int &list_configured = list_configured_dev[current_device()];
    cudaError_t e;
    if (list_bytes > list_configured) {
        e = cudaFuncSetAttribute(list_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, list_bytes);
        if (e != cudaSuccess) return e;
        list_configured = list_bytes;
    }
    list_kernel<<<n_frames, kListNT, list_bytes, st>>>(p, b.mask, b.keys, b.counts, b.offsets, b.header, b.ticket, n_frames, dense_cap);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // re-FFT path: one more Doppler FFT of the rows that have hits, then the angle spectra as FFTs
    if (detect_uses_refft(p, b.rows != nullptr && b.snap != nullptr)) {
        const int rgrid = (dense_cap + 255) / 256 < sm_count * 4 ? (dense_cap + 255) / 256 : sm_count * 4;
        rows_kernel<<<rgrid < 1 ? 1 : rgrid, 256, 0, st>>>(p, b.keys, b.offsets, b.rows, b.ticket + 2, n_frames, dense_cap);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        e = launch_doppler_extract(p, b.rs, b.keys, b.offsets, b.rows, b.ticket + 2, b.snap, dense_cap, n_frames * p.Sp, st);
        if (e != cudaSuccess) return e;
        switch (p.n_theta) {
        case 64:  return run_angle_fft<64, 8, 8>(p, b, n_frames, dense_cap, sm_count, st);
        case 128: return run_angle_fft<128, 8, 16>(p, b, n_frames, dense_cap, sm_count, st);
        case 256: return run_angle_fft<256, 16, 16>(p, b, n_frames, dense_cap, sm_count, st);
        default:  return cudaErrorInvalidValue;
        }
    }
    const bool wide = p.A >= kMeasWideA;
    const int bytes = p.n_theta * 8 + (wide ? kMeasWideG : kMeasWarps * kMeasG) * p.A * 8;
    static int configured_dev[kMaxDevices][2] = {{0}};
    int *configured = configured_dev[current_device()];
    if (bytes > configured[wide]) {
        e = wide ? cudaFuncSetAttribute(measure_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
                 : cudaFuncSetAttribute(measure_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        configured[wide] = bytes;
    }
    // persistent grids sized for the resident CTAs; a one- or two-frame batch (latency mode) cannot feed that many and
    // pays for every CTA it launches, so the grid also scales with the frame count
    const int by_frames = n_frames * 64 < sm_count ? sm_count : n_frames * 64;
    const int grid_wide = sm_count * 2 < by_frames ? sm_count * 2 : by_frames;
    const int grid_narrow = sm_count * 4 < by_frames ? sm_count * 4 : by_frames;
    if (wide)
        measure_wide_kernel<<<grid_wide, kMeasNT, bytes, st>>>(p, b.rs, p.keep_cube ? b.cube : nullptr, b.pmap, b.noise_map, b.mask,
                                                                  b.keys, b.offsets, b.dense, b.ticket + 1, n_frames, dense_cap);
    else
        measure_kernel<<<grid_narrow, kMeasNT, bytes, st>>>(p, b.rs, p.keep_cube ? b.cube : nullptr, b.pmap, b.noise_map, b.mask, b.keys,
                                                             b.offsets, b.dense, b.ticket + 1, n_frames, dense_cap);
    return cudaGetLastError();
}

}  // namespace mmw
