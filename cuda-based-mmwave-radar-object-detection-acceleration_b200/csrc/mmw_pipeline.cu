// mmw_pipeline.cu — stages 1 and 2 of the batched radar chain (the two FFT kernels) for sm_100a.
//
//   K1 range_fft_kernel    int16 IIQQ unpack + range window + Sp-point FFT per (chirp, antenna);
//                          output written corner-turned ([ant][range][chirp]) and pre-multiplied
//                          by the Doppler window.                  (replaces acceleration.cu:91-150)
//   K2 doppler_fft_kernel  Cp-point FFT across chirps per (range, antenna), |X|^2 accumulated over
//                          antennas in registers -> power map; Doppler cube optional.
//   (K3 cfar_kernel, K4a list_kernel, K4b measure_kernel: mmw_detect.cu)
//
// Both FFT kernels use the same scheme: a tile is BT transforms x N points held in shared
// memory, staged in by 1-D TMA bulk copies (one contiguous row per transform), the 32 lanes
// of a warp are 32 different transforms ("lane = batch"), and the transform is a two-pass
// (R1 x R2) decimation-in-frequency whose radix-R1 / radix-R2 butterflies run entirely in
// registers (fft_regs.cuh).  Because lanes are batch elements, the final pass writes the
// corner-turned layout directly with fully coalesced stores: the transpose never exists as a
// separate step and never round-trips HBM.
//
// Both kernels are persistent (grid = resident CTAs; K1 takes its tiles from a counter, K2 at a fixed stride) and
// software-pipelined: the TMA copies of the next tile are issued as soon as the staging buffer
// of the current one has been consumed, so the copy latency hides behind the second FFT pass.
#include <stdlib.h>

#include "fft_regs.cuh"
#include "mmw_common.cuh"

namespace mmw {

// Pass-1 twiddles are stored in the order pass 1 consumes them: entry (n2, k1) = W_N^(n2*k1) sits at
// float2 index ((n2 >> 1) * R1 + k1) * 2 + (n2 & 1), so that the two butterflies of a pair share one
// 16-byte load and every address is a compile-time offset from a per-butterfly base.
__host__ __device__ constexpr int tw1_index(int n2, int k1, int R1) { return ((n2 >> 1) * R1 + k1) * 2 + (n2 & 1); }

void plan_radices(int n, int *r1, int *r2)
{
    switch (n) {
    case 64:   *r1 = 8;  *r2 = 8;  break;
    case 128:  *r1 = 8;  *r2 = 16; break;
    case 256:  *r1 = 16; *r2 = 16; break;
    case 512:  *r1 = 16; *r2 = 32; break;
    default:   *r1 = 32; *r2 = 32; break;     // 1024
    }
}

// K1's tile counter (PlanDev.sched: {next tile, CTAs retired}).  The last CTA to retire puts both back to zero for the next
// launch on the stream (launches that share the counter pair are stream-ordered).
__device__ __forceinline__ void sched_retire(unsigned int *ctr)
{
    __threadfence();
    if (atomicAdd(&ctr[1], 1u) == gridDim.x - 1u) {
        ctr[0] = 0u;
        ctr[1] = 0u;
    }
}

// ---------------------------------------------------------------------------
// K1: range FFT
// ---------------------------------------------------------------------------
template <int N, int BT, bool BASE = false>
struct RangeSmem {
    static constexpr int kStageStride = 4 * N + 16;                 // bytes per staged int16 row
    static constexpr int kOffTw = 16;
    static constexpr int kOffWin = kOffTw + 8 * N;
    static constexpr int kOffStage = kOffWin + 4 * N;
    static constexpr int kStageBytes = BT * kStageStride;
    static constexpr int kOffBase = kOffStage + kStageBytes;            // BASE: the tile's rows of the base frame, staged alongside
    static constexpr int kOffWork = kOffBase + (BASE ? kStageBytes : 0);
    static constexpr int kBytes = kOffWork + BT * (N + 1) * 8;
};

// PAIR: a thread runs butterflies n2 and n2+1 together (one 8-byte load yields both samples of an IIQQ group).
// PAD : n_samples < N (zero padding needs a bound check per load); CT: compile-time n_chirps, 0 = run time.
// One staging buffer, refilled behind pass 2 (a double buffer refilled a whole tile ahead measured slower:
// profiles/experiments/r1_k1_variants_sweep.log).
// BASE: static-clutter removal — p.base_adc (one frame in capture format) is subtracted sample by sample, in integers,
// before the window (the reference's base-frame subtraction, acceleration.cu:152-166, for every antenna).  The tile's
// rows of the base frame are staged by the same TMA copies as the capture rows (they come from L2: the base frame is a
// few MB read by every CTA); reading them with per-lane global loads instead costs 4x sector over-fetch and +70 % time.
template <int N, int R1, int R2, int BT, int NW, bool PAIR, bool PAD, int CT, bool BASE>
__global__ void __launch_bounds__(NW * 32, (2 * RangeSmem<N, BT, BASE>::kBytes <= 226 * 1024 && NW <= 8) ? 2 : 1) range_fft_kernel(PlanDev p, const int16_t *__restrict__ adc, float2 *__restrict__ rs,
                                                            int n_tiles)
{
    static_assert(R1 * R2 == N, "plan");
    using L = RangeSmem<N, BT, BASE>;
    constexpr int NT = NW * 32;
    constexpr int SUBS = 32 / BT;
    constexpr int NSLOT = NW * SUBS;
    constexpr int LR1 = ilog2(R1), LR2 = ilog2(R2);

    extern __shared__ __align__(16) unsigned char smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem);
    float2 *tw = reinterpret_cast<float2 *>(smem + L::kOffTw);
    float *win = reinterpret_cast<float *>(smem + L::kOffWin);
    unsigned char *stage = smem + L::kOffStage;
    unsigned char *bstage = smem + L::kOffBase;                      // BASE only
    float2 *work = reinterpret_cast<float2 *>(smem + L::kOffWork);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = lane % BT, sub = lane / BT, slot = warp * SUBS + sub;
    const int S = PAD ? p.S : N, A = p.A;
    const int C = CT ? CT : p.C;
    const int nct = (C + BT - 1) / BT;

    auto issue = [&](int tile) {            // one warp: stage the BT int16 rows of `tile`
        const int ct = tile % nct, fa = tile / nct;
        const int a = fa % A, f = fa / A;
        const int c0 = ct * BT;
        const int nrows = min(BT, C - c0);
        uint64_t *b = &bar[0];
        if (lane == 0) {
            fence_proxy_async();
            mbar_arrive_expect_tx(b, (uint32_t)(nrows * S * 4) * (BASE ? 2u : 1u));
        }
        __syncwarp();
        if (lane < nrows) {
            const int16_t *src = adc + (((size_t)f * C + c0 + lane) * A + a) * (size_t)(2 * S);
            bulk_g2s(stage + lane * L::kStageStride, src, (uint32_t)(S * 4), b);
            if constexpr (BASE) {
                const int16_t *bsrc = p.base_adc + ((size_t)(c0 + lane) * A + a) * (size_t)(2 * S);
                bulk_g2s(bstage + lane * L::kStageStride, bsrc, (uint32_t)(S * 4), b);
            }
        }
    };

    // Tiles are handed out by a counter (PlanDev.sched), not by a fixed stride: a CTA that starts late — its SM was still held by
    // a kernel of another stream (another batch in flight, the exchange's merge kernel) — simply takes fewer tiles instead of
    // finishing its fixed share late.  The first tile of a CTA is blockIdx.x; the next one is fetched while pass 1 runs.
    __shared__ int s_next[2];
    unsigned int *ctr = p.sched;                                      // [0] next tile - gridDim.x, [1] CTAs done
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        fence_mbar_init();
    }
    __syncthreads();
    int tile = blockIdx.x;
    if (warp == 0 && tile < n_tiles) issue(tile);
    for (int i = tid; i < N; i += NT) tw[i] = p.tw1_r[i];
    for (int i = tid; i < N; i += NT) win[i] = i < S ? p.win_r[i] : 0.f;
    __syncthreads();

    float2 *wrow = work + row * (N + 1);
    int it = 0;                                                       // tiles done by this CTA

#pragma unroll 1
    for (; tile < n_tiles; ++it) {
        const int ct = tile % nct, fa = tile / nct;
        const int c0 = ct * BT;
        const bool row_ok = c0 + row < C;
        const float wdop = row_ok ? p.win_d[c0 + row] : 0.f;
        unsigned int fetched = 0u;
        if (tid == 0) fetched = atomicAdd(&ctr[0], 1u);               // answer needed after pass 1 only
        mbar_wait(&bar[0], (uint32_t)(it & 1));
        const unsigned char *srow = stage + row * L::kStageStride;
        const unsigned char *brow = BASE ? bstage + row * L::kStageStride : nullptr;

        // ---- pass 1: R2 butterflies of radix R1 over stride R2, reading the staged int16 rows ----
        if constexpr (PAIR) {
#pragma unroll 1
            for (int u = slot; u < R2 / 2; u += NSLOT) {
                const int n2 = 2 * u;
                float2 xa[R1], xb[R1];
#pragma unroll
                for (int m = 0; m < R1; ++m) {
                    const int n = n2 + m * R2;
                    if (!PAD || n < S) {
                        const uint2 raw = *reinterpret_cast<const uint2 *>(srow + 4 * n);   // [I(n) I(n+1)] [Q(n) Q(n+1)]
                        const float2 w = *reinterpret_cast<const float2 *>(win + n);
                        int i0 = (short)(raw.x & 0xffffu), q0 = (short)(raw.y & 0xffffu), i1 = (int)raw.x >> 16, q1 = (int)raw.y >> 16;
                        if constexpr (BASE) {
                            const uint2 rb = *reinterpret_cast<const uint2 *>(brow + 4 * n);
                            i0 -= (short)(rb.x & 0xffffu); q0 -= (short)(rb.y & 0xffffu);
                            i1 -= (int)rb.x >> 16;         q1 -= (int)rb.y >> 16;
                        }
                        xa[m] = make_float2((float)i0 * w.x, (float)q0 * w.x);
                        xb[m] = make_float2((float)i1 * w.y, (float)q1 * w.y);
                    } else {
                        xa[m] = xb[m] = make_float2(0.f, 0.f);
                    }
                }
                dft_regs<R1>(xa);
                dft_regs<R1>(xb);
                const float4 *twu = reinterpret_cast<const float4 *>(tw) + u * R1;   // {W^(n2 k1), W^((n2+1) k1)}
                float2 *wo = wrow + n2;
#pragma unroll
                for (int k1 = 0; k1 < R1; ++k1) {
                    float2 va = xa[bitrev(k1, LR1)], vb = xb[bitrev(k1, LR1)];
                    if (k1 > 0) {
                        const float4 t = twu[k1];
                        va = cmul(va, make_float2(t.x, t.y));
                        vb = cmul(vb, make_float2(t.z, t.w));
                    }
                    wo[k1 * R2] = va;
                    wo[k1 * R2 + 1] = vb;
                }
            }
        } else {
#pragma unroll 1
            for (int u = slot; u < R2; u += NSLOT) {
                const int n2 = u;
                const int odd = n2 & 1;
                float2 x[R1];
#pragma unroll
                for (int m = 0; m < R1; ++m) {
                    const int n = n2 + m * R2;
                    if (!PAD || n < S) {
                        const uint2 raw = *reinterpret_cast<const uint2 *>(srow + 4 * (n - odd));
                        const float w = win[n];
                        int iv = odd ? ((int)raw.x >> 16) : (int)(short)(raw.x & 0xffffu);
                        int qv = odd ? ((int)raw.y >> 16) : (int)(short)(raw.y & 0xffffu);
                        if constexpr (BASE) {
                            const uint2 rb = *reinterpret_cast<const uint2 *>(brow + 4 * (n - odd));
                            iv -= odd ? ((int)rb.x >> 16) : (int)(short)(rb.x & 0xffffu);
                            qv -= odd ? ((int)rb.y >> 16) : (int)(short)(rb.y & 0xffffu);
                        }
                        x[m] = make_float2((float)iv * w, (float)qv * w);
                    } else {
                        x[m] = make_float2(0.f, 0.f);
                    }
                }
                dft_regs<R1>(x);
                const float2 *twu = tw + tw1_index(n2, 0, R1);
                float2 *wo = wrow + n2;
#pragma unroll
                for (int k1 = 0; k1 < R1; ++k1) {
                    float2 v = x[bitrev(k1, LR1)];
                    if (k1 > 0) v = cmul(v, twu[2 * k1]);
                    wo[k1 * R2] = v;
                }
            }
        }
        if (tid == 0) s_next[(it + 1) & 1] = (int)min(fetched + gridDim.x, (unsigned int)n_tiles);
        __syncthreads();
        const int next_tile = s_next[(it + 1) & 1];
        // the staging buffer is consumed now: prefetch the next tile behind pass 2.  (Refilling it earlier — as
        // soon as the last warp has pulled its pass-1 inputs into registers — removes the wait on the copy but not a
        // microsecond of run time: the stall moves to the barrier, profiles/experiments/r1_k1_early_release.md.  L2 prefetch
        // hints for the tiles after that made it slower, r1_k1_l2_prefetch.log.)
        if (warp == 0 && next_tile < n_tiles) issue(next_tile);

        // ---- pass 2: R1 butterflies of radix R2 on contiguous runs; outputs go straight to HBM ----
        float2 *out = rs + (size_t)fa * (size_t)N * C + c0 + row;
#pragma unroll 1
        for (int u = slot; u < R1; u += NSLOT) {
            const int k1 = u;
            float2 y[R2];
            const float2 *wi = wrow + k1 * R2;
#pragma unroll
            for (int n2 = 0; n2 < R2; ++n2) y[n2] = wi[n2];
            dft_regs<R2>(y);
            if (row_ok) {
                float2 *o = out + (size_t)k1 * C;
#pragma unroll
                for (int k2 = 0; k2 < R2; ++k2) {
                    const float2 v = y[bitrev(k2, LR2)];
                    st_global_f2(o + (size_t)(R1 * k2) * C, cscale(v, wdop));
                }
            }
        }
        __syncthreads();
        tile = next_tile;
    }
    if (tid == 0) sched_retire(ctr);
}

// ---------------------------------------------------------------------------
// K2: Doppler FFT + non-coherent integration
// ---------------------------------------------------------------------------
// |X|^2 and the running sum over antennas with the roundings pinned (no FMA contraction across the two), so that the
// one-pass kernels and the antenna-split path for small batches (per-antenna maps + power_sum_kernel) give the same bits.
__device__ __forceinline__ float accumulate_power(float acc, float2 v)
{
    return __fadd_rn(acc, __fmaf_rn(v.x, v.x, __fmul_rn(v.y, v.y)));
}
// two bins at once: each |X|^2 with the roundings above, the two running sums as one packed add (same bits, one issue slot less)
__device__ __forceinline__ float2 accumulate_power2(float2 acc, float2 v0, float2 v1)
{
    const float2 pw = make_float2(__fmaf_rn(v0.x, v0.x, __fmul_rn(v0.y, v0.y)), __fmaf_rn(v1.x, v1.x, __fmul_rn(v1.y, v1.y)));
    return __fadd2_rn(acc, pw);
}

// INPLACE: pass 1 writes its outputs back into the staging row it read (a thread reads and writes the same R1
// addresses, so there is no hazard), which frees the separate work buffer: the same footprint then holds three
// staging buffers instead of two, i.e. two loads in flight per CTA while a third is being transformed.
template <int N, int BT, int NSTAGE, bool INPLACE = false>
struct DopplerSmem {
    static constexpr int kStageRow = N + 2;                          // float2 per staged row (16-byte multiple; conflict-free
                                                                     // for 16 rows x 2 sub-slots of 8-byte accesses)
    static constexpr int kOffTw = 32;                                // up to four mbarriers in front
    static constexpr int kOffStage = kOffTw + 8 * N;
    static constexpr int kStageBytes = BT * kStageRow * 8;
    static constexpr int kOffWork = kOffStage + NSTAGE * kStageBytes;
    static constexpr int kBytes = kOffWork + (INPLACE ? 0 : BT * (N + 1) * 8);
    static constexpr int kWorkRow = INPLACE ? kStageRow : N + 1;
};

// PAD: n_chirps < N.  SPT: compile-time Sp (range FFT length = stride of the power map / cube), 0 = run time.
// NSTAGE = 2: the next step is prefetched while the current one is transformed (double buffer);
// NSTAGE = 1: one staging buffer, refilled behind pass 2 (smaller footprint -> more CTAs per SM).
template <int N, int BT, int NW, int NSTAGE, bool INPLACE>
constexpr int doppler_min_ctas()
{
    constexpr int by_smem = (226 * 1024) / DopplerSmem<N, BT, NSTAGE, INPLACE>::kBytes;
    constexpr int by_threads = 768 / (NW * 32);                      // keeps >= 85 registers per thread
    constexpr int m = by_smem < by_threads ? by_smem : by_threads;
    return m < 1 ? 1 : (m > 3 ? 3 : m);
}

// The two passes of a CTA-shared Doppler tile, shared by doppler_fft_kernel and doppler_extract_kernel so that K2x's
// snapshots are the very values K2 computes.  A slot (the lanes of a warp that work on one row) owns the butterflies
// slot, slot + NSLOT, ... of each pass.
// Pass 1: R2 butterflies of radix R1 over stride R2 (Doppler window already applied by K1), read from srow and written to
// wrow, which may be srow (a thread reads and writes the same R1 addresses).  TWREG: the slot's twiddles are held in twr;
// otherwise they are read from tw.  The butterfly's registers x are the caller's, and the zero-fill of padded chirps is
// written per component: with an array of the helper's own or one float2 select, ptxas allocates doppler_fft_kernel's
// registers differently from the form the sweeps under profiles/ measured.
template <int R1, int R2, int NSLOT, bool PAD, bool TWREG>
__device__ __forceinline__ void doppler_pass1(const float2 *srow, float2 *wrow, const float2 *tw, const float2 (*twr)[TWREG ? R1 - 1 : 1],
                                              int slot, int C, float2 (&x)[R1])
{
    constexpr int LR1 = ilog2(R1);
    constexpr int UPS1 = (R2 + NSLOT - 1) / NSLOT;
#pragma unroll
    for (int ui = 0; ui < UPS1; ++ui) {
        const int n2 = slot + ui * NSLOT;
        if (UPS1 * NSLOT == R2 || n2 < R2) {
#pragma unroll
            for (int m = 0; m < R1; ++m) {
                const int n = n2 + m * R2;
                float vy = 0.f, vx = 0.f;
                if (!PAD || n < C) { const float2 t = srow[n]; vy = t.y; vx = t.x; }
                x[m] = make_float2(vx, vy);
            }
            dft_regs<R1>(x);
            float2 *wo = wrow + n2;
            wo[0] = x[0];
#pragma unroll
            for (int k1 = 1; k1 < R1; ++k1) {
                const float2 w = TWREG ? twr[ui][k1 - 1] : tw[tw1_index(n2, k1, R1)];
                wo[k1 * R2] = cmul(x[bitrev(k1, LR1)], w);
            }
        }
    }
}

// Pass 2 of one run: radix R2 on the R2 contiguous pass-1 outputs at wi; bin k1 + R1 * k2 lands in y[bitrev(k2)].
template <int R2>
__device__ __forceinline__ void doppler_pass2(const float2 *wi, float2 (&y)[R2])
{
#pragma unroll
    for (int n2 = 0; n2 < R2; ++n2) y[n2] = wi[n2];
    dft_regs<R2>(y);
}

template <int N, int R1, int R2, int BT, int NW, bool PAD, int SPT, int NSTAGE, bool INPLACE>
__global__ void __launch_bounds__(NW * 32, doppler_min_ctas<N, BT, NW, NSTAGE, INPLACE>()) doppler_fft_kernel(PlanDev p, const float2 *__restrict__ rs, float2 *__restrict__ cube,
                                                               float *__restrict__ pmap, int n_tiles)
{
    static_assert(R1 * R2 == N, "plan");
    static_assert(NSTAGE >= 1 && NSTAGE <= 4, "stages");
    static_assert(!INPLACE || NSTAGE >= 2, "in-place needs a second buffer to prefetch into");
    using L = DopplerSmem<N, BT, NSTAGE, INPLACE>;
    constexpr int NT = NW * 32;
    constexpr int SUBS = 32 / BT;
    constexpr int NSLOT = NW * SUBS;
    constexpr int LR2 = ilog2(R2);
    constexpr int UPS2 = (R1 + NSLOT - 1) / NSLOT;                   // pass-2 butterflies per slot
    constexpr int UPS1 = (R2 + NSLOT - 1) / NSLOT;                   // pass-1 butterflies per slot
    // a slot's pass-1 butterflies are the same for every step, so their twiddles can live in registers
    constexpr bool TWREG = UPS1 * (R1 - 1) <= 16;

    extern __shared__ __align__(16) unsigned char smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem);              // NSTAGE barriers
    float2 *tw = reinterpret_cast<float2 *>(smem + L::kOffTw);
    float2 *stage = reinterpret_cast<float2 *>(smem + L::kOffStage);
    float2 *work = reinterpret_cast<float2 *>(smem + L::kOffWork);      // unused when INPLACE

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = lane % BT, sub = lane / BT, slot = warp * SUBS + sub;
    const int C = PAD ? p.C : N, A = p.A;
    const int Sp = SPT ? SPT : p.Sp;
    const int nrt = Sp / BT;

    // a "step" is one antenna of one tile; the q-th step of this CTA is antenna q % A of its (q / A)-th tile, and
    // steps of consecutive tiles are pipelined back to back.  The tile of ordinal o is blockIdx.x + o * gridDim.x: K2 keeps
    // the fixed stride (K1's counter was slower on cfg3 and cfg5, faster on cfg2: profiles/r2/sweep_tile_scheduling.log).
    auto issue_step = [&](int q) {                                    // warp 0
        const int itq = q / A, a = q - itq * A;
        const unsigned int t = blockIdx.x + (unsigned int)itq * gridDim.x;
        if (t >= (unsigned int)n_tiles) return;
        const int tile = (int)t;
        const int rt = tile % nrt, f = tile / nrt;
        const int buf = q % NSTAGE;
        uint64_t *b = &bar[buf];
        if (lane == 0) {
            fence_proxy_async();
            mbar_arrive_expect_tx(b, (uint32_t)(BT * C * 8));
        }
        __syncwarp();
        if (lane < BT) {
            const float2 *src = rs + (((size_t)f * A + a) * Sp + rt * BT + lane) * (size_t)C;
            bulk_g2s(stage + (size_t)buf * (BT * L::kStageRow) + lane * L::kStageRow, src, (uint32_t)(C * 8), b);
        }
    };
    // how far ahead of the step being transformed the loads run
    constexpr int AHEAD = INPLACE ? NSTAGE - 1 : 1;

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < NSTAGE; ++i) mbar_init(&bar[i], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < AHEAD; ++i) issue_step(i);
    }
    for (int i = tid; i < N; i += NT) tw[i] = p.tw1_d[i];
    __syncthreads();

    int s = 0;                                                        // running step counter of this CTA
    float2 twr[TWREG ? UPS1 : 1][TWREG ? R1 - 1 : 1];
    if constexpr (TWREG) {
#pragma unroll
        for (int ui = 0; ui < UPS1; ++ui)
#pragma unroll
            for (int k1 = 1; k1 < R1; ++k1) twr[ui][k1 - 1] = tw[tw1_index(min(slot + ui * NSLOT, R2 - 1), k1, R1)];
    }

#pragma unroll 1
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int rt = tile % nrt, f = tile / nrt;
        const int r0 = rt * BT;
        float acc[UPS2][R2];
#pragma unroll
        for (int i = 0; i < UPS2; ++i)
#pragma unroll
            for (int j = 0; j < R2; ++j) acc[i][j] = 0.f;

#pragma unroll 1
        for (int a = 0; a < A; ++a, ++s) {
            // the buffer step s + AHEAD lands in was released by the barrier that ended step s - 1 (in-place) /
            // is the other half of the double buffer
            if ((INPLACE || NSTAGE == 2) && warp == 0) issue_step(s + AHEAD);
            mbar_wait(&bar[s % NSTAGE], (uint32_t)((s / NSTAGE) & 1));
            float2 *srow = stage + (size_t)(s % NSTAGE) * (BT * L::kStageRow) + row * L::kStageRow;
            float2 *wrow = INPLACE ? srow : work + row * (N + 1);

            float2 x[R1];
            doppler_pass1<R1, R2, NSLOT, PAD, TWREG>(srow, wrow, tw, twr, slot, C, x);
            __syncthreads();
            if (!INPLACE && NSTAGE == 1 && warp == 0) issue_step(s + 1);   // staging buffer consumed: refill behind pass 2

            // pass 2: radix R2 on contiguous runs; accumulate |X|^2 (ascending antenna order)
#pragma unroll
            for (int ui = 0; ui < UPS2; ++ui) {
                const int k1 = slot + ui * NSLOT;
                if (k1 < R1) {
                    float2 y[R2];
                    doppler_pass2<R2>(wrow + k1 * R2, y);
#pragma unroll
                    for (int k2 = 0; k2 < R2; ++k2) {
                        const float2 v = y[bitrev(k2, LR2)];
                        acc[ui][k2] = accumulate_power(acc[ui][k2], v);
                    }
                    if (cube != nullptr) {
                        float2 *o = cube + (((size_t)f * A + a) * (size_t)N + k1) * Sp + r0 + row;
#pragma unroll
                        for (int k2 = 0; k2 < R2; ++k2) st_global_f2(o + (size_t)(R1 * k2) * Sp, y[bitrev(k2, LR2)]);
                    }
                }
            }
            __syncthreads();
        }

        float *po = pmap + (size_t)f * N * Sp + r0 + row;
#pragma unroll
        for (int ui = 0; ui < UPS2; ++ui) {
            const int k1 = slot + ui * NSLOT;
            if (k1 < R1) {
                float *o = po + (size_t)k1 * Sp;
#pragma unroll
                for (int k2 = 0; k2 < R2; ++k2) o[(size_t)(R1 * k2) * Sp] = acc[ui][k2];
            }
        }
    }
}

// ---------------------------------------------------------------------------
// K2x: selective Doppler re-FFT (fused mode, wide arrays): antenna snapshots of the detected cells
// ---------------------------------------------------------------------------
// In fused mode the Doppler cube is never written, so the angle stage has to re-derive, for every detection (f, r, d), the
// Doppler bin d of all A antennas at range bin r.  A direct DFT per detection costs A * C complex MACs and a pass over the
// A x C block of the range spectrum; on the imaging cube (A = 192, C = 512: 786 KB per range bin) with thousands of hits
// that was the longest stage of the chain.  Here every (frame, range bin) that has at least one hit — `rows`, made by
// rows_kernel from the ordered key list — is transformed ONCE more with the very FFT K2 runs (doppler_pass1 and
// doppler_pass2: the snapshot is bit-identical to what the Doppler cube would hold), and only the detected bins are written
// out, to snap[dense index][antenna].  Cost: one K2 step per hit row, whatever the number of hits in it — bounded by one K2
// pass.  A tile is BT arbitrary hit rows (each row is its own bulk copy, so they need not be neighbours); staging, the
// in-place pass 1 and the three-stage ring are those of doppler_fft_kernel<.., INPLACE>.
template <int N, int BT>
struct ExtractSmem {
    static constexpr int kStageRow = N + 2;
    static constexpr int kNStage = 3;
    static constexpr int kOffRows = 32;                              // three mbarriers in front
    static constexpr int kOffTw = kOffRows + BT * 16 + (BT + 1) * 4 + 12;   // uint4 row refs + prefix counts (padded to 16)
    static constexpr int kOffStage = ((kOffTw + 8 * N) + 15) / 16 * 16;
    static constexpr int kBytes = kOffStage + kNStage * BT * kStageRow * 8;
};

template <int N, int R1, int R2, int BT, int NW, bool PAD>
__global__ void __launch_bounds__(NW * 32, (2 * ExtractSmem<N, BT>::kBytes <= 226 * 1024 && NW <= 8) ? 2 : 1)
    doppler_extract_kernel(PlanDev p, const float2 *__restrict__ rs, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ offsets,
                           const uint4 *__restrict__ rows, const unsigned int *__restrict__ n_rows_ptr, float2 *__restrict__ snap, int dense_cap)
{
    static_assert(R1 * R2 == N, "plan");
    using L = ExtractSmem<N, BT>;
    constexpr int NT = NW * 32;
    constexpr int NSTAGE = L::kNStage, AHEAD = NSTAGE - 1;
    constexpr int SUBS = 32 / BT;
    constexpr int NSLOT = NW * SUBS;
    constexpr int LR2 = ilog2(R2);
    constexpr int UPS2 = (R1 + NSLOT - 1) / NSLOT;

    extern __shared__ __align__(16) unsigned char smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem);
    uint4 *s_row = reinterpret_cast<uint4 *>(smem + L::kOffRows);     // {frame, range bin, dense index of the first hit, hits} per tile row
    uint32_t *s_pref = reinterpret_cast<uint32_t *>(smem + L::kOffRows + BT * 16);   // [BT + 1] exclusive prefix of the hit counts
    float2 *tw = reinterpret_cast<float2 *>(smem + L::kOffTw);
    float2 *stage = reinterpret_cast<float2 *>(smem + L::kOffStage);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = lane % BT, sub = lane / BT, slot = warp * SUBS + sub;
    const int C = PAD ? p.C : N, A = p.A;
    const int Sp = p.Sp;
    const uint32_t n_rows = *n_rows_ptr;
    const int n_tiles = (int)((n_rows + BT - 1) / BT);
    if (n_tiles == 0) return;
    // Antennas are independent here (nothing is accumulated across them), so a tile's antennas are cut into chunks and a
    // work item is (tile, chunk): a handful of hit rows — a sparse scene — still spreads over every CTA instead of walking
    // A antennas one after the other inside a few.  Aim: ~8 items per CTA, chunks of at least 4 antennas.
    int n_chunks = (int)((8LL * gridDim.x + n_tiles - 1) / n_tiles);
    n_chunks = max(1, min(n_chunks, (A + 3) / 4));
    const int AC = (A + n_chunks - 1) / n_chunks;                     // antennas per chunk (the last one may be shorter)
    n_chunks = (A + AC - 1) / AC;
    const long long n_items = (long long)n_tiles * n_chunks;
    if ((long long)blockIdx.x >= n_items) return;
    auto item_antennas = [&](long long item) { const int ch = (int)(item % n_chunks); return min(AC, A - ch * AC); };

    // issue side (warp 0): the staging copies run AHEAD steps in front of the transform, across item boundaries
    long long is_item = blockIdx.x;
    int is_a = 0;
    auto issue_next = [&](int q) {                                    // warp 0: stage the next step in line into buffer q % NSTAGE
        if (is_item >= n_items) return;
        const int tile = (int)(is_item / n_chunks), a = (int)(is_item % n_chunks) * AC + is_a;
        const uint32_t ri = (uint32_t)tile * BT + lane;
        const bool live = lane < BT && ri < n_rows;
        const uint32_t nlive = min((uint32_t)BT, n_rows - (uint32_t)tile * BT);
        const int buf = q % NSTAGE;
        uint64_t *b = &bar[buf];
        if (lane == 0) {
            fence_proxy_async();
            mbar_arrive_expect_tx(b, nlive * (uint32_t)(C * 8));
        }
        __syncwarp();
        if (live) {
            const uint4 rr = rows[ri];
            const float2 *src = rs + (((size_t)rr.x * A + a) * Sp + rr.y) * (size_t)C;
            bulk_g2s(stage + (size_t)buf * (BT * L::kStageRow) + lane * L::kStageRow, src, (uint32_t)(C * 8), b);
        }
        if (++is_a >= item_antennas(is_item)) { is_a = 0; is_item += gridDim.x; }
    };

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < NSTAGE; ++i) mbar_init(&bar[i], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < AHEAD; ++i) issue_next(i);
    }
    for (int i = tid; i < N; i += NT) tw[i] = p.tw1_d[i];

    int s = 0;
    int cur_tile = -1;
    uint32_t H = 0;
#pragma unroll 1
    for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int tile = (int)(item / n_chunks), a0 = (int)(item % n_chunks) * AC, na = item_antennas(item);
        if (tile != cur_tile) {
            // ---- the tile's rows: where their hits sit in the dense list and how many there are ----
            __syncthreads();                                          // s_row / s_pref of the previous tile are no longer read
            for (int i = warp; i < BT; i += NW) {
                const uint32_t ri = (uint32_t)tile * BT + i;
                uint4 rr = make_uint4(0u, 0u, 0u, 0u);
                if (ri < n_rows) {
                    rr = rows[ri];
                    const uint32_t fbeg = offsets[rr.x], fend = min(offsets[rr.x + 1], (uint32_t)dense_cap);
                    const uint32_t *kf = keys + (size_t)rr.x * p.max_det - fbeg;     // kf[g] = key of dense position g
                    uint32_t n = 0;
                    for (uint32_t g = rr.z;; g += 32) {               // the run of equal range bin that starts at rr.z
                        const bool same = g + lane < fend && (kf[g + lane] >> 16) == rr.y;
                        const uint32_t m = __ballot_sync(0xffffffffu, same);
                        const uint32_t k = m == 0xffffffffu ? 32u : (uint32_t)(__ffs(~m) - 1);
                        n += k;
                        if (k < 32u) break;
                    }
                    rr.w = n;
                }
                if (lane == 0) s_row[i] = rr;
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t acc = 0;
                for (int i = 0; i < BT; ++i) { s_pref[i] = acc; acc += s_row[i].w; }
                s_pref[BT] = acc;
            }
            __syncthreads();
            H = s_pref[BT];
            cur_tile = tile;
        }

#pragma unroll 1
        for (int a = a0; a < a0 + na; ++a, ++s) {
            if (warp == 0) issue_next(s + AHEAD);
            mbar_wait(&bar[s % NSTAGE], (uint32_t)((s / NSTAGE) & 1));
            float2 *sbuf = stage + (size_t)(s % NSTAGE) * (BT * L::kStageRow);
            float2 *srow = sbuf + row * L::kStageRow;

            float2 x[R1];
            doppler_pass1<R1, R2, NSLOT, PAD, false>(srow, srow, tw, nullptr, slot, C, x);      // in place
            __syncthreads();
            // pass 2; bin k1 + R1 * k2 goes back to srow[k1 * R2 + k2] (the run this thread has just read)
#pragma unroll
            for (int ui = 0; ui < UPS2; ++ui) {
                const int k1 = slot + ui * NSLOT;
                if (k1 < R1) {
                    float2 y[R2];
                    float2 *wi = srow + k1 * R2;
                    doppler_pass2<R2>(wi, y);
#pragma unroll
                    for (int k2 = 0; k2 < R2; ++k2) wi[k2] = y[bitrev(k2, LR2)];
                }
            }
            __syncthreads();
            // the detected bins of this antenna -> snap[dense index][a]
            for (uint32_t h = tid; h < H; h += NT) {
                int i = 0;
#pragma unroll
                for (int j = 1; j < BT; ++j) i += (h >= s_pref[j]) ? 1 : 0;
                const uint4 rr = s_row[i];
                const uint32_t g = rr.z + (h - s_pref[i]);
                const uint32_t d = keys[(size_t)rr.x * p.max_det + (g - offsets[rr.x])] & 0xffffu;
                const float2 v = sbuf[i * L::kStageRow + (d % R1) * R2 + d / R1];
                st_global_f2(snap + (size_t)g * A + a, v);
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// K2w: Doppler FFT with warp-private tiles (fused mode: power map only)
// ---------------------------------------------------------------------------
// doppler_fft_kernel above shares a 16-row tile between the warps of a CTA, so the two passes are separated by CTA-wide
// barriers and all warps of the CTA sit in the same phase (ncu: barrier is the top stall, issue slots < 50 % busy).
// Here a warp owns its rows outright: lanes = ROWS rows x SUBS butterflies of one row, the hand-over between the passes
// is a __syncwarp, every warp has its own mbarrier-tracked staging ring, and the 16 warps of an SM drift apart so that one
// warp's shared-memory latency hides behind another's arithmetic.  Pass 1 runs in place: a thread first pulls all its
// inputs into registers, and the outputs go back into the same row in a layout padded by one element per R2 so that
// pass 2 (lanes = different k1 of one row, stride R2) is bank-conflict free.
template <int N, int R1, int R2>
struct DopplerWarp {
    static constexpr int kSubs = (R1 < R2 ? R1 : R2) > 16 ? 16 : (R1 < R2 ? R1 : R2);
    static constexpr int kRows = 32 / kSubs;
    static constexpr int kU1 = R2 / kSubs;                           // pass-1 butterflies per thread
    static constexpr int kU2 = R1 / kSubs;                           // pass-2 butterflies per thread
    static constexpr int kRowStride = N + R1;                        // float2: N points + one pad per R2
    static constexpr int kStage = kRows * kRowStride;                // float2 per staging buffer of one warp
    static constexpr int kOffTw = 512;                               // room for NW * NSTAGE mbarriers
    static constexpr int bytes(int nw, int nstage) { return kOffTw + 8 * N + nw * nstage * kStage * 8; }
};

template <int N, int R1, int R2, int NW, bool PAD, int SPT, int NSTAGE, int MINB = 2>
__global__ void __launch_bounds__(NW * 32, MINB) doppler_fft_warp_kernel(PlanDev p, const float2 *__restrict__ rs, float *__restrict__ pmap,
                                                                      int n_tiles)
{
    static_assert(R1 * R2 == N, "plan");
    using L = DopplerWarp<N, R1, R2>;
    constexpr int SUBS = L::kSubs, ROWS = L::kRows, U1 = L::kU1, U2 = L::kU2;
    constexpr int LR1 = ilog2(R1), LR2 = ilog2(R2);
    constexpr bool TWREG = U1 * (R1 - 1) <= 16;
    static_assert(NW * NSTAGE * 8 <= L::kOffTw, "barriers");

    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem) + warp * NSTAGE;
    float2 *tw = reinterpret_cast<float2 *>(smem + L::kOffTw);
    float2 *ring = reinterpret_cast<float2 *>(smem + L::kOffTw + 8 * N) + (size_t)warp * NSTAGE * L::kStage;

    const int row = lane / SUBS, sub = lane % SUBS;
    const int C = PAD ? p.C : N, A = p.A;
    const int Sp = SPT ? SPT : p.Sp;
    const int nrt = Sp / ROWS;
    const long long gw = (long long)blockIdx.x * NW + warp, nwarp = (long long)gridDim.x * NW;

    // A warp walks the tiles gw, gw + nwarp, gw + 2 nwarp, ...: the fixed stride of doppler_fft_kernel.
    // Staging side.  The ROWS rows of a tile are neighbours in rs ([f][a][Sp][C]), so one step is ONE bulk copy of ROWS * C
    // elements, issued by lane 0: the rows land back to back at the head of the ring slot (row i at i * C), pass 1 pulls them
    // into registers and writes its outputs over them in the padded layout (row i at i * kRowStride).  The step to stage next
    // runs NSTAGE - 1 steps ahead of the transform and is running state — its antenna, its tile, its ring slot, its source
    // address — advanced by additions; the only division left is one per tile.
    const uint32_t step_bytes = (uint32_t)(ROWS * C * 8);
    const size_t ant_stride = (size_t)Sp * C;                       // float2 between the antennas of one (frame, range bin)
    auto tile_src = [&](long long tl) -> const float2 * {
        const int tile = (int)tl;
        const int rt = tile % nrt, f = tile / nrt;
        return rs + ((size_t)f * A * Sp + (size_t)rt * ROWS) * (size_t)C;
    };
    long long is_tile = gw;
    int is_a = 0, is_slot = 0;
    const float2 *is_src = rs;
    auto issue_next = [&]() {
        if (is_tile < n_tiles) {
            if (is_a == 0) is_src = tile_src(is_tile);
            if (lane == 0) {
                uint64_t *b = &bar[is_slot];
                fence_proxy_async();
                mbar_arrive_expect_tx(b, step_bytes);
                bulk_g2s(ring + (size_t)is_slot * L::kStage, is_src, step_bytes, b);
            }
            is_src += ant_stride;
        }
        is_slot = is_slot + 1 == NSTAGE ? 0 : is_slot + 1;
        if (++is_a == A) {
            is_a = 0;
            is_tile += nwarp;
        }
    };

    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NSTAGE; ++i) mbar_init(&bar[i], 1);
        fence_mbar_init();
    }
    for (int i = tid; i < N; i += NW * 32) tw[i] = p.tw1_d[i];
    __syncthreads();                                                 // the only CTA-wide barrier
#pragma unroll
    for (int i = 0; i < NSTAGE - 1; ++i) issue_next();

    float2 twr[TWREG ? U1 : 1][TWREG ? R1 - 1 : 1];
    if constexpr (TWREG) {
#pragma unroll
        for (int u = 0; u < U1; ++u)
#pragma unroll
            for (int k1 = 1; k1 < R1; ++k1) twr[u][k1 - 1] = tw[tw1_index(sub + u * SUBS, k1, R1)];
    }

    int q = 0;
#pragma unroll 1
    for (long long t = gw; t < n_tiles; t += nwarp) {
        const int tile = (int)t;
        const int rt = tile % nrt, f = tile / nrt;
        float2 acc[U2][R2 / 2];                                     // bins k2 = 2 j, 2 j + 1
#pragma unroll
        for (int u = 0; u < U2; ++u)
#pragma unroll
            for (int j = 0; j < R2 / 2; ++j) acc[u][j] = make_float2(0.f, 0.f);

#pragma unroll 1
        for (int a = 0; a < A; ++a, ++q) {
            issue_next();                                            // step q + NSTAGE - 1, into the slot step q - 1 has just left
            mbar_wait(&bar[q % NSTAGE], (uint32_t)((q / NSTAGE) & 1));
            float2 *slot = ring + (size_t)(q % NSTAGE) * L::kStage;
            const float2 *rin = slot + row * C;                      // as staged
            float2 *r = slot + row * L::kRowStride;                  // as transformed

            // pass 1: all inputs into registers first (the outputs overwrite other threads' inputs)
            float2 x[U1][R1];
#pragma unroll
            for (int u = 0; u < U1; ++u) {
                const int n2 = sub + u * SUBS;
#pragma unroll
                for (int m = 0; m < R1; ++m) {
                    const int n = n2 + m * R2;
                    x[u][m] = (!PAD || n < C) ? rin[n] : make_float2(0.f, 0.f);
                }
            }
            __syncwarp();
#pragma unroll
            for (int u = 0; u < U1; ++u) {
                const int n2 = sub + u * SUBS;
                dft_regs<R1>(x[u]);
                r[n2] = x[u][0];
#pragma unroll
                for (int k1 = 1; k1 < R1; ++k1) {
                    const float2 w = TWREG ? twr[u][k1 - 1] : tw[tw1_index(n2, k1, R1)];
                    r[k1 * (R2 + 1) + n2] = cmul(x[u][bitrev(k1, LR1)], w);
                }
            }
            __syncwarp();
            // pass 2: radix R2 on (padded) contiguous runs; accumulate |X|^2 (ascending antenna order)
#pragma unroll
            for (int u = 0; u < U2; ++u) {
                const int k1 = sub + u * SUBS;
                float2 y[R2];
                const float2 *wi = r + k1 * (R2 + 1);
#pragma unroll
                for (int n2 = 0; n2 < R2; ++n2) y[n2] = wi[n2];
                dft_regs<R2>(y);
#pragma unroll
                for (int j = 0; j < R2 / 2; ++j) acc[u][j] = accumulate_power2(acc[u][j], y[bitrev(2 * j, LR2)], y[bitrev(2 * j + 1, LR2)]);
            }
            __syncwarp();
        }

        float *po = pmap + (size_t)f * N * Sp + rt * ROWS + row;
#pragma unroll
        for (int u = 0; u < U2; ++u) {
            const int k1 = sub + u * SUBS;
#pragma unroll
            for (int j = 0; j < R2 / 2; ++j) {
                po[(size_t)(k1 + R1 * (2 * j)) * Sp] = acc[u][j].x;
                po[(size_t)(k1 + R1 * (2 * j + 1)) * Sp] = acc[u][j].y;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// antenna-split path for small batches (latency mode)
// ---------------------------------------------------------------------------
// A tile of K2 walks its antennas one after the other, so a batch of one or a few frames occupies a handful of CTAs for
// A steps each (one 256 x 128 x 12 frame: 16 CTAs x 12 steps).  For such batches the same kernels are launched over
// F*A single-antenna "frames" — [F][A][Sp][C] is [F*A][1][Sp][C] — which spreads the steps over F*A times as many CTAs,
// and the per-antenna power maps are then summed in ascending antenna order (the order and roundings of the one-pass
// accumulation, see accumulate_power).
__global__ void __launch_bounds__(256) power_sum_kernel(const float *__restrict__ per_antenna, float *__restrict__ pmap, int A, size_t M,
                                                        size_t total)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t f = i / M, m = i - f * M;
        const float *src = per_antenna + f * (size_t)A * M + m;
        float acc = 0.f;
        for (int a = 0; a < A; ++a) acc = __fadd_rn(acc, src[(size_t)a * M]);
        pmap[i] = acc;
    }
}

// ---------------------------------------------------------------------------
// export kernels (not on the hot path)
// ---------------------------------------------------------------------------
__global__ void export_cube_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, int A, int Sp, int Cp)
{   // in [A][Cp][Sp] -> out [A][Sp][Cp]
    const size_t n = (size_t)A * Sp * Cp;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int d = i % Cp;
        const int r = (i / Cp) % Sp;
        const int a = i / ((size_t)Cp * Sp);
        out[i] = in[((size_t)a * Cp + d) * Sp + r];
    }
}
__global__ void export_pmap_kernel(const float *__restrict__ in, float *__restrict__ out, int Sp, int Cp)
{
    const int n = Sp * Cp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int d = i % Cp, r = i / Cp;
        out[i] = in[(size_t)d * Sp + r];
    }
}
__global__ void export_mask_kernel(const uint32_t *__restrict__ in, uint8_t *__restrict__ out, int Sp, int Cp)
{
    const int n = Sp * Cp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int d = i % Cp, r = i / Cp;
        out[i] = (uint8_t)((in[(size_t)(d >> 5) * Sp + r] >> (d & 31)) & 1u);
    }
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
// Function attributes (opt-in shared memory) and occupancy are per device: a process may hold contexts on several GPUs
// (mmw_config.device), so everything cached about a kernel is cached per device ordinal.
int current_device()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return dev < 0 ? 0 : (dev >= kMaxDevices ? kMaxDevices - 1 : dev);
}

static int sm_count()
{
    static int count[kMaxDevices] = {0};
    const int dev = current_device();
    if (!count[dev]) {
        cudaDeviceGetAttribute(&count[dev], cudaDevAttrMultiProcessorCount, dev);
        if (count[dev] <= 0) count[dev] = 148;
    }
    return count[dev];
}

bool doppler_prefers_split(const PlanDev &p, int n_frames)
{
    // fewer tiles than half the SMs (tiles are 16 range bins or the equivalent number of warp-private tiles)
    return p.A > 1 && (long long)n_frames * (p.Sp / 16) * 2 <= sm_count();
}

cudaError_t launch_power_sum(const PlanDev &p, const float *per_antenna, float *pmap, int n_frames, cudaStream_t st)
{
    const size_t M = (size_t)p.Sp * p.Cp, total = M * n_frames;
    const int grid = (int)((total + 255) / 256 < (size_t)sm_count() * 8 ? (total + 255) / 256 : (size_t)sm_count() * 8);
    power_sum_kernel<<<grid, 256, 0, st>>>(per_antenna, pmap, p.A, M, total);
    return cudaGetLastError();
}

// Resident CTAs per SM of `Kernel` at `threads` threads and `smem_bytes` of dynamic shared memory, on the current device
// (which also opts the kernel in to that much shared memory); looked up once per device.  A kernel that cannot be resident
// at all is an error.
template <auto Kernel>
static cudaError_t resident_per_sm(int threads, int smem_bytes, int *per_sm)
{
    static int cached[kMaxDevices] = {0};
    int &n = cached[current_device()];
    if (!n) {
        int m = 0;
        cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&m, Kernel, threads, smem_bytes);
        if (e != cudaSuccess) return e;
        if (m < 1) return cudaErrorLaunchOutOfResources;
        n = m;
    }
    *per_sm = n;
    return cudaSuccess;
}

// Grid of a persistent FFT kernel: every resident CTA slot, or fewer when there is less work than that
static int persistent_grid(int per_sm, long long work_items)
{
    const long long slots = (long long)per_sm * sm_count();
    return (int)(work_items < slots ? work_items : slots);
}

template <int N, int R1, int R2, int BT, int NW, bool PAIR, bool PAD, int CT, bool BASE = false>
static cudaError_t run_range_t(const PlanDev &p, const int16_t *adc, float2 *rs, int n_frames, cudaStream_t st)
{
    constexpr auto k = range_fft_kernel<N, R1, R2, BT, NW, PAIR, PAD, CT, BASE>;
    constexpr int bytes = RangeSmem<N, BT, BASE>::kBytes;
    int per_sm = 0;
    const cudaError_t e = resident_per_sm<k>(NW * 32, bytes, &per_sm);
    if (e != cudaSuccess) return e;
    const int nct = (p.C + BT - 1) / BT;
    const long long tiles = (long long)n_frames * p.A * nct;
    const int grid = persistent_grid(per_sm, tiles);
    k<<<grid, NW * 32, bytes, st>>>(p, adc, rs, (int)tiles);
    return cudaGetLastError();
}

// picks the PAD / compile-time-chirps specialisation
// BBT / BNW: tile rows and warps of the static-clutter-removal instantiation (the second staging buffer has to fit)
template <int N, int R1, int R2, int BT, int NW, bool PAIR, int CT0, int CT1, int BBT = BT, int BNW = NW>
static cudaError_t run_range(const PlanDev &p, const int16_t *adc, float2 *rs, int n_frames, cudaStream_t st)
{
    if (p.base_adc != nullptr) {          // static-clutter removal: one generic instantiation per padding mode
        if (p.S == N) return run_range_t<N, R1, R2, BBT, BNW, PAIR, false, 0, true>(p, adc, rs, n_frames, st);
        return run_range_t<N, R1, R2, BBT, BNW, PAIR, true, 0, true>(p, adc, rs, n_frames, st);
    }
    if (p.S == N) {
        if (CT0 && p.C == CT0) return run_range_t<N, R1, R2, BT, NW, PAIR, false, CT0>(p, adc, rs, n_frames, st);
        if (CT1 && p.C == CT1) return run_range_t<N, R1, R2, BT, NW, PAIR, false, CT1>(p, adc, rs, n_frames, st);
        return run_range_t<N, R1, R2, BT, NW, PAIR, false, 0>(p, adc, rs, n_frames, st);
    }
    return run_range_t<N, R1, R2, BT, NW, PAIR, true, 0>(p, adc, rs, n_frames, st);
}

template <int N, int R1, int R2, int BT, int NW, bool PAD, int SPT, int NSTAGE, bool INPLACE>
static cudaError_t run_doppler_t(const PlanDev &p, const float2 *rs, float2 *cube, float *pmap, int n_frames, cudaStream_t st)
{
    constexpr auto k = doppler_fft_kernel<N, R1, R2, BT, NW, PAD, SPT, NSTAGE, INPLACE>;
    constexpr int bytes = DopplerSmem<N, BT, NSTAGE, INPLACE>::kBytes;
    int per_sm = 0;
    const cudaError_t e = resident_per_sm<k>(NW * 32, bytes, &per_sm);
    if (e != cudaSuccess) return e;
    const long long tiles = (long long)n_frames * (p.Sp / BT);
    const int grid = persistent_grid(per_sm, tiles);
    k<<<grid, NW * 32, bytes, st>>>(p, rs, cube, pmap, (int)tiles);
    return cudaGetLastError();
}

template <int N, int R1, int R2, int NW, bool PAD, int SPT, int NSTAGE, int MINB = 2>
static cudaError_t run_doppler_warp_t(const PlanDev &p, const float2 *rs, float *pmap, int n_frames, cudaStream_t st)
{
    constexpr auto k = doppler_fft_warp_kernel<N, R1, R2, NW, PAD, SPT, NSTAGE, MINB>;
    using L = DopplerWarp<N, R1, R2>;
    constexpr int bytes = L::bytes(NW, NSTAGE);
    int per_sm = 0;
    const cudaError_t e = resident_per_sm<k>(NW * 32, bytes, &per_sm);
    if (e != cudaSuccess) return e;
    const long long tiles = (long long)n_frames * (p.Sp / L::kRows);
    const long long want = (tiles + NW - 1) / NW;
    const int grid = persistent_grid(per_sm, want);
    k<<<grid, NW * 32, bytes, st>>>(p, rs, pmap, (int)tiles);
    return cudaGetLastError();
}

template <int N, int R1, int R2, int NW, int SP0, int NSTAGE, int MINB = 2>
static cudaError_t run_doppler_warp(const PlanDev &p, const float2 *rs, float *pmap, int n_frames, cudaStream_t st)
{
    if (p.C == N) {
        if (SP0 && p.Sp == SP0) return run_doppler_warp_t<N, R1, R2, NW, false, SP0, NSTAGE, MINB>(p, rs, pmap, n_frames, st);
        return run_doppler_warp_t<N, R1, R2, NW, false, 0, NSTAGE, MINB>(p, rs, pmap, n_frames, st);
    }
    return run_doppler_warp_t<N, R1, R2, NW, true, 0, NSTAGE, MINB>(p, rs, pmap, n_frames, st);
}

template <int N, int R1, int R2, int BT, int NW, int SP0, int SP1, int NSTAGE = 2, bool INPLACE = false>
static cudaError_t run_doppler(const PlanDev &p, const float2 *rs, float2 *cube, float *pmap, int n_frames, cudaStream_t st)
{
    if (p.C == N) {
        if (SP0 && p.Sp == SP0) return run_doppler_t<N, R1, R2, BT, NW, false, SP0, NSTAGE, INPLACE>(p, rs, cube, pmap, n_frames, st);
        if (SP1 && p.Sp == SP1) return run_doppler_t<N, R1, R2, BT, NW, false, SP1, NSTAGE, INPLACE>(p, rs, cube, pmap, n_frames, st);
        return run_doppler_t<N, R1, R2, BT, NW, false, 0, NSTAGE, INPLACE>(p, rs, cube, pmap, n_frames, st);
    }
    return run_doppler_t<N, R1, R2, BT, NW, true, 0, NSTAGE, INPLACE>(p, rs, cube, pmap, n_frames, st);
}

bool plan_supported(int Sp, int Cp, const char **why)
{
    auto ok = [](int n) { return n == 64 || n == 128 || n == 256 || n == 512 || n == 1024; };
    if (!ok(Sp)) { if (why) *why = "range FFT length (nextPow2(n_samples)) must be 64..1024"; return false; }
    if (!ok(Cp)) { if (why) *why = "Doppler FFT length (nextPow2(n_chirps)) must be 64..1024"; return false; }
    return true;
}

// Tile shapes (rows per tile BT, warps per CTA NW) were chosen by sweeping on a B200 (profiles/experiments/README.md):
// BT = 16 keeps two CTAs resident per SM, which hides the barrier between the two passes better than one
// CTA with BT = 32.  The radices must match plan_radices().
cudaError_t launch_range_fft(const PlanDev &p, const int16_t *adc, float2 *rs, int n_frames, cudaStream_t st)
{
    switch (p.Sp) {
    case 64:   return run_range<64, 8, 8, 16, 4, true, 0, 0>(p, adc, rs, n_frames, st);
    case 128:  return run_range<128, 8, 16, 16, 4, true, 128, 0>(p, adc, rs, n_frames, st);
    // double-buffered staging and BT = 8 tiles were measured slower for 256 and 512 points
    // (profiles/experiments/r1_k1_variants_sweep.log)
    // Tile height = bytes per range row in one corner-turned store: a 1 : 2 read:write mover reaches 5.2 TB/s with 128-byte pieces
    // and 5.6-5.7 TB/s with 256-byte ones (profiles/membench_r1.txt).  256 points: 32-row tiles still fit two CTAs of 8 warps per SM
    // and measured 4.5 % faster than 16-row tiles with three CTAs of 4 warps (cfg2 0.293 -> 0.280 ms).  512 points: a 32-row tile
    // needs 203 KB, one CTA of 16 warps per SM, and loses more to the barrier between the passes than the stores gain (0.224 ->
    // 0.238 ms), profiles/experiments/r1_k1_tile_height.log.  Re-measured with tiles from the counter
    // (profiles/r2/sweep_k1_tiles_dynamic.log): same ranking, 8-row tiles at 512 points (four CTAs of 4 warps) 0.225 vs 0.201 ms.
    case 256:  return run_range<256, 16, 16, 32, 8, true, 128, 0, 16, 4>(p, adc, rs, n_frames, st);
    case 512:  return run_range<512, 16, 32, 16, 8, true, 256, 0, 8, 4>(p, adc, rs, n_frames, st);
    // 1024 points: a 16-row tile needs 209 KB (one CTA per SM).  With 8 warps it lost 2.4 % to 8-row tiles at two CTAs per SM
    // (profiles/experiments/r1_cfg4_tile_sweep.log); with 16 warps it wins 1-4 % (64-byte store pieces are the worst case of
    // profiles/membench_r1.txt: 4.2 TB/s), profiles/experiments/r1_k1_tile_height.log.
    case 1024: return run_range<1024, 32, 32, 16, 16, false, 512, 0, 4, 4>(p, adc, rs, n_frames, st);
    default:   return cudaErrorInvalidValue;
    }
}

// (walking the batch from its last frame to its first, so that K2 starts on what K1 wrote last, changed nothing:
// profiles/experiments/r1_k2_frame_order.log)
cudaError_t launch_doppler_fft(const PlanDev &p, const float2 *rs, float2 *cube, float *pmap, int n_frames, cudaStream_t st)
{
    switch (p.Cp) {
    case 64:   return run_doppler<64, 8, 8, 16, 4, 0, 0>(p, rs, cube, pmap, n_frames, st);
    // Other tile shapes, in-place staging and other warp counts were swept and lost: profiles/experiments/r1_k2_variants_sweep.log,
    // profiles/r2/sweep_k2_occupancy.log, profiles/r2/sweep_k2_warp_512_128.log.
    // 128 points: warp-private tiles (K2w, 4 rows x 8 lanes, two butterflies per thread) are slower: 0.222 vs 0.207 ms
    case 128:  return run_doppler<128, 8, 16, 16, 4, 256, 128>(p, rs, cube, pmap, n_frames, st);
    case 256:
        // fused mode (power map only): warp-private tiles, 0.156 vs 0.171 ms on cfg3 (profiles/experiments/r1_k2_warp_private.log)
        if (!cube) return run_doppler_warp<256, 16, 16, 8, 512, 2>(p, rs, pmap, n_frames, st);
        return run_doppler<256, 16, 16, 16, 8, 512, 0>(p, rs, cube, pmap, n_frames, st);
    // 512 points: 8-row tiles, in place, three staging buffers = 103 KB, two CTAs per SM: 0.76 ms against 1.00 ms for the
    // 16-row double-buffered shape (201 KB, one CTA per SM) on the cfg4 cube (profiles/experiments/r1_cfg4_tile_sweep.log)
    // (warp-private tiles at 512 points — 2 rows x 16 lanes, two radix-16 butterflies per lane in pass 1, one radix-32 in pass 2,
    // 165 registers, 12 warps per SM — measured 1.32-1.69 ms against 0.69 on the cfg4 cube: profiles/r2/sweep_k2_warp_512_128.log)
    // four warps per 8-row tile (every slot busy in both passes; 2 or 3 CTAs per SM): 0.80-0.81 ms, same log
    case 512:  return run_doppler<512, 16, 32, 8, 8, 1024, 0, 3, true>(p, rs, cube, pmap, n_frames, st);
    case 1024: return run_doppler<1024, 32, 32, 8, 8, 0, 0>(p, rs, cube, pmap, n_frames, st);
    default:   return cudaErrorInvalidValue;
    }
}

template <int N, int R1, int R2, int BT, int NW, bool PAD>
static cudaError_t run_extract_t(const PlanDev &p, const float2 *rs, const uint32_t *keys, const uint32_t *offsets, const uint4 *rows,
                                 const unsigned int *n_rows, float2 *snap, int dense_cap, int max_rows, cudaStream_t st)
{
    constexpr auto k = doppler_extract_kernel<N, R1, R2, BT, NW, PAD>;
    constexpr int bytes = ExtractSmem<N, BT>::kBytes;
    int per_sm = 0;
    const cudaError_t e = resident_per_sm<k>(NW * 32, bytes, &per_sm);
    if (e != cudaSuccess) return e;
    // the number of hit rows is only known on the device: a persistent grid of every resident CTA, capped by the most work
    // items there can be (a tile's antennas are split into chunks of >= 4 inside the kernel); idle CTAs leave at once
    const long long items_max = (((long long)max_rows + BT - 1) / BT) * ((p.A + 3) / 4);
    const long long resident = (long long)per_sm * sm_count();
    const int grid = (int)(items_max < resident ? (items_max < 1 ? 1 : items_max) : resident);
    k<<<grid, NW * 32, bytes, st>>>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap);
    return cudaGetLastError();
}

template <int N, int R1, int R2, int BT, int NW>
static cudaError_t run_extract(const PlanDev &p, const float2 *rs, const uint32_t *keys, const uint32_t *offsets, const uint4 *rows,
                               const unsigned int *n_rows, float2 *snap, int dense_cap, int max_rows, cudaStream_t st)
{
    if (p.C == N) return run_extract_t<N, R1, R2, BT, NW, false>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    return run_extract_t<N, R1, R2, BT, NW, true>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
}

// max_rows: upper bound of the hit rows (n_frames * Sp); the true count is read from *n_rows on the device
cudaError_t launch_doppler_extract(const PlanDev &p, const float2 *rs, const uint32_t *keys, const uint32_t *offsets, const uint4 *rows,
                                   const unsigned int *n_rows, float2 *snap, int dense_cap, int max_rows, cudaStream_t st)
{
    switch (p.Cp) {
    case 64:   return run_extract<64, 8, 8, 8, 4>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    case 128:  return run_extract<128, 8, 16, 8, 4>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    case 256:  return run_extract<256, 16, 16, 8, 8>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    case 512:  return run_extract<512, 16, 32, 8, 8>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    case 1024: return run_extract<1024, 32, 32, 8, 8>(p, rs, keys, offsets, rows, n_rows, snap, dense_cap, max_rows, st);
    default:   return cudaErrorInvalidValue;
    }
}

cudaError_t launch_export_cube(const PlanDev &p, const float2 *cube_frame, float2 *out, cudaStream_t st)
{
    export_cube_kernel<<<592, 256, 0, st>>>(cube_frame, out, p.A, p.Sp, p.Cp);
    return cudaGetLastError();
}
cudaError_t launch_export_pmap(const PlanDev &p, const float *pmap_frame, float *out, cudaStream_t st)
{
    export_pmap_kernel<<<296, 256, 0, st>>>(pmap_frame, out, p.Sp, p.Cp);
    return cudaGetLastError();
}
cudaError_t launch_export_mask(const PlanDev &p, const uint32_t *mask_frame, uint8_t *out, cudaStream_t st)
{
    export_mask_kernel<<<296, 256, 0, st>>>(mask_frame, out, p.Sp, p.Cp);
    return cudaGetLastError();
}

}  // namespace mmw
