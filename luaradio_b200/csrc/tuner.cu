// Register-tiled polyphase decimating FIR (complex in, real taps) with an optional fused frequency
// translator in front and an optional fused frequency discriminator behind: the TunerBlock / DecimatorBlock
// kernel, and the dominant kernel of the WBFM-mono chain.
//
// Reference dataflow being fused (composites/tuner.lua:40-47, examples/rtlsdr_wbfm_mono.lua:12-14):
//     FrequencyTranslatorBlock(offset) -> LowpassFilterBlock(128, bw/2) -> DownsamplerBlock(D) [-> FrequencyDiscriminator]
// i.e. three (four) processes and socket hops, with the FIR computing D times more outputs than are kept
// (firfilter.lua:121-124 runs one dot product per INPUT sample).  Here only the kept outputs are computed
// (M/D complex-by-real MACs per input sample) and the input is read from HBM exactly once:
// algorithmic traffic 8 + 8/D bytes per input sample (8 + 4/D with the discriminator fused).
//
// Tile.  A CTA produces PT_TO = PT_THREADS (64) threads x R = 8 consecutive decimated outputs from one shared-memory tile of
// rotated input samples kept in their natural (interleaved) order.  With reversed taps hr[0 .. T), T = Q*D + 1
// (Q = ceil(M/D); one spare leading tap lets the host make every tile start on an even input index, so every
// global load is an aligned 128-bit load and there is a single code path), and B the first input the tile needs,
//     y[m0 + r] = sum_{i' < T} hr[i'] * X[B + r*D + i'].
// A thread walks window positions j = 0 .. R+Q-1; at each it loads the D consecutive samples X[B + (tR + j)D + p]
// (40 contiguous bytes for D = 5: two LDS.128 + one LDS.64) and feeds them to every output r with 0 <= j-r <= Q:
// one packed FFMA2 (f32x2 complex sample x scalar-broadcast real tap from the constant bank) per MAC, no
// register window to rotate, no de-interleaving.  Thread t's samples start at element t*(R*D) and the layout is
// padded by 2 samples every R*D, which makes the per-thread stride (R*D+2)*8 B conflict-free for 128-bit loads.
//
// Rotation.  x[i] e^{jw(g0+i)} = P_tile * (x[i] * E[i - B]) with E the tile-relative phasor and P_tile the phasor of
// the tile origin.  E is applied while staging: a thread always stages the same tile-relative sample pairs, so
// E[2u] = A0 * step[it] with A0 = E[2 tid] held in registers for the whole (persistent) kernel and step[it] a
// per-iteration constant from the constant bank -- no table stream, no transcendental per sample.  P_tile commutes
// with the filter and is applied to the 1/D kept outputs (not at all under the fused discriminator, which only
// sees y[m] conj(y[m-1])).
//
// History of this kernel (ncu summaries in profiles/): v1 guarded loads, 1.43 ms per 256 Mi samples, 85 % of
// stall samples on first use of a load; v2 batched loads 0.90 ms; v3 persistent + cross-tile prefetch + fused
// discriminator 1.00 ms (0.90 + 0.13 before); a warp-specialised producer/consumer variant of v3 gained only 5 %
// because v3 was issue-bound, not latency-bound: 60 instructions per staged sample PAIR (de-interleave index
// arithmetic + two phasor products).  v4 (natural-order tile, ~13 instructions per pair, phasor table) 0.82 ms with
// 42 % of the stall samples on the staging loads; v5 (this file: phasors by arithmetic, deeper prefetch, packed
// 25-instruction atan2 epilogue) 0.73-0.75 ms, FP32 pipe 67 % active.
#include "common.cuh"
#include "blocks.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

namespace lrb {

namespace {

#ifndef LRB_PT_THREADS
// 64-thread CTAs, 8 per SM (round 2; was 128 x 4): the same 16 warps and 180 KB of tiles per SM in twice as many,
// half-sized barrier domains -- 2.8 % faster on the chain's tuner stage, and a short call spreads over twice as many
// CTAs (lower latency per vector); the 26-block halo of a tile is 5 % of its loads instead of 2.5 % (L2 hits)
#define LRB_PT_THREADS 64
#define LRB_PT_R 8
#define LRB_PT_CTAS 8
#define LRB_PT_PREFETCH 9
#define LRB_PT_BATCH 7
#endif
#ifndef LRB_PT_EXPERIMENT
#define LRB_PT_EXPERIMENT 0      // timing experiments only: 1 = stage the first tile only, 2 = skip the MAC loop
#endif
#ifndef LRB_PT_EARLY_REST
#define LRB_PT_EARLY_REST 0
#endif
constexpr int PT_THREADS = LRB_PT_THREADS;
constexpr int PT_R = LRB_PT_R;
constexpr int PT_TO = PT_THREADS * PT_R;     // filter outputs per tile
constexpr int PT_MAXTAPS = 144;              // Q*D + 1 upper bound for the instantiated shapes
constexpr int PT_BATCH = LRB_PT_BATCH;       // 128-bit loads issued back to back per staging batch

constexpr int PT_MAXIT = 48;                 // staging iterations (pairs per thread) upper bound
struct PolyParams {
    float hr[PT_MAXTAPS];        // reversed taps with the launch's alignment shift, zero padded to Q*D + 1
    float2 step[PT_MAXIT];       // exp(j*2*pi*turns * 2*PT_THREADS*it): phasor advance of staging iteration `it`
    uint64_t turns_fix;          // turns per sample, 2^-64 units
    uint64_t g0;                 // global index of x[0]
    long long off;               // B(tile) = off + tile * TS * D   (even)
    int M;
    float pole_c;                // POLE: the output-rate pole c (z[m] = c z[m-1] + w[m])
    float pole_cp[6];            // c^(R * 2^k), k < 5; c^(R * 32)
};
// POLE: outputs of warm-up in front of every run (|c|^PT_POLE_WARM <= 1e-8 is required by the host); a whole number of
// threads' outputs and a multiple of 4 (16-byte aligned stores)
constexpr int PT_POLE_WARM = (64 % LRB_PT_R == 0) ? 64 : ((72 % LRB_PT_R == 0) ? 72 : 4 * LRB_PT_R);
static_assert(PT_POLE_WARM % LRB_PT_R == 0 && PT_POLE_WARM % 4 == 0 && PT_POLE_WARM >= 64, "pole warm-up must cover whole threads");

template <int D, int Q>
struct PolyShape {
    static constexpr int RD = PT_R * D;                          // samples per thread per window step block
    static constexpr int T = Q * D + 1;                          // taps incl. the alignment spare
    static constexpr int SPAN = (PT_TO + Q - 1) * D + 1;         // samples a tile needs: e in [0, SPAN)
    static constexpr int PAIRS = (SPAN + 1) / 2;
    static constexpr int ITERS = (PAIRS + PT_THREADS - 1) / PT_THREADS;
    static constexpr int LOADED = 2 * ITERS * PT_THREADS;        // samples actually staged (>= SPAN)
    __host__ __device__ static constexpr int pad(int e) { return e + 2 * (e / RD); }
    static constexpr int ELEMS = LOADED + 2 * (LOADED / RD) + 2;
    static constexpr size_t SMEM = (size_t)ELEMS * sizeof(float2);
};

// compile-time loop: f(std::integral_constant<int, I>) for I in [B, E) -- guarantees full unrolling with
// constant register indices (a plain `#pragma unroll` gave up on the 34 x 8 x 5 nest and spilled to indexing)
template <int B, int E, typename F>
__device__ __forceinline__ void static_for(F&& f) {
    if constexpr (B < E) {
        f(std::integral_constant<int, B>{});
        static_for<B + 1, E>(f);
    }
}

// DISC: consecutive tiles overlap by two outputs (tile stride PT_TO - 2, even so that tile origins keep their
// parity): slot 0 is the output just before the tile's first discriminator output, slot PT_TO-1 is unused.
template <bool DISC>
struct TileStride { static constexpr int TS = DISC ? PT_TO - 2 : PT_TO; };

// REAL: real input, real taps, real output (the audio low-pass + de-emphasis + Downsampler(5) stage of the chain,
// firfilter.lua:147-163 behind the noble identity, see graph.cu).  The two lanes of every packed register are two
// INDEPENDENT real streams: element e of the staged tile is (xr[B + e], xr[B + PT_TO*D + e]), so lane 0 computes the
// tile's first PT_TO outputs and lane 1 the next PT_TO, and every FFMA2 of the unchanged compute phase is two useful
// real MACs.  x / hist then point to float32 data.
//
// POLE (REAL only): a single pole at the OUTPUT rate fused behind the filter, z[m] = c z[m-1] + w[m] (the c^D pole the
// noble identity leaves of an IIR in front of a Downsampler, graph.cu).  Each lane's run of PT_TO outputs starts with
// PT_POLE_WARM outputs of warm-up that are scanned but not stored (runs overlap by that much), so a run needs nothing
// from its predecessor beyond float32 resolution; the stream's very first run takes the carried state instead.  The
// scan is thread-sequential (R) -> warp Kogge-Stone -> Horner over the 4 warps, both lanes at once on packed registers.
template <int D, int Q, bool ROT, bool DISC, bool EDGE, bool REAL = false, bool POLE = false>
__global__ void __launch_bounds__(PT_THREADS, LRB_PT_CTAS)
polyphase_crcf_kernel(const float2* __restrict__ x, const float2* __restrict__ hist, long long n,
                      void* __restrict__ yv, long long n_out, const __grid_constant__ PolyParams P,
                      long long t_lo, long long t_hi,
                      const float2* __restrict__ prev_in, float2* __restrict__ prev_out, float inv_gain) {
    using S = PolyShape<D, Q>;
    static_assert(!(REAL && (ROT || DISC)), "the real-stream variant has no translator / discriminator");
    static_assert(REAL || !POLE, "the fused pole exists in the real-stream variant only");
    constexpr int PW = POLE ? PT_POLE_WARM : 0;                    // warm-up outputs in front of each lane's run
    constexpr int PAY = PT_TO - PW;                                // outputs a lane's run stores
    constexpr int TS = REAL ? 2 * PAY : TileStride<DISC>::TS;      // outputs per tile
    constexpr int NPRE = S::ITERS < LRB_PT_PREFETCH ? S::ITERS : LRB_PT_PREFETCH;   // pairs prefetched across the compute phase
    constexpr int LANE1 = PAY * D;                                 // REAL: input distance between the two lanes' streams
    const float* __restrict__ xr = reinterpret_cast<const float*>(x);
    const float* __restrict__ histr = reinterpret_cast<const float*>(hist);
    extern __shared__ __align__(16) float2 smem[];
    __shared__ float2 s_edge[PT_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Hm1 = P.M - 1;

    // tile-relative phasors of this thread's first sample pair, E[2 tid] and E[2 tid + 1]; the pair of staging
    // iteration `it` is 2*PT_THREADS*it samples later: E[2u] = A0 * step[it].  (A phasor TABLE in global memory
    // cost one more load stream whose latency was exposed three times per tile -- 42 % of all stall samples.)
    float2 A0 = make_float2(1.f, 0.f), A1 = make_float2(1.f, 0.f);
    if constexpr (ROT) {
        A0 = phasor_from_fix(P.turns_fix * (uint64_t)(2 * tid));
        A1 = phasor_from_fix(P.turns_fix * (uint64_t)(2 * tid + 1));
    }
    auto tile_of = [&](long long idx) -> long long { return EDGE ? (idx < t_lo ? idx : t_hi + (idx - t_lo)) : (t_lo + idx); };
    const long long n_work = EDGE ? 0 : (t_hi - t_lo);
    long long widx = blockIdx.x;

    // staging addresses: pair u = tid + 128*it holds samples e = 2u, 2u+1 -> padded element 2u + 2*floor(2u / RD)
    // (RD is even, so a pair never straddles a padding gap and stays 16-byte aligned)
    // pair u = tid + k*PT_THREADS of the tile whose first input index is Bt, as (elem 2u, elem 2u+1)
    auto ld_pair = [&](long long Bt, int k) -> float4 {
        if constexpr (REAL) {
            const float2* pa = reinterpret_cast<const float2*>(xr + Bt) + (tid + k * PT_THREADS);
            const float2 a = __ldcs(pa), b = __ldcs(pa + LANE1 / 2);
            return make_float4(a.x, b.x, a.y, b.y);
        } else {
            return __ldcs(reinterpret_cast<const float4*>(x + Bt) + (tid + k * PT_THREADS));
        }
    };
    float4 pre[NPRE];
    // the next REST pairs: requested before the EPILOGUE of the previous tile (LRB_PT_EARLY_REST), so that their latency
    // hides behind the epilogue's dependent chains instead of being exposed at the top of the staging phase (ncu, round 2:
    // 44 % of the stall samples sat in the staging / epilogue regions, mostly long-scoreboard waits on these loads)
    constexpr int REST = (S::ITERS - NPRE) < PT_BATCH ? (S::ITERS - NPRE) : PT_BATCH;
    float4 rest[REST > 0 ? REST : 1];
    if constexpr (!EDGE) {
        if (widx < n_work) {
            const long long Bt = P.off + tile_of(widx) * (long long)(TS * D);
#pragma unroll
            for (int k = 0; k < NPRE; ++k) pre[k] = ld_pair(Bt, k);
            if constexpr (LRB_PT_EARLY_REST) {
#pragma unroll
                for (int k = 0; k < REST; ++k) rest[k] = ld_pair(Bt, NPRE + k);
            }
        }
    }

    for (;;) {
        if constexpr (!EDGE) { if (widx >= n_work) break; }
        const long long tile = tile_of(widx);
        const long long B = P.off + tile * (long long)(TS * D);      // first input index of the tile (even)
        const long long m0 = tile * TS - (DISC ? 1 : 0) - PW;        // output index of slot 0

        // ---- stage: global -> (x E) -> shared, natural order
        auto stage_pair = [&](float4 v, int it) {
            const int u = tid + it * PT_THREADS;
            float2 a = make_float2(v.x, v.y), b = make_float2(v.z, v.w);
            if constexpr (ROT) {
                const float2 st = P.step[it];
                a = cmul(a, cmul(A0, st));
                b = cmul(b, cmul(A1, st));
            }
            *reinterpret_cast<float4*>(smem + S::pad(2 * u)) = make_float4(a.x, a.y, b.x, b.y);
        };
        if constexpr (!EDGE && LRB_PT_EXPERIMENT == 1) {
            if (widx == blockIdx.x) {
#pragma unroll 1
                for (int it = 0; it < S::ITERS; ++it) stage_pair(ld_pair(B, it), it);
            }
        } else if constexpr (!EDGE) {
            // the first NPRE pairs were prefetched during the previous tile's compute phase; the rest of the tile
            // is requested now and lands while those are rotated and stored
            if constexpr (!LRB_PT_EARLY_REST) {
#pragma unroll
                for (int k = 0; k < REST; ++k) rest[k] = ld_pair(B, NPRE + k);
            }
#pragma unroll
            for (int k = 0; k < NPRE; ++k) stage_pair(pre[k], k);
#pragma unroll
            for (int k = 0; k < REST; ++k) stage_pair(rest[k], NPRE + k);
#pragma unroll 1
            for (int it0 = NPRE + REST; it0 < S::ITERS; it0 += PT_BATCH) {
                float4 buf[PT_BATCH];
#pragma unroll
                for (int k = 0; k < PT_BATCH; ++k)
                    if (it0 + k < S::ITERS) buf[k] = ld_pair(B, it0 + k);
#pragma unroll
                for (int k = 0; k < PT_BATCH; ++k)
                    if (it0 + k < S::ITERS) stage_pair(buf[k], it0 + k);
            }
        } else {
#pragma unroll 7
            for (int it = 0; it < S::ITERS; ++it) {
                const long long i0 = B + 2LL * (tid + it * PT_THREADS);
                if constexpr (REAL) {
                    auto g = [&](long long i) -> float {
                        return (i >= 0) ? (i < n ? __ldg(xr + i) : 0.f) : ((Hm1 + i >= 0) ? __ldg(histr + (Hm1 + i)) : 0.f);
                    };
                    stage_pair(make_float4(g(i0), g(i0 + LANE1), g(i0 + 1), g(i0 + 1 + LANE1)), it);
                    continue;
                }
                const float2 a = (i0 >= 0) ? (i0 < n ? __ldg(x + i0) : make_float2(0.f, 0.f))
                                           : ((Hm1 + i0 >= 0) ? __ldg(hist + (Hm1 + i0)) : make_float2(0.f, 0.f));
                const long long i1 = i0 + 1;
                const float2 b = (i1 >= 0) ? (i1 < n ? __ldg(x + i1) : make_float2(0.f, 0.f))
                                           : ((Hm1 + i1 >= 0) ? __ldg(hist + (Hm1 + i1)) : make_float2(0.f, 0.f));
                stage_pair(make_float4(a.x, a.y, b.x, b.y), it);
            }
        }
        __syncthreads();

        // ---- prefetch the first batch of this CTA's next tile; it stays in registers across the compute phase
        if constexpr (!EDGE && LRB_PT_EXPERIMENT != 1) {
            const long long nidx = widx + gridDim.x;
            if (nidx < n_work) {
                const long long Bn = P.off + tile_of(nidx) * (long long)(TS * D);
#pragma unroll
                for (int k = 0; k < NPRE; ++k) pre[k] = ld_pair(Bn, k);
            }
        }

        // ---- compute: walk the window positions; every position feeds all outputs it overlaps
        float2 acc[PT_R];
#pragma unroll
        for (int r = 0; r < PT_R; ++r) acc[r] = make_float2(0.f, 0.f);
        const float2* tb = smem + tid * (S::RD + 2);
        static_for<0, (LRB_PT_EXPERIMENT == 2 ? 1 : PT_R + Q)>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            // samples X[B + (tid*R + j)*D + p], p < D: padded offset j*D + p + 2*floor((j*D + p)/RD)
            float2 xs[D];
            constexpr int e0 = j * D;
            if constexpr (j == PT_R + Q - 1) {
                xs[0] = tb[S::pad(e0)];                            // the last position only feeds tap Q*D (p = 0)
            } else {
                static_for<0, D>([&](auto pc) {
                    constexpr int pp = decltype(pc)::value;
                    constexpr int e = e0 + pp;
                    if constexpr ((e & 1) && pp >= 1) {
                        // already loaded as the upper half of a 128-bit pair
                    } else if constexpr (!(e & 1) && pp + 1 < D) {
                        const float4 v = *reinterpret_cast<const float4*>(tb + S::pad(e));
                        xs[pp] = make_float2(v.x, v.y);
                        xs[pp + 1] = make_float2(v.z, v.w);
                    } else {
                        xs[pp] = tb[S::pad(e)];
                    }
                });
            }
            static_for<0, PT_R>([&](auto rc) {
                constexpr int r = decltype(rc)::value;
                constexpr int qq = j - r;
                if constexpr (qq >= 0 && qq <= Q) {
                    static_for<0, D>([&](auto pc) {
                        constexpr int pp = decltype(pc)::value;
                        if constexpr (qq * D + pp < S::T) {
                            const float h = P.hr[qq * D + pp];
                            acc[r] = __ffma2_rn(xs[pp], make_float2(h, h), acc[r]);
                        }
                    });
                }
            });
        });
        if constexpr (!EDGE && LRB_PT_EARLY_REST) {
            const long long nidx = widx + gridDim.x;
            if (nidx < n_work) {
                const long long Bn = P.off + tile_of(nidx) * (long long)(TS * D);
#pragma unroll
                for (int k = 0; k < REST; ++k) rest[k] = ld_pair(Bn, NPRE + k);
            }
        }
        // tile phasor: the staged samples carry only the tile-relative rotation E; P_tile = exp(jw(g0 + B)) commutes
        // with the filter.  The discriminator output y[m] conj(y[m-1]) does not depend on it (|P| = 1), so with DISC
        // it is only applied to the two samples that cross the call boundary (prev_in / prev_out).
        if constexpr (ROT && !DISC) {
            const float2 Pt = phasor_from_fix(P.turns_fix * (P.g0 + (uint64_t)B));
#pragma unroll
            for (int r = 0; r < PT_R; ++r) acc[r] = cmul(acc[r], Pt);
        }

        const long long mbase = m0 + (long long)tid * PT_R;     // output index of acc[0]
        if constexpr (POLE) {
            const float c = P.pole_c;
            if (tile == 0 && tid < PW / PT_R) {
                // the stream's first run: the carried state z[-1] takes the place of the warm-up (whose inputs precede
                // the M-1 samples of history the block keeps)
#pragma unroll
                for (int r = 0; r < PT_R; ++r) acc[r].x = 0.f;
                if (tid == PW / PT_R - 1) acc[PT_R - 1].x = __ldg(reinterpret_cast<const float*>(prev_in));
            }
#pragma unroll
            for (int r = 1; r < PT_R; ++r) acc[r] = __ffma2_rn(acc[r - 1], make_float2(c, c), acc[r]);
            float2 Bv = acc[PT_R - 1];                        // zero-state end value of this thread's R outputs
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float2 o = make_float2(__shfl_up_sync(0xffffffffu, Bv.x, 1 << k), __shfl_up_sync(0xffffffffu, Bv.y, 1 << k));
                if (lane >= (1 << k)) Bv = __ffma2_rn(o, make_float2(P.pole_cp[k], P.pole_cp[k]), Bv);
            }
            if (lane == 31) s_edge[warp] = Bv;
            float2 prevB = make_float2(__shfl_up_sync(0xffffffffu, Bv.x, 1), __shfl_up_sync(0xffffffffu, Bv.y, 1));
            if (lane == 0) prevB = make_float2(0.f, 0.f);
            __syncthreads();                                  // (the tile's last shared-memory read is behind every thread)
            float2 carryW = make_float2(0.f, 0.f);
            for (int w = 0; w < warp; ++w) carryW = __ffma2_rn(carryW, make_float2(P.pole_cp[5], P.pole_cp[5]), s_edge[w]);
            float f_lane = 1.f;
#pragma unroll
            for (int k = 0; k < 5; ++k) if (lane & (1 << k)) f_lane *= P.pole_cp[k];
            const float2 excl = __ffma2_rn(carryW, make_float2(f_lane, f_lane), prevB);   // z just before acc[0]
            float cpow = c;
#pragma unroll
            for (int r = 0; r < PT_R; ++r) { acc[r] = __ffma2_rn(excl, make_float2(cpow, cpow), acc[r]); cpow *= c; }
        }
        if constexpr (REAL) {
            // ---- store: lane 0 -> outputs mbase + r, lane 1 -> outputs mbase + PAY + r (slots below PW are warm-up)
            float* y = reinterpret_cast<float*>(yv);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const long long mb = mbase + half * PAY;
                if (POLE && tid < PW / PT_R) continue;
                float v[PT_R];
#pragma unroll
                for (int r = 0; r < PT_R; ++r) v[r] = half ? acc[r].y : acc[r].x;
                if (mb + PT_R <= n_out && ((reinterpret_cast<uintptr_t>(y + mb) & 15) == 0)) {
#pragma unroll
                    for (int r = 0; r < PT_R; r += 4)
                        __stcs(reinterpret_cast<float4*>(y + mb + r), make_float4(v[r], v[r + 1], v[r + 2], v[r + 3]));
                } else {
#pragma unroll
                    for (int r = 0; r < PT_R; ++r)
                        if (mb + r < n_out) y[mb + r] = v[r];
                }
                if constexpr (POLE) {
                    // the call's last output is the carried state of the next call
                    if (mb <= n_out - 1 && n_out - 1 < mb + PT_R) {
#pragma unroll
                        for (int r = 0; r < PT_R; ++r)
                            if (mb + r == n_out - 1) *reinterpret_cast<float*>(prev_out) = v[r];
                    }
                }
            }
            __syncthreads();                               // shared tile is reused by the next iteration
        } else if constexpr (!DISC) {
            // ---- store: 8 consecutive complex outputs per thread
            float2* y = reinterpret_cast<float2*>(yv);
            if (mbase + PT_R <= n_out && ((reinterpret_cast<uintptr_t>(y + mbase) & 15) == 0)) {
                float4* y4 = reinterpret_cast<float4*>(y + mbase);
#pragma unroll
                for (int r = 0; r < PT_R; r += 2)
                    __stcs(y4 + r / 2, make_float4(acc[r].x, acc[r].y, acc[r + 1].x, acc[r + 1].y));
            } else {
#pragma unroll
                for (int r = 0; r < PT_R; ++r)
                    if (mbase + r < n_out) y[mbase + r] = acc[r];
            }
            __syncthreads();                               // shared tile is reused by the next iteration
        } else {
            // ---- fused FrequencyDiscriminator (frequencydiscriminator.lua:68-88):
            //      d[m] = atan2(im, re of y[m] * conj(y[m-1])) * (1/gain); slot 0 only supplies y[m-1] for slot 1
            float* yd = reinterpret_cast<float*>(yv);
            float2 left;                                   // y just before acc[0]
            left.x = __shfl_up_sync(0xffffffffu, acc[PT_R - 1].x, 1);
            left.y = __shfl_up_sync(0xffffffffu, acc[PT_R - 1].y, 1);
            if (lane == 31) s_edge[warp] = acc[PT_R - 1];
            __syncthreads();                               // also fences the shared tile for the next iteration
            if (lane == 0 && warp > 0) left = s_edge[warp - 1];
            bool zero_prev = false;                        // the carried sample is exactly (0, 0): stream start
            if (tid == 0 && tile == 0) {
                // stream state: the previous call's last output (absolute phase) brought into this tile's frame
                const float2 Pt = ROT ? phasor_from_fix(P.turns_fix * (P.g0 + (uint64_t)B)) : make_float2(1.f, 0.f);
                const float2 pv = __ldg(prev_in);
                acc[0] = cmul(pv, make_float2(Pt.x, -Pt.y));
                if constexpr (EDGE) zero_prev = pv.x == 0.f && pv.y == 0.f;   // tile 0 reaches into the history: always an edge tile
            }
            // slots are tile-relative 32-bit indices: slot s holds y[m0 + s]; slots 1 .. lim-1 produce outputs
            const long long room = n_out - m0;             // > 1 for every launched tile
            const int lim = room < (long long)(TS + 1) ? (int)room : TS + 1;
            const int s0 = tid * PT_R;
            float* yt = yd + m0;
            // y[m] * conj(y[m-1]) for the 8 slots, two at a time on packed lanes
            float dout[PT_R];
#pragma unroll
            for (int r = 0; r < PT_R; r += 2) {
                const float2 c0 = acc[r], p0 = (r == 0) ? left : acc[r - 1];
                const float2 c1 = acc[r + 1], p1 = acc[r];
                // c * conj(p) = (c.x p.x + c.y p.y,  c.y p.x - c.x p.y)
                const float2 t0 = __ffma2_rn(c0, make_float2(p0.x, p0.x), __fmul2_rn(make_float2(c0.y, -c0.x), make_float2(p0.y, p0.y)));
                const float2 t1 = __ffma2_rn(c1, make_float2(p1.x, p1.x), __fmul2_rn(make_float2(c1.y, -c1.x), make_float2(p1.y, p1.y)));
                const float2 ang = fast_atan2f_x2(make_float2(t0.y, t1.y), make_float2(t0.x, t1.x));
                dout[r] = ang.x * inv_gain;
                dout[r + 1] = ang.y * inv_gain;
            }
            if (EDGE && zero_prev) {
                // y[0] * conj(0): the reference multiplies by prev_sample = ComplexFloat32() all the same
                // (frequencydiscriminator.lua:72, complexfloat32.lua:79-81) and takes atan2f of a product of SIGNED zeros:
                // real = yr*0 - yi*(-0) is -0 when yr and yi are both negative, and atan2f(+0, -0) = pi -- a click of
                // pi / gain at the start of one stream in four.  The packed fast atan2 above works in the tile's rotated
                // frame and tests x < 0, so this one sample is redone in the absolute frame with IEEE operations.
                const float2 Pt = ROT ? phasor_from_fix(P.turns_fix * (P.g0 + (uint64_t)B)) : make_float2(1.f, 0.f);
                const float2 ya = ROT ? cmul(acc[1], Pt) : acc[1];
                const float pz = 0.f, nz = -0.f;
                const float re = __fsub_rn(__fmul_rn(ya.x, pz), __fmul_rn(ya.y, nz));
                const float im = __fadd_rn(__fmul_rn(ya.x, nz), __fmul_rn(ya.y, pz));
                dout[1] = atan2f(im, re) * inv_gain;
            }
#pragma unroll
            for (int r = 0; r < PT_R; ++r) {
                const int sl = s0 + r;
                if (sl >= 1 && sl < lim) {
                    yt[sl] = dout[r];
                    if ((long long)sl == room - 1) {        // last output of the call: carried to the next one, in absolute phase
                        const float2 Pt = ROT ? phasor_from_fix(P.turns_fix * (P.g0 + (uint64_t)B)) : make_float2(1.f, 0.f);
                        *prev_out = cmul(acc[r], Pt);
                    }
                }
            }
        }
        if constexpr (EDGE) break;
        widx += gridDim.x;
    }
}

template <int D, int Q, bool ROT, bool DISC, bool REAL = false, bool POLE = false>
int launch_shape(PolyParams P, const float* hr_base, const float2* x, const float2* hist, long long n,
                 void* y, long long first, long long n_out, const float2* prev_in, float2* prev_out, float inv_gain,
                 cudaStream_t s) {
    using S = PolyShape<D, Q>;
    static_assert(S::T <= PT_MAXTAPS, "taps table too small");
    // function attributes are per device: a process that drives several GPUs configures each once
    static bool configured_dev[LRB_MAX_DEVICES] = {false};
    static int ctas_dev[LRB_MAX_DEVICES] = {0};
    bool& configured = configured_dev[ctx().device & (LRB_MAX_DEVICES - 1)];
    int& ctas_per_sm = ctas_dev[ctx().device & (LRB_MAX_DEVICES - 1)];
    auto kern_i = polyphase_crcf_kernel<D, Q, ROT, DISC, false, REAL, POLE>;
    auto kern_e = polyphase_crcf_kernel<D, Q, ROT, DISC, true, REAL, POLE>;
    if (!configured) {
        LRB_CHECK(cudaFuncSetAttribute(kern_i, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::SMEM));
        LRB_CHECK(cudaFuncSetAttribute(kern_e, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::SMEM));
        LRB_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern_i, PT_THREADS, S::SMEM));
        if (ctas_per_sm < 1) ctas_per_sm = 1;
        configured = true;
    }
    constexpr int PW = POLE ? PT_POLE_WARM : 0;
    constexpr int PAY = PT_TO - PW;
    constexpr int TS = REAL ? 2 * PAY : TileStride<DISC>::TS;
    // B(tile) = first + m0*D - (Q*D - 1) - shift, m0 = tile*TS - (DISC ? 1 : 0) - PW; shift in {0,1} makes it even
    long long off = first - (DISC ? D : 0) - (long long)PW * D - (long long)(Q * D - 1);
    const int shift = (int)(((off % 2) + 2) % 2);
    off -= shift;
    P.off = off;
    // hr'[i'] = hr[i' - shift] (hr_base has Q*D entries): one spare zero tap at either end
    for (int i = 0; i < PT_MAXTAPS; ++i) {
        const int k = i - shift;
        P.hr[i] = (k >= 0 && k < Q * D) ? hr_base[k] : 0.0f;
    }
    const long long tiles = (n_out + TS - 1) / TS;
    // interior tiles: every staged sample B(t) .. B(t)+LOADED-1 inside [lead, n) and x 16-byte aligned (lead > 0: the
    // first samples arrive with the neighbour exchange of a sharded run, see Ctx::lead_samples)
    cudaEvent_t lead_event = ctx().lead_samples > 0 ? ctx().lead_event : nullptr;
    const long long lead = lead_event ? ctx().lead_samples : 0;
    long long t_lo = 0, t_hi = 0;
    if ((reinterpret_cast<uintptr_t>(x) & (REAL ? 7 : 15)) == 0) {
        const long long step = (long long)TS * D;
        const long long need = lead - off;                                   // B(t) = off + t * step >= lead
        t_lo = need <= 0 ? 0 : (need + step - 1) / step;
        const long long lim = n - (long long)S::LOADED - off - (REAL ? (long long)PAY * D : 0);
        t_hi = lim < 0 ? 0 : lim / step + 1;
        if (t_hi > tiles) t_hi = tiles;
        if (t_lo > t_hi) t_lo = t_hi;
    }
    const long long n_int = t_hi - t_lo, n_edge = tiles - n_int;
    // the edge tiles (first / last few) go to the side stream so that they overlap the interior kernel
    cudaStream_t side = ((n_int > 0 && n_edge > 0) || (lead_event && n_edge > 0)) ? side_fork(s) : s;
    if (n_edge > 0) {
        if (lead_event && side != s) LRB_CHECK(cudaStreamWaitEvent(side, lead_event, 0));
        else if (lead_event) LRB_CHECK(cudaStreamWaitEvent(s, lead_event, 0));
        kern_e<<<(unsigned)n_edge, PT_THREADS, S::SMEM, side>>>(x, hist, n, y, n_out, P, t_lo, t_hi, prev_in, prev_out, inv_gain);
        count_launch();
    }
    if (n_int > 0) {
        long long grid = (long long)ctx().sm_count * ctas_per_sm - ctx().reserve_ctas;
        if (grid < 1) grid = 1;
        if (grid > n_int) grid = n_int;
        kern_i<<<(unsigned)grid, PT_THREADS, S::SMEM, s>>>(x, hist, n, y, n_out, P, t_lo, t_hi, prev_in, prev_out, inv_gain);
        count_launch();
    }
    side_join(s, side);
    LRB_CHECK(cudaGetLastError());
    return 1;
}

}  // namespace

struct PolyTaps {
    int M, D, Q;
    float hr[PT_MAXTAPS];        // reversed taps, Q*D entries: hr[i'] = h[Q*D-1-i']
    uint64_t turns_fix;
    float2 step[PT_MAXIT];       // per-staging-iteration phasor advance (see PolyParams)
    bool rotates = false;        // a translator is fused
    bool real_data = false;      // float32 stream (REAL kernel variant)
};

static int shape_q(int M, int D, bool rotates) {
    // Instantiated shapes.  Each one is a handful of fully unrolled ~2500-instruction kernels (minutes of ptxas
    // time), so the list is exactly what the reference's own graphs produce on the hot path:
    //   (D, Q) = (5, 26): TunerBlock / DecimatorBlock with the default 128 taps and decimation 5
    //            (examples/rtlsdr_wbfm_mono.lua), with or without the translator / discriminator;
    //   (1, 16), (1, 32): plain FIRs with up to 16 / 32 real taps (below the overlap-save break-even).
    // Every other decimating or translating FIR runs the overlap-save kernel (fir_fft.cu), which fuses both.
    if (D == 1 && !rotates) return M <= 16 ? 16 : (M <= 32 ? 32 : 0);
    if (D == 5 && M > 65 && M <= 128) return 26;
    return 0;
}

// real input / real taps decimators (REAL variant): the chain's audio stage Lowpass(128) * de-emphasis(6) -> /5 is
// 133 taps, Q = 27; the plain DecimatorBlock on Float32 (composites/decimator.lua:34-41) with 128 taps is Q = 26.
static int shape_q_real(int M, int D) {
    if (D == 5 && M > 130 && M <= 135) return 27;
    return 0;
}

PolyTaps* polyphase_prepare(const float* taps, int M, int D, double turns_per_sample, bool phasor_table, bool real_data) {
    int Q = real_data ? shape_q_real(M, D) : shape_q(M, D, phasor_table);
    if (!Q) return nullptr;
    PolyTaps* p = new (std::nothrow) PolyTaps();
    if (!p) return nullptr;
    p->M = M; p->D = D; p->Q = Q;
    p->real_data = real_data;
    // hr[i'] multiplies X[c - (Q*D-1) + i']  =>  hr[i'] = h[Q*D-1-i'] (zero for tap index >= M)
    for (int i = 0; i < PT_MAXTAPS; ++i) {
        int k = Q * D - 1 - i;
        p->hr[i] = (i < Q * D && k < M) ? taps[k] : 0.0f;
    }
    p->turns_fix = turns_to_fix(turns_per_sample);
    p->rotates = phasor_table;
    {
        // step[it] = exp(j 2 pi turns * 2*PT_THREADS*it) from the SAME fixed-point turns the kernel uses
        const double two_pi = 6.283185307179586476925286766559;
        const long double tq = ldexpl((long double)p->turns_fix, -64);
        for (int it = 0; it < PT_MAXIT; ++it) {
            long double a = tq * (long double)(2 * PT_THREADS) * (long double)it;
            a -= floorl(a);
            p->step[it] = make_float2((float)std::cos(two_pi * (double)a), (float)std::sin(two_pi * (double)a));
        }
    }
    return p;
}

void polyphase_release(PolyTaps* p) { delete p; }

#define LRB_SHAPE_FULL(DD, QQ)                                                                                         \
    if (p->D == DD && p->Q == QQ) {                                                                                    \
        static_assert(PolyShape<DD, QQ>::ITERS <= PT_MAXIT, "step table too short");                                   \
        if (disc) return launch_shape<DD, QQ, true, true>(P, p->hr, x, hist, n, y, first, n_out, prev_in, prev_out, inv_gain, s); \
        return rot ? launch_shape<DD, QQ, true, false>(P, p->hr, x, hist, n, y, first, n_out, nullptr, nullptr, 0.f, s)    \
                   : launch_shape<DD, QQ, false, false>(P, p->hr, x, hist, n, y, first, n_out, nullptr, nullptr, 0.f, s);  \
    }
#define LRB_SHAPE_PLAIN(DD, QQ)                                                                                        \
    if (p->D == DD && p->Q == QQ && !rot && !disc) {                                                                   \
        static_assert(PolyShape<DD, QQ>::ITERS <= PT_MAXIT, "step table too short");                                   \
        return launch_shape<DD, QQ, false, false>(P, p->hr, x, hist, n, y, first, n_out, nullptr, nullptr, 0.f, s); \
    }

static int launch_polyphase_any(const PolyTaps* p, const float2* x, const float2* hist, long long n, void* y,
                                long long first, long long n_out, bool rotate, bool disc, uint64_t g0,
                                const float2* prev_in, float2* prev_out, float inv_gain, cudaStream_t s) {
    if (!p) return 0;
    if (n_out <= 0) return 1;
    const bool rot = rotate && p->rotates;
    if (disc && !rot) {
        // the fused discriminator is instantiated together with the translator; a zero offset gets the all-ones table
        set_error("tuner: discriminator fusion needs the translator path");
        return -1;
    }
    PolyParams P;
    std::memset(&P, 0, sizeof(P));
    P.turns_fix = p->turns_fix;
    std::memcpy(P.step, p->step, sizeof(P.step));
    P.g0 = g0;
    P.M = p->M;
    if (p->real_data) {
        if (rot || disc) { set_error("polyphase: the real-stream kernel has no translator / discriminator"); return -1; }
        const bool pole = prev_in != nullptr;
        if (pole) {
            // inv_gain carries the pole c; prev_in / prev_out its carried state (float32)
            const double c = (double)inv_gain;
            P.pole_c = inv_gain;
            double pw = std::pow(c, (double)PT_R);
            for (int k = 0; k < 6; ++k) { P.pole_cp[k] = (float)pw; pw = pw * pw; }
        }
        if (p->D == 5 && p->Q == 27)
            return pole ? launch_shape<5, 27, false, false, true, true>(P, p->hr, x, hist, n, y, first, n_out, prev_in, prev_out, 0.f, s)
                        : launch_shape<5, 27, false, false, true, false>(P, p->hr, x, hist, n, y, first, n_out, nullptr, nullptr, 0.f, s);
        return 0;
    }
    LRB_SHAPE_PLAIN(1, 16) LRB_SHAPE_PLAIN(1, 32)
    LRB_SHAPE_FULL(5, 26)
    return 0;
}

bool polyphase_pole_ok(float c) { return std::pow(std::fabs((double)c), (double)PT_POLE_WARM) <= 1e-8; }

int launch_polyphase_rrrf(const PolyTaps* p, const float* x, const float* hist, long long n, float* y,
                          long long first, long long n_out, cudaStream_t s, float pole_c, const float* z_in, float* z_out) {
    return launch_polyphase_any(p, (const float2*)x, (const float2*)hist, n, y, first, n_out, false, false, 0,
                                (const float2*)z_in, (float2*)z_out, pole_c, s);
}

int launch_polyphase_crcf(const PolyTaps* p, const float2* x, const float2* hist, long long n, float2* y,
                          long long first, long long n_out, bool rotate, uint64_t turns_fix, uint64_t g0,
                          cudaStream_t s) {
    (void)turns_fix;
    return launch_polyphase_any(p, x, hist, n, y, first, n_out, rotate, false, g0, nullptr, nullptr, 0.f, s);
}

// ---------------------------------------------------------------------------------------------
// TunerBlock: Rotator -> FIR(crcf) -> Downsampler as one stage of the graph
// ---------------------------------------------------------------------------------------------
struct TunerBlock : DecimatingBlock {
    int M;
    double turns;
    std::vector<float> h_taps;
    PolyTaps* pt = nullptr;
    Carried hist;
    Carried prev;                              // fused discriminator: previous tuner output
    bool disc = false;
    float gain = 1.f;
    std::string label;

    TunerBlock(double turns_per_sample, const float* taps, int ntaps, int decim, float disc_gain)
        : M(ntaps), turns(turns_per_sample), h_taps(taps, taps + ntaps) {
        D = decim;
        disc = disc_gain != 0.0f;
        gain = disc_gain;
        in_size = 8;
        out_size = disc ? 4 : 8;
        dev_ptrs = true;
        label = std::string(disc ? "tuner+discrim(" : "tuner(") + std::to_string(M) + ",/" + std::to_string(D) + ")";
        name = label.c_str();
    }
    ~TunerBlock() override { polyphase_release(pt); }
    int init() override {
        pt = polyphase_prepare(h_taps.data(), M, D, turns, true);
        if (!pt) return -1;      // unsupported shape: the graph keeps the blocks separate
        if (carry(hist, (size_t)(M > 1 ? M - 1 : 1) * 8) != 0) return -1;
        return carry(prev, 8);
    }
    long long memory_in() const override { return M - 1 + (disc ? D : 0); }
    bool supports_lead_wait() const override { return true; }
    bool state_only_on_side_stream() const override { return true; }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override {
        const auto [first, no] = plan(n);
        *n_out = (size_t)no;
        if (n == 0) return 0;
        // the history for the next call depends only on x and the old history: update it on the side stream,
        // concurrently with the filter kernels
        cudaStream_t side = s;
        if (M > 1) {
            if (n >= SIDE_STREAM_MIN) side = side_fork(s);
            if (launch_hist_update(dx, (long long)n, hist.in(), hist.out(), M - 1, 8, side) != 0) return -1;
        }
        int rc = launch_polyphase_any(pt, (const float2*)dx, (const float2*)hist.in(), (long long)n, dy, first, no, true,
                                      disc, consumed, (const float2*)prev.in(), (float2*)prev.out(),
                                      disc ? 1.0f / gain : 0.f, s);
        side_join(s, side);
        if (rc <= 0) { if (rc == 0) set_error("tuner: unsupported shape"); return -1; }
        if (disc && no > 0) prev.flip();
        if (M > 1) hist.flip();
        consumed += n;
        return 0;
    }
};

Block* make_tuner(double turns_per_sample, const float* taps, int ntaps, int decim, float disc_gain) {
    return make_block<TunerBlock>(turns_per_sample, taps, ntaps, decim, disc_gain);
}

}  // namespace lrb
