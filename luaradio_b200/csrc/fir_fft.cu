// Fused overlap-save FIR: load -> 1024-point FFT -> x tap spectrum -> inverse FFT -> store, one kernel,
// the spectrum never leaves the SM.
//
// Reference algorithm: FIRFilterBlock:process_fft (radio/blocks/signal/firfilter.lua:320-398) with
// spectrum_utils.DFT/IDFT (radio/utilities/spectrum_utils.lua:86-113,317-349): N = 2^floor(log2(8M)),
// L = N-M+1, per block two FFTW executes + a VOLK multiply + a 1/N scaling loop + three ffi.copy, i.e. five
// passes over memory.  For M = 128 the reference picks N = 1024, L = 897; this kernel uses N = 1024 for
// every M it accepts (L = 1025 - M).  Unlike process_fft the block stays length-preserving (SURVEY.md 7f):
// the M-1 sample overlap is re-read from the input (or the carried history), never delayed.
//
// Why FFT at all on a GPU (DESIGN.md): direct form costs M packed FFMA2 per complex sample, 128 at M = 128,
// which caps the kernel at ~35 % of the HBM roofline on the FP32 pipe; overlap-save costs ~34 per sample.
//
// Mapping.  One WARP owns one 1024-point block: N = 32 x 32, every lane holds 32 complex points in 32 packed
// f32x2 registers and runs a fully unrolled radix-2 DIT network on them (tools/gen_fft32.py); the only data
// exchange is one 32x32 transpose through a warp-private padded shared-memory tile per transform, so there is
// no CTA-wide barrier in the block loop at all (only __syncwarp).  With n = 32*n1 + n2 and k = k1 + 32*k2:
//   forward:  lane = n2: DFT32 over n1 -> * W1024^(n2*k1) -> transpose -> lane = k1: DFT32 over n2  => X[k1+32k2]
//   multiply: X[k] * H[k]/N      (H in shared memory in [k2][k1] order: conflict-free)
//   inverse:  lane = k1: IDFT32 over k2 -> * conj W1024^(k1*n2) -> transpose -> lane = n2: IDFT32 over k1 => y[n2+32n1]
// so global loads and stores are both lane-contiguous (256 B per warp instruction).
#include "common.cuh"
#include "blocks.h"
#include "fft32_gen.cuh"
#include "../../include/lrb200.h"

#include <algorithm>
#include <cmath>
#include <complex>
#include <new>
#include <vector>

namespace lrb {

namespace {

constexpr int FF_N = 1024;
constexpr int FF_WARPS = 8;                       // warps (= concurrent FFT blocks) per CTA
constexpr int FF_THREADS = FF_WARPS * 32;
constexpr int FF_XSTRIDE = 33;                    // padded row stride of the transpose tile (float2 units)
constexpr int FF_XCH = 32 * FF_XSTRIDE;           // float2 per warp-private tile

__device__ __forceinline__ float2 cmul_conj_if(float2 a, float2 w, bool conj) {
    // a * w  or  a * conj(w)
    const float wi = conj ? -w.y : w.y;
    float2 t = __fmul2_rn(make_float2(-a.y, a.x), make_float2(wi, wi));
    return __ffma2_rn(a, make_float2(w.x, w.x), t);
}

struct FftArgs {
    const void* x;
    const void* hist;
    void* y;
    const float2* H;          // [k2][k1] tap spectrum / N
    const float2* tw;         // [a][b] W1024^(a*b)
    const float2* E;          // [r][lane] exp(j*2*pi*turns*(32 r + lane))  (ROT only)
    long long n;
    long long b_lo, b_hi, nwork;
    long long first;          // decimation: keep outputs at input index first + j*D
    uint64_t turns_fix, g0;   // fused translator
    int M, D;
};

// floor division helpers for (possibly negative) t and positive d
__device__ __forceinline__ void floor_divmod(long long t, int d, long long* q, int* r) {
    long long qq = t / d;
    long long rr = t - qq * d;
    if (rr < 0) { rr += d; qq -= 1; }
    *q = qq;
    *r = (int)rr;
}

// IN   0: complex in / complex out (crcf, cccf)         1: real in, two blocks packed per FFT / real out (rrrf)
//      2: real in / complex out with complex taps (Hilbert: taps = delay + j*hilbert)
// EDGE false: interior blocks [b_lo, b_hi): all N inputs inside x, unconditional coalesced loads (one code path:
//             guarded loads made the compiler clone the butterfly networks behind each branch);
//      true : blocks touching the carried history (b = 0) or the end of the input (b >= b_hi), bounds-checked;
//             work index e < b_lo -> block e, else block b_hi + (e - b_lo).
// ROT  (IN 0): fused FrequencyTranslator: x[i] * exp(j w (g0+i)) = P_b * (x[i] * E[i - base]); E is applied at the
//             load, the per-block phasor P_b commutes with the (linear) filter and is applied to kept outputs only.
// DEC  fused Downsampler: only outputs at input index first + j*D are stored, at y[j].
template <int IN, bool EDGE, bool ROT, bool DEC>
__global__ void __launch_bounds__(FF_THREADS, 2)
fir_fft1024_kernel(const __grid_constant__ FftArgs A) {
    extern __shared__ __align__(16) float2 sm[];
    float2* s_tw = sm;                            // [k1][n2]  W1024^(k1*n2)
    float2* s_H = sm + FF_N;                      // [k2][k1]  H[k1 + 32 k2] / N
    float2* s_E = sm + 2 * FF_N;                  // [r][lane] (ROT)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float2* xch = sm + (ROT ? 3 : 2) * FF_N + warp * FF_XCH;
    for (int i = tid; i < FF_N; i += FF_THREADS) {
        s_tw[i] = A.tw[i];
        s_H[i] = A.H[i];
        if constexpr (ROT) s_E[i] = A.E[i];
    }
    __syncthreads();

    const int M = A.M;
    const long long n = A.n;
    const int L = FF_N - (M - 1);
    const int Hm1 = M - 1;
    const int D = A.D;
    const int s32 = DEC ? 32 % D : 0, q32 = DEC ? 32 / D : 0;
    const long long wstride = (long long)gridDim.x * FF_WARPS;
    for (long long wi = (long long)blockIdx.x * FF_WARPS + warp; wi < A.nwork; wi += wstride) {
        const long long b = EDGE ? (wi < A.b_lo ? wi : A.b_hi + (wi - A.b_lo)) : (A.b_lo + wi);
        float2 v[32];
        // ---- load: v[r] = X[base + 32 r + lane]
        if constexpr (IN == 0) {
            const float2* x = reinterpret_cast<const float2*>(A.x);
            const float2* hist = reinterpret_cast<const float2*>(A.hist);
            const long long base = b * L - Hm1;
            if constexpr (!EDGE) {
                const float2* xb = x + base + lane;
#pragma unroll
                for (int r = 0; r < 32; ++r) v[r] = __ldcs(xb + 32 * r);
            } else {
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    const long long i = base + 32 * r + lane;
                    v[r] = (i >= 0) ? (i < n ? __ldg(x + i) : make_float2(0.f, 0.f))
                                    : ((Hm1 + i >= 0) ? __ldg(hist + (Hm1 + i)) : make_float2(0.f, 0.f));
                }
            }
            if constexpr (ROT) {
#pragma unroll
                for (int r = 0; r < 32; ++r) v[r] = cmul_conj_if(v[r], s_E[r * 32 + lane], false);
            }
        } else if constexpr (IN == 1) {
            // two consecutive real blocks 2b, 2b+1 as real / imaginary part
            const float* x = reinterpret_cast<const float*>(A.x);
            const float* hist = reinterpret_cast<const float*>(A.hist);
            const long long base0 = (2 * b) * L - Hm1, base1 = base0 + L;
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const long long i0 = base0 + 32 * r + lane, i1 = base1 + 32 * r + lane;
                if constexpr (!EDGE) {
                    v[r] = make_float2(__ldcs(x + i0), __ldcs(x + i1));
                } else {
                    const float a = (i0 >= 0) ? (i0 < n ? __ldg(x + i0) : 0.f) : __ldg(hist + (Hm1 + i0));
                    const float c = (i1 >= 0) ? (i1 < n ? __ldg(x + i1) : 0.f) : ((Hm1 + i1 >= 0) ? __ldg(hist + (Hm1 + i1)) : 0.f);
                    v[r] = make_float2(a, c);
                }
            }
        } else {
            const float* x = reinterpret_cast<const float*>(A.x);
            const float* hist = reinterpret_cast<const float*>(A.hist);
            const long long base = b * L - Hm1;
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const long long i = base + 32 * r + lane;
                float a;
                if constexpr (!EDGE) a = __ldcs(x + i);
                else a = (i >= 0) ? (i < n ? __ldg(x + i) : 0.f) : __ldg(hist + (Hm1 + i));
                v[r] = make_float2(a, 0.f);
            }
        }

        // ---- forward pass 1: lane = n2, registers n1 -> k1 (result for k1 in v[bitrev5(k1)])
        fft32_nat2br<false>(v);
        __syncwarp();                               // previous iteration's tile reads are done
#pragma unroll
        for (int k1 = 0; k1 < 32; ++k1) {
            float2 t = v[bitrev5(k1)];
            if (k1 > 0) t = cmul_conj_if(t, s_tw[k1 * 32 + lane], false);
            xch[k1 * FF_XSTRIDE + lane] = t;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 32; ++r) v[r] = xch[lane * FF_XSTRIDE + r];      // lane = k1, r = n2
        // ---- forward pass 2: registers n2 -> k2 (X[k1 + 32 k2] in v[bitrev5(k2)])
        fft32_nat2br<false>(v);
        // ---- multiply by the tap spectrum (1/N folded in)
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2) v[bitrev5(k2)] = cmul_conj_if(v[bitrev5(k2)], s_H[k2 * 32 + lane], false);
        // ---- inverse pass 1: lane = k1, registers k2 (bit-reversed placement) -> n2 (natural)
        fft32_br2nat<true>(v);
        __syncwarp();                               // tile reads of the forward transpose are done
#pragma unroll
        for (int n2 = 0; n2 < 32; ++n2) {
            float2 t = v[n2];
            if (n2 > 0) t = cmul_conj_if(t, s_tw[n2 * 32 + lane], true);
            xch[n2 * FF_XSTRIDE + lane] = t;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 32; ++r) v[r] = xch[lane * FF_XSTRIDE + r];      // lane = n2, r = k1
        // ---- inverse pass 2: registers k1 -> n1 (y[n2 + 32 n1] in v[bitrev5(n1)])
        fft32_nat2br<true>(v);

        // ---- store the L valid outputs: block index nn = 32 n1 + lane >= M-1  ->  input-aligned index o = obase + nn
        if constexpr (IN == 0 || IN == 2) {
            float2* y = reinterpret_cast<float2*>(A.y);
            const long long obase = b * L - Hm1;
            if constexpr (!DEC) {
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) {
                    const int nn = 32 * n1 + lane;
                    const long long o = obase + nn;
                    if (nn >= Hm1 && (!EDGE || o < n)) {
                        __stcs(y + o, v[bitrev5(n1)]);
                    }
                }
            } else {
                float2 Pb = make_float2(1.f, 0.f);
                if constexpr (ROT) Pb = phasor_from_fix(A.turns_fix * (A.g0 + (uint64_t)obase));
                long long q;
                int r;
                floor_divmod(obase + lane - A.first, D, &q, &r);
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) {
                    const int nn = 32 * n1 + lane;
                    if (r == 0 && q >= 0 && nn >= Hm1 && (!EDGE || obase + nn < n)) {
                        float2 t = v[bitrev5(n1)];
                        if constexpr (ROT) t = cmul_conj_if(t, Pb, false);
                        y[q] = t;
                    }
                    r += s32;
                    q += q32;
                    if (r >= D) { r -= D; ++q; }
                }
            }
        } else {
            float* y = reinterpret_cast<float*>(A.y);
            const long long obase0 = (2 * b) * L - Hm1, obase1 = obase0 + L;
            if constexpr (!DEC) {
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) {
                    const int nn = 32 * n1 + lane;
                    if (nn >= Hm1) {
                        const float2 t = v[bitrev5(n1)];
                        if (!EDGE || obase0 + nn < n) y[obase0 + nn] = t.x;
                        if (!EDGE || obase1 + nn < n) y[obase1 + nn] = t.y;
                    }
                }
            } else {
                long long q0, q1;
                int r0, r1;
                floor_divmod(obase0 + lane - A.first, D, &q0, &r0);
                floor_divmod(obase1 + lane - A.first, D, &q1, &r1);
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) {
                    const int nn = 32 * n1 + lane;
                    const float2 t = v[bitrev5(n1)];
                    if (nn >= Hm1) {
                        if (r0 == 0 && q0 >= 0 && (!EDGE || obase0 + nn < n)) y[q0] = t.x;
                        if (r1 == 0 && q1 >= 0 && (!EDGE || obase1 + nn < n)) y[q1] = t.y;
                    }
                    r0 += s32; q0 += q32; if (r0 >= D) { r0 -= D; ++q0; }
                    r1 += s32; q1 += q32; if (r1 >= D) { r1 -= D; ++q1; }
                }
            }
        }
    }
}

template <int IN, bool ROT, bool DEC>
int launch_fft(const FftArgs& base_args, long long n_int, long long n_edge, cudaStream_t s) {
    static bool configured_dev[LRB_MAX_DEVICES] = {false};     // function attributes are per device
    bool& configured = configured_dev[ctx().device & (LRB_MAX_DEVICES - 1)];
    constexpr size_t smem = (size_t)((ROT ? 3 : 2) * FF_N + FF_WARPS * FF_XCH) * sizeof(float2);
    auto ki = fir_fft1024_kernel<IN, false, ROT, DEC>;
    auto ke = fir_fft1024_kernel<IN, true, ROT, DEC>;
    if (!configured) {
        LRB_CHECK(cudaFuncSetAttribute(ki, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        LRB_CHECK(cudaFuncSetAttribute(ke, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    const long long max_ctas = (long long)ctx().sm_count * 2;
    // edge blocks on the side stream (they only overlap the interior kernel and touch disjoint outputs)
    cudaStream_t side = (n_int > 0 && n_edge > 0) ? side_fork(s) : s;
    if (n_edge > 0) {
        FftArgs a = base_args;
        a.nwork = n_edge;
        long long ctas = (n_edge + FF_WARPS - 1) / FF_WARPS;
        ke<<<(unsigned)ctas, FF_THREADS, smem, side>>>(a);
        count_launch();
    }
    if (n_int > 0) {
        FftArgs a = base_args;
        a.nwork = n_int;
        long long ctas = (n_int + FF_WARPS - 1) / FF_WARPS;
        if (ctas > max_ctas) ctas = max_ctas;
        ki<<<(unsigned)ctas, FF_THREADS, smem, s>>>(a);
        count_launch();
    }
    side_join(s, side);
    LRB_CHECK(cudaGetLastError());
    return 1;
}

// ---------------------------------------------------------------------------------------------
// Long filters (513 < M <= 8192): uniformly partitioned overlap-save with a frequency-domain delay line.
// The taps are cut into P partitions of 512; with hop 512 and N = 1024 every input block is transformed ONCE,
//     Y_b = sum_p X_{b-p} * H_p,      y[512 b + j] = IFFT(Y_b)[512 + j],  j < 512,
// so a block costs one forward FFT, P spectrum multiply-accumulates and one inverse FFT (the old scheme ran P full
// passes over memory: P forward + P inverse transforms and P-1 read-modify-writes of y).  A CTA owns a contiguous
// run of blocks; its FD_W warps transform FD_W consecutive blocks, park the spectra in a shared-memory ring of
// FD_W + P - 1 slots (register layout [k2][lane], so no transposition and no bank conflicts), and after one CTA
// barrier each warp accumulates the spectra of its own and the P-1 previous blocks.  The ring slots double as the
// 32x32 transposition tiles of both transforms (a slot is dead between its block leaving the delay line and the next
// block landing in it), so a CTA needs 8 + 8.25 (FD_W + P - 1) KB and two CTAs fit per SM.  The run starts with one
// group that only fills the ring (P-1 redundant transforms per ~1800 blocks).  P <= 4 per launch (ring = 91 KB);
// longer filters run ceil(P/4) launches, the later ones accumulating into y.
// ---------------------------------------------------------------------------------------------
constexpr int FD_W = 8;
constexpr int FD_MAXPC = 4;
constexpr int FD_HOP = 512;

struct FdlArgs {
    const float2* x;
    const float2* hist;
    float2* y;
    const float2* H;          // pc tap spectra [p][k2][k1], already scaled by 1/N
    const float2* tw;
    long long n;
    long long b_lo, b_hi, nblocks, chunk;
    int pc;                   // partitions handled by this launch
    int hist_len;
    int in_shift;             // 512 * index of the first partition of this launch
    int accumulate;
};

template <bool EDGE, int PC>
__global__ void __launch_bounds__(FD_W * 32, 2)
fir_fft_fdl_kernel(const __grid_constant__ FdlArgs A) {
    extern __shared__ __align__(16) float2 sm[];
    float2* s_tw = sm;
    float2* ring = sm + FF_N;                              // R slots of FF_XCH float2 (padded 32x33 tile / [k2][lane] spectrum)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < FF_N; i += FD_W * 32) s_tw[i] = A.tw[i];
    constexpr int R = FD_W + PC - 1;                        // compile-time: slot arithmetic folds to constants
    long long r0, r1;
    if constexpr (EDGE) {
        if (blockIdx.x == 0) { r0 = 0; r1 = A.b_lo; } else { r0 = A.b_hi; r1 = A.nblocks; }
    } else {
        r0 = A.b_lo + (long long)blockIdx.x * A.chunk;
        r1 = r0 + A.chunk < A.b_hi ? r0 + A.chunk : A.b_hi;
    }
    if (r0 >= r1) return;
    const long long rbase = r0 - (PC - 1);
    const long long n = A.n;
    const int nrel = (int)(r1 - rbase);                     // blocks of this run, relative to rbase: [0, PC-1) only fill the ring
    const float2* xrun = A.x + ((rbase - 1) * FD_HOP - A.in_shift) + lane;      // interior: never dereferenced out of range
    float2* yrun = A.y + rbase * FD_HOP + lane;
    __syncthreads();
    // slot of block rel: rel mod R.  The slot a warp transposes through in the forward pass is the one its
    // spectrum then lives in; for the inverse pass it borrows the slot of block rel + FD_W (== block rel - PC + 1, dead
    // once every warp has finished its multiply-accumulate), which is also the slot it owns in the next group.
    for (int g = PC - 1 - FD_W; g < nrel; g += FD_W) {
        const int rel = g + warp;
        const bool fwd = rel >= 0 && rel < nrel;            // warp-uniform
        const bool emit = rel >= PC - 1 && rel < nrel;
        float2 v[32];
        if (fwd) {
            float2* xch = ring + (rel % R) * FF_XCH;
            if constexpr (!EDGE) {
                const float2* xb = xrun + (long long)rel * FD_HOP;
#pragma unroll
                for (int r = 0; r < 32; ++r) v[r] = __ldcs(xb + 32 * r);
            } else {
                const int HL = A.hist_len;
                const long long base = (rbase + rel - 1) * FD_HOP - A.in_shift;
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    const long long i = base + 32 * r + lane;
                    v[r] = (i >= 0) ? (i < n ? __ldg(A.x + i) : make_float2(0.f, 0.f))
                                    : ((HL + i >= 0) ? __ldg(A.hist + (HL + i)) : make_float2(0.f, 0.f));
                }
            }
            fft32_nat2br<false>(v);
#pragma unroll
            for (int k1 = 0; k1 < 32; ++k1) {
                float2 t = v[bitrev5(k1)];
                if (k1 > 0) t = cmul_conj_if(t, s_tw[k1 * 32 + lane], false);
                xch[k1 * FF_XSTRIDE + lane] = t;
            }
            __syncwarp();
#pragma unroll
            for (int r = 0; r < 32; ++r) v[r] = xch[lane * FF_XSTRIDE + r];
            fft32_nat2br<false>(v);                        // X[lane + 32 k2] in v[bitrev5(k2)]
            __syncwarp();                                  // tile reads done before the spectrum overwrites it
            float4* sp = reinterpret_cast<float4*>(xch) + lane;           // [k2/2][lane] pairs: 128-bit, conflict-free
#pragma unroll
            for (int k2 = 0; k2 < 32; k2 += 2)
                sp[(k2 / 2) * 32] = make_float4(v[bitrev5(k2)].x, v[bitrev5(k2)].y, v[bitrev5(k2 + 1)].x, v[bitrev5(k2 + 1)].y);
        }
        __syncthreads();                                   // the spectra of this group are in the ring
        if (g >= PC - 1) {
            // Multiply-accumulate, split by FREQUENCY: warp w owns bins k2 = 4w .. 4w+3 (two 128-bit rows of every slot)
            // for all FD_W blocks of the group, so a tap-spectrum value is loaded once per group instead of once per
            // block, and each delay-line value once instead of PC times.  Y_j lands in the slot of block j - (PC-1),
            // which leaves the delay line after this group; only this warp touches these rows in this phase.
            if constexpr (!EDGE) {
                // pull the next group's input block towards L2 while this group multiplies and inverts
                if (rel + FD_W < nrel) {
                    const char* nx = reinterpret_cast<const char*>(xrun - lane + (long long)(rel + FD_W) * FD_HOP) + lane * 256;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + 128));
                }
            }
            // slot offsets (float4 units) of blocks g-3 .. g+7 and of the FD_W output slots, shared by both row halves.
            // Blocks of this group beyond the end of the run hold stale spectra; their Y lands in slots nobody reads.
            int xoff[FD_W + FD_MAXPC - 1], yoff[FD_W];
            {
                int sl = (g - (FD_MAXPC - 1) + R * 4) % R;
#pragma unroll
                for (int i = 0; i < FD_W + FD_MAXPC - 1; ++i) { xoff[i] = sl * (FF_XCH / 2); sl = sl + 1 == R ? 0 : sl + 1; }
                int so = (g + FD_W) % R;
#pragma unroll
                for (int j = 0; j < FD_W; ++j) { yoff[j] = so * (FF_XCH / 2); so = so + 1 == R ? 0 : so + 1; }
            }
            const float4* ring4 = reinterpret_cast<const float4*>(ring);
            float4* ring4w = reinterpret_cast<float4*>(ring);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int row = (2 * warp + half) * 32 + lane;
                float4 Hr[PC];
#pragma unroll
                for (int pp = 0; pp < PC; ++pp) Hr[pp] = __ldg(reinterpret_cast<const float4*>(A.H) + pp * (FF_N / 2) + row);
                float4 Xr[FD_W + FD_MAXPC - 1];
#pragma unroll
                for (int i = FD_MAXPC - PC; i < FD_W + FD_MAXPC - 1; ++i) Xr[i] = ring4[xoff[i] + row];
#pragma unroll
                for (int j = 0; j < FD_W; ++j) {
                    float4 a = Xr[j + FD_MAXPC - 1];
                    float2 t0 = __fmul2_rn(make_float2(-a.y, a.x), make_float2(Hr[0].y, Hr[0].y));
                    float2 ye = __ffma2_rn(make_float2(a.x, a.y), make_float2(Hr[0].x, Hr[0].x), t0);
                    float2 t1 = __fmul2_rn(make_float2(-a.w, a.z), make_float2(Hr[0].w, Hr[0].w));
                    float2 yo = __ffma2_rn(make_float2(a.z, a.w), make_float2(Hr[0].z, Hr[0].z), t1);
#pragma unroll
                    for (int pp = 1; pp < PC; ++pp) {
                        a = Xr[j + FD_MAXPC - 1 - pp];
                        ye = __ffma2_rn(make_float2(a.x, a.y), make_float2(Hr[pp].x, Hr[pp].x), ye);
                        ye = __ffma2_rn(make_float2(-a.y, a.x), make_float2(Hr[pp].y, Hr[pp].y), ye);
                        yo = __ffma2_rn(make_float2(a.z, a.w), make_float2(Hr[pp].z, Hr[pp].z), yo);
                        yo = __ffma2_rn(make_float2(-a.w, a.z), make_float2(Hr[pp].w, Hr[pp].w), yo);
                    }
                    ring4w[yoff[j] + row] = make_float4(ye.x, ye.y, yo.x, yo.y);
                }
            }
        }
        __syncthreads();                                   // every Y_b is in the slot its owner transposes through next
        if (emit) {
            float2* xch = ring + ((rel + FD_W) % R) * FF_XCH;
            {
                const float4* yp = reinterpret_cast<const float4*>(xch) + lane;
#pragma unroll
                for (int k2 = 0; k2 < 32; k2 += 2) {
                    const float4 t = yp[(k2 / 2) * 32];
                    v[bitrev5(k2)] = make_float2(t.x, t.y);
                    v[bitrev5(k2 + 1)] = make_float2(t.z, t.w);
                }
            }
            __syncwarp();                                  // Y is in registers before the slot becomes the transposition tile
            fft32_br2nat<true>(v);
#pragma unroll
            for (int n2 = 0; n2 < 32; ++n2) {
                float2 t = v[n2];
                if (n2 > 0) t = cmul_conj_if(t, s_tw[n2 * 32 + lane], true);
                xch[n2 * FF_XSTRIDE + lane] = t;
            }
            __syncwarp();
#pragma unroll
            for (int r = 0; r < 32; ++r) v[r] = xch[lane * FF_XSTRIDE + r];
            __syncwarp();
            fft32_nat2br<true>(v);                         // y-block sample lane + 32 n1 in v[bitrev5(n1)]
            float2* yb = yrun + (long long)rel * FD_HOP;
            const long long o0 = (rbase + rel) * FD_HOP + lane;
#pragma unroll
            for (int n1 = 16; n1 < 32; ++n1) {
                if (!EDGE || o0 + 32 * (n1 - 16) < n) {
                    float2 t = v[bitrev5(n1)];
                    if (A.accumulate) t = __fadd2_rn(t, yb[32 * (n1 - 16)]);
                    __stcs(yb + 32 * (n1 - 16), t);
                }
            }
        }
    }
}

template <int PC>
int launch_fdl_pc(FdlArgs a, cudaStream_t s) {
    static bool configured_dev[LRB_MAX_DEVICES] = {false};     // function attributes are per device
    bool& configured = configured_dev[ctx().device & (LRB_MAX_DEVICES - 1)];
    constexpr size_t smem = (size_t)(FF_N + (FD_W + PC - 1) * FF_XCH) * sizeof(float2);
    auto ki = fir_fft_fdl_kernel<false, PC>;
    auto ke = fir_fft_fdl_kernel<true, PC>;
    if (!configured) {
        LRB_CHECK(cudaFuncSetAttribute(ki, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        LRB_CHECK(cudaFuncSetAttribute(ke, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    const long long n_int = a.b_hi - a.b_lo;
    const bool edges = a.b_lo > 0 || a.nblocks > a.b_hi;
    cudaStream_t side = (n_int > 0 && edges) ? side_fork(s) : s;
    if (edges) {
        ke<<<2, FD_W * 32, smem, side>>>(a);
        count_launch();
    }
    if (n_int > 0) {
        long long ctas = (n_int + FD_W - 1) / FD_W;
        if (ctas > 2LL * ctx().sm_count) ctas = 2LL * ctx().sm_count;
        long long chunk = (n_int + ctas - 1) / ctas;
        chunk = (chunk + FD_W - 1) / FD_W * FD_W;
        ctas = (n_int + chunk - 1) / chunk;
        a.chunk = chunk;
        ki<<<(unsigned)ctas, FD_W * 32, smem, s>>>(a);
        count_launch();
    }
    side_join(s, side);
    LRB_CHECK(cudaGetLastError());
    return 1;
}

int launch_fdl(const FdlArgs& a, cudaStream_t s) {
    switch (a.pc) {
        case 1: return launch_fdl_pc<1>(a, s);
        case 2: return launch_fdl_pc<2>(a, s);
        case 3: return launch_fdl_pc<3>(a, s);
        default: return launch_fdl_pc<4>(a, s);
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Host-side plan: tap spectrum (float64 DFT of the zero-extended taps, scaled by 1/N, as
// firfilter.lua:337-343 does with spectrum_utils.DFT) and the 32x32 inter-pass twiddle table.
// ---------------------------------------------------------------------------------------------
struct FirFast {
    int nparts = 1;            // > 1: uniformly partitioned overlap-save for filters longer than one block allows
    int part_taps = 0;
    float2* d_H = nullptr;     // nparts tap spectra, FF_N each
    float2* d_tw = nullptr;
    float2* d_E = nullptr;
    int in_mode = 0;
};

static constexpr int FFT_MAX_TAPS = 513;       // L >= 512: at most half of every block is overlap

int FirBlock::fast_init() {
    // register-tiled direct kernel: decimators with <= 128 taps and plain FIRs with <= 32 taps (complex in, real taps)
    if (kind == FIR_CRCF && !rotate) poly = polyphase_prepare((const float*)h_taps.data(), M, D, 0.0);
    if (kind == FIR_RRRF && D > 1) poly = polyphase_prepare((const float*)h_taps.data(), M, D, 0.0, false, true);
    gen_poly = !rotate && D >= 2 && poly_generic_supports(kind, M, D);
    if (kind == FIR_HILBERT && D != 1) return 0;
    const bool long_filter = M > FFT_MAX_TAPS;
    // long filters: complex-input, no fused decimation/translator -> P partitions of 512 taps, P passes over x
    if (long_filter && !((kind == FIR_CRCF || kind == FIR_CCCF) && D == 1 && !rotate && M <= 16 * 512)) return 0;
    fast = new (std::nothrow) FirFast();
    if (!fast) { set_error("out of memory"); return -1; }
    fast->in_mode = (kind == FIR_RRRF) ? 1 : (kind == FIR_HILBERT ? 2 : 0);
    fast->part_taps = long_filter ? 512 : M;
    fast->nparts = long_filter ? (M + 511) / 512 : 1;
    const double two_pi = 6.283185307179586476925286766559;
    std::vector<std::complex<double>> h(M);
    const float* tf = (const float*)h_taps.data();
    for (int k = 0; k < M; ++k) {
        if (kind == FIR_CCCF) h[k] = std::complex<double>(tf[2 * k], tf[2 * k + 1]);
        else if (kind == FIR_HILBERT) h[k] = std::complex<double>(k == (M - 1) / 2 ? 1.0 : 0.0, tf[k]);   // delay + j*hilbert (hilberttransform.lua:120-124)
        else h[k] = std::complex<double>(tf[k], 0.0);
    }
    std::vector<float2> H((size_t)FF_N * fast->nparts), tw(FF_N), E(FF_N);
    std::vector<std::complex<double>> wtab(FF_N);
    for (int e = 0; e < FF_N; ++e) wtab[e] = std::complex<double>(std::cos(two_pi * e / FF_N), -std::sin(two_pi * e / FF_N));
    for (int part = 0; part < fast->nparts; ++part) {
        const int m0 = part * fast->part_taps;
        const int mc = std::min(fast->part_taps, M - m0);
        for (int k = 0; k < FF_N; ++k) {
            std::complex<double> acc(0.0, 0.0);
            for (int m = 0; m < mc; ++m) acc += h[m0 + m] * wtab[(int)(((long long)k * m) % FF_N)];
            acc /= (double)FF_N;
            const int k1 = k % 32, k2 = k / 32;
            // single block: [k2][k1]; partitioned (delay-line kernel): [k2/2][k1][k2&1] for 128-bit loads
            const size_t at = long_filter ? (size_t)(k2 / 2) * 64 + k1 * 2 + (k2 & 1) : (size_t)k2 * 32 + k1;
            H[(size_t)part * FF_N + at] = make_float2((float)acc.real(), (float)acc.imag());
        }
    }
    for (int a = 0; a < 32; ++a)
        for (int c = 0; c < 32; ++c) {
            const int e = (a * c) % FF_N;
            tw[a * 32 + c] = make_float2((float)std::cos(two_pi * e / FF_N), (float)(-std::sin(two_pi * e / FF_N)));
        }
    LRB_CHECK(cudaMalloc(&fast->d_H, sizeof(float2) * H.size()));
    LRB_CHECK(cudaMalloc(&fast->d_tw, sizeof(float2) * FF_N));
    LRB_CHECK(cudaMemcpy(fast->d_H, H.data(), sizeof(float2) * H.size(), cudaMemcpyHostToDevice));
    LRB_CHECK(cudaMemcpy(fast->d_tw, tw.data(), sizeof(float2) * FF_N, cudaMemcpyHostToDevice));
    if (rotate) {
        // E[n] = exp(j 2 pi turns n) from the same 2^-64 fixed-point turns the kernel uses for the block phasor
        const long double tq = ldexpl((long double)rot_fix, -64);
        for (int i = 0; i < FF_N; ++i) {
            long double a = tq * (long double)i;
            a -= floorl(a);
            E[i] = make_float2((float)std::cos(two_pi * (double)a), (float)std::sin(two_pi * (double)a));
        }
        LRB_CHECK(cudaMalloc(&fast->d_E, sizeof(float2) * FF_N));
        LRB_CHECK(cudaMemcpy(fast->d_E, E.data(), sizeof(float2) * FF_N, cudaMemcpyHostToDevice));
    }
    return 0;
}

void FirBlock::fast_free() {
    polyphase_release(poly);
    poly = nullptr;
    if (fast) {
        cudaFree(fast->d_H);
        cudaFree(fast->d_tw);
        cudaFree(fast->d_E);
        delete fast;
        fast = nullptr;
    }
}

// The algorithm that would run for a long input (what lrb200_fir_get_algorithm reports).
int FirBlock::effective_algorithm() const {
    if (rotate) return LRB200_FIR_FFT;                         // the fused translator exists only in the FFT kernel
    if (!fast || algo == LRB200_FIR_DIRECT) return LRB200_FIR_DIRECT;
    if (algo == LRB200_FIR_FFT) return LRB200_FIR_FFT;
    if (poly) return LRB200_FIR_DIRECT;                        // register-tiled polyphase decimator
    // automatic: overlap-save once the direct form would be FP32-bound.  Packed FFMA2 per INPUT sample:
    //   direct = M/D (crcf), 2M/D (cccf), M/2D (rrrf, hilbert);  overlap-save ~ 31 / (L/N) (half for packed real blocks)
    // Direct kernels for these shapes: the generic polyphase kernel where it covers the shape (measured, profiles/
    // r02_decim_shapes.json: it beats the overlap-save kernel only for short complex-input real-tap filters, e.g. (D, M) =
    // (2, 16), (3, 33); tap loads from the constant bank pace it), else the catch-all (about 8x off), hence the factors.
    const double per_tap = kind == FIR_CCCF ? 2.0 : (kind == FIR_CRCF ? 1.0 : (gen_poly ? 1.0 : 0.5));
    const double direct_cost = (gen_poly ? 3.0 : 8.0) * per_tap * M / D;
    const int mp = fast->part_taps;
    const double fft_cost = fast->nparts * 31.0 * FF_N / (double)(FF_N - mp + 1) * (kind == FIR_RRRF ? 0.5 : 1.0);
    return direct_cost > fft_cost ? LRB200_FIR_FFT : LRB200_FIR_DIRECT;
}

int FirBlock::set_algorithm(int a) {
    if (a < LRB200_FIR_AUTO || a > LRB200_FIR_FFT) { set_error("fir: unknown algorithm %d", a); return -1; }
    algo = a;
    return 0;
}

int FirBlock::fast_run(const void* dx, size_t n, void* dy, long long first, long long n_out, cudaStream_t s) {
    if (poly && algo != LRB200_FIR_FFT && kind == FIR_RRRF)
        return launch_polyphase_rrrf(poly, (const float*)dx, (const float*)hist.in(), (long long)n, (float*)dy, first, n_out, s,
                                     pole_c, has_pole ? (const float*)pole.in() : nullptr, has_pole ? (float*)pole.out() : nullptr);
    if (has_pole) { set_error("fir: the fused output-rate pole needs the real polyphase kernel"); return -1; }
    if (poly && algo != LRB200_FIR_FFT)
        return launch_polyphase_crcf(poly, (const float2*)dx, (const float2*)hist.in(), (long long)n, (float2*)dy,
                                     first, n_out, false, 0, consumed, s);
    const int eff = effective_algorithm();
    if (gen_poly && eff == LRB200_FIR_DIRECT) {
        const int rc = launch_poly_generic(kind, dx, hist.in(), h_taps.data(), M, D, first, (long long)n, n_out, dy, s);
        if (rc != 0) return rc;
    }
    if (!fast || eff != LRB200_FIR_FFT) {
        if (rotate) { set_error("fir: fused translator needs the overlap-save path (ntaps <= %d)", FFT_MAX_TAPS); return -1; }
        return 0;
    }
    const int Mp = fast->part_taps;                      // taps convolved per launch (== M unless partitioned)
    const int L = FF_N - (Mp - 1);
    // a forced FFT (or a fused translator) always runs; the automatic choice leaves short calls to the direct kernel
    if (algo != LRB200_FIR_FFT && !rotate && (long long)n < 8LL * L) return 0;
    // blocks of L outputs; in packed-real mode one FFT covers two of them
    const long long per = (fast->in_mode == 1) ? 2LL * L : (long long)L;
    const long long nblocks = ((long long)n + per - 1) / per;
    if (fast->nparts > 1) {
        // frequency-domain delay line: hop 512, blocks b cover outputs [512 b, 512 b + 512)
        const long long nb = ((long long)n + FD_HOP - 1) / FD_HOP;
        for (int p0 = 0; p0 < fast->nparts; p0 += FD_MAXPC) {
            FdlArgs a;
            a.x = (const float2*)dx; a.hist = (const float2*)hist.in(); a.y = (float2*)dy;
            a.H = fast->d_H + (size_t)p0 * FF_N; a.tw = fast->d_tw; a.n = (long long)n;
            a.pc = std::min(FD_MAXPC, fast->nparts - p0);
            a.nblocks = nb;
            a.b_lo = std::min<long long>(nb, a.pc + p0);          // first block whose ring pre-fill reads x[>= 0]
            a.b_hi = std::max<long long>(a.b_lo, (long long)n / FD_HOP);
            if (a.b_hi > nb) a.b_hi = nb;
            a.chunk = 0; a.hist_len = M - 1; a.in_shift = p0 * FD_HOP; a.accumulate = p0 > 0 ? 1 : 0;
            if (launch_fdl(a, s) < 0) return -1;
        }
        return 1;
    }
    {
        // interior blocks [b_lo, b_hi): b*per - (M-1) >= 0  and  (b+1)*per <= n
        long long b_lo = ((long long)(Mp - 1) + per - 1) / per;
        if (b_lo < 1) b_lo = 1;
        long long b_hi = (long long)n / per;
        if (b_hi > nblocks) b_hi = nblocks;
        if (b_hi < b_lo) b_hi = b_lo;
        if (b_lo > nblocks) { b_lo = nblocks; b_hi = nblocks; }
        FftArgs a;
        a.x = dx; a.hist = hist.in(); a.y = dy; a.H = fast->d_H; a.tw = fast->d_tw; a.E = fast->d_E;
        a.n = (long long)n; a.b_lo = b_lo; a.b_hi = b_hi; a.nwork = 0; a.first = first;
        a.turns_fix = rot_fix; a.g0 = consumed; a.M = Mp; a.D = D;
        // edge work list: blocks [0, b_lo) and [b_hi, nblocks); the kernel maps e -> (e < b_lo ? e : b_hi + e - b_lo)
        const long long n_int = b_hi - b_lo, n_edge = b_lo + (nblocks - b_hi);
        const bool dec = D > 1;
        int rc;
        switch (fast->in_mode) {
            case 0:
                if (rotate) rc = launch_fft<0, true, true>(a, n_int, n_edge, s);   // fused translator always uses the DEC store (D may be 1)
                else rc = dec ? launch_fft<0, false, true>(a, n_int, n_edge, s) : launch_fft<0, false, false>(a, n_int, n_edge, s);
                break;
            case 1:
                rc = dec ? launch_fft<1, false, true>(a, n_int, n_edge, s) : launch_fft<1, false, false>(a, n_int, n_edge, s);
                break;
            default:
                rc = launch_fft<2, false, false>(a, n_int, n_edge, s);
        }
        if (rc < 0) return -1;
    }
    return 1;
}

}  // namespace lrb
