// Resampling family (SURVEY.md 8f row 4): MultiplyConstantBlock, UpsamplerBlock and the fused polyphase
// interpolating / rational-resampling FIR behind InterpolatorBlock and RationalResamplerBlock.
//
// Reference:
//   radio/blocks/signal/multiplyconstant.lua        y[i] = x[i] * c          (complex x complex, complex x real, real x real)
//   radio/blocks/signal/upsampler.lua:44-52         y[i*L] = x[i], zeros in between
//   radio/composites/interpolator.lua:31-41         MultiplyConstant(L) -> Upsampler(L) -> Lowpass(ntaps, 1/L, nyquist 1.0)
//   radio/composites/rationalresampler.lua:33-46    ... -> Downsampler(D), cutoff min(1/L, 1/D)
// The reference filters the zero-stuffed stream with the ordinary dot-product FIR (L-1 of every L products are
// 0 * tap, and D-1 of every D outputs are dropped).  The fused kernel computes only kept outputs from only the
// non-zero products: with u the zero-stuffed stream (u[iL] = c*x[i]) and J = m*D the upsampled index of output m,
//     y[m] = sum_k h[k] u[J-k] = sum_{t >= 0, k = (J mod L) + tL < M} h[k] * (c * x[floor(J/L) - t]),
// i.e. ceil(M/L) multiply-adds per output instead of M*D; the stuffed stream never exists in memory.
// Algorithmic bytes: 8 (in) + 8 L/D (out) per complex input sample.
#include "common.cuh"
#include "blocks.h"

#include <algorithm>
#include <new>
#include <vector>

namespace lrb {

namespace {

template <bool CDATA, bool CCONST>
__global__ void __launch_bounds__(256)
scale_kernel(const void* __restrict__ xv, void* __restrict__ yv, long long n, float cre, float cim) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if constexpr (CDATA) {
            const float2 v = reinterpret_cast<const float2*>(xv)[i];
            float2 o;
            if constexpr (CCONST) o = make_float2(v.x * cre - v.y * cim, v.x * cim + v.y * cre);
            else o = make_float2(v.x * cre, v.y * cre);
            reinterpret_cast<float2*>(yv)[i] = o;
        } else {
            reinterpret_cast<float*>(yv)[i] = reinterpret_cast<const float*>(xv)[i] * cre;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
upsample_kernel(const T* __restrict__ x, T* __restrict__ y, long long n_out, int L) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_out; j += stride) {
        const long long q = j / L;
        T v{};
        if (j - q * L == 0) v = x[q];
        y[j] = v;
    }
}

__device__ __forceinline__ float2 fma_tap(float2 acc, float2 v, float h) { return __ffma2_rn(v, make_float2(h, h), acc); }
__device__ __forceinline__ float fma_tap(float acc, float v, float h) { return fmaf(v, h, acc); }
__device__ __forceinline__ float2 scaled(float2 v, float c) { return make_float2(v.x * c, v.y * c); }
__device__ __forceinline__ float scaled(float v, float c) { return v * c; }

// one thread per kept output m (global decimated index m0 + idx): J = m*D, q = floor(J/L), k0 = J mod L
template <typename T, bool SCALE>
__global__ void __launch_bounds__(256)
interp_fir_kernel(const T* __restrict__ x, const T* __restrict__ hist, T* __restrict__ y, const float* __restrict__ taps,
                  long long n_out, long long m0, long long c0, int Hn, int L, int D, int M, float c) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n_out; idx += stride) {
        const long long J = (m0 + idx) * D;
        const long long q = J / L;
        int k = (int)(J - q * L);
        int i = (int)(q - c0);                     // local input index of the newest contributing sample (< n)
        T acc{};
        for (; k < M; k += L, --i) {
            T v{};
            if (i >= 0) v = x[i];
            else if (Hn + i >= 0) v = hist[Hn + i];
            else break;                            // before the start of the stream: zeros
            if constexpr (SCALE) v = scaled(v, c);
            acc = fma_tap(acc, v, __ldg(taps + k));
        }
        y[idx] = acc;
    }
}

// ---- Interpolator (D == 1) and small-D rational resampler (D <= 4), 2 <= L <= 8: register-tiled polyphase kernel
// (for D > 1 all phases are computed and D-1 of D dropped at the store: still ~3x faster than one thread per kept output).  A thread owns IT_R consecutive inputs and
// all L phases (IT_R * L accumulators); per tap row t it needs x[i - t] for its IT_R inputs, a window that slides by one
// sample per row, so one new shared-memory value per row feeds IT_R * L multiply-adds.  The window is held as two aligned
// register chunks A = x[s0 - tb*R .. +R) and B = x[s0 - (tb+1)*R .. +R): every index below is a compile-time constant and
// the chunk loads are 128-bit.  Taps sit in shared memory as [t][p] and are read as warp-wide broadcasts.
constexpr int IT_R = 4;
constexpr int IT_THREADS = 128;

// 4 consecutive samples from a 16-byte aligned shared-memory position (index a multiple of 4)
__device__ __forceinline__ void load_chunk4(const float2* p, float2 (&o)[4]) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    o[0] = make_float2(a.x, a.y); o[1] = make_float2(a.z, a.w); o[2] = make_float2(b.x, b.y); o[3] = make_float2(b.z, b.w);
}
__device__ __forceinline__ void load_chunk4(const float* p, float (&o)[4]) {
    const float4 a = reinterpret_cast<const float4*>(p)[0];
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w;
}
constexpr int IT_TILE = IT_R * IT_THREADS;        // inputs per CTA tile

template <typename T, int L, bool SCALE>
__global__ void __launch_bounds__(IT_THREADS)
interp_tiled_kernel(const T* __restrict__ x, const T* __restrict__ hist, T* __restrict__ y, const float* __restrict__ taps_tp,
                    long long n, int Hn, int Tt, float c, int D, long long J0, long long m_lo) {
    extern __shared__ __align__(16) unsigned char it_smem[];
    float* hs = reinterpret_cast<float*>(it_smem);                       // [Tt][L]
    T* xs = reinterpret_cast<T*>(it_smem + (((size_t)Tt * L * sizeof(float) + 15) & ~(size_t)15));   // [Tt + IT_TILE], xs[Tt + j] = x[tile0 + j]
    const int tid = threadIdx.x;
    for (int i = tid; i < Tt * L; i += IT_THREADS) hs[i] = taps_tp[i];
    const long long ntiles = (n + IT_TILE - 1) / IT_TILE;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long tile0 = tile * IT_TILE;
        __syncthreads();                                                 // previous tile's reads are done (and hs is staged)
        for (int j = tid; j < Tt + IT_TILE; j += IT_THREADS) {
            const long long i = tile0 - Tt + j;
            T v{};
            if (i >= 0) { if (i < n) v = x[i]; }
            else if (Hn + i >= 0) v = hist[Hn + i];
            if constexpr (SCALE) v = scaled(v, c);
            xs[j] = v;
        }
        __syncthreads();
        const int s0 = Tt + tid * IT_R;                                  // smem position of this thread's first input
        T acc[IT_R][L];
#pragma unroll
        for (int r = 0; r < IT_R; ++r)
#pragma unroll
            for (int p = 0; p < L; ++p) acc[r][p] = T{};
        T A[IT_R], B[IT_R];
        load_chunk4(xs + s0, A);
#pragma unroll 1
        for (int tb = 0; tb < Tt / IT_R; ++tb) {
            load_chunk4(xs + s0 - (tb + 1) * IT_R, B);
#pragma unroll
            for (int sft = 0; sft < IT_R; ++sft) {
                float h[L];
#pragma unroll
                for (int p = 0; p < L; ++p) h[p] = hs[(tb * IT_R + sft) * L + p];
#pragma unroll
                for (int r = 0; r < IT_R; ++r) {
                    const T xv = (r - sft >= 0) ? A[(r - sft >= 0) ? r - sft : 0] : B[(r - sft < 0) ? IT_R + r - sft : 0];
#pragma unroll
                    for (int p = 0; p < L; ++p) acc[r][p] = fma_tap(acc[r][p], xv, h[p]);
                }
            }
#pragma unroll
            for (int r = 0; r < IT_R; ++r) A[r] = B[r];
        }
        const long long i0 = tile0 + (long long)tid * IT_R;
        if (D == 1) {
#pragma unroll
            for (int r = 0; r < IT_R; ++r) {
                if (i0 + r < n) {
                    T* yo = y + (i0 + r) * L;
#pragma unroll
                    for (int p = 0; p < L; ++p) yo[p] = acc[r][p];
                }
            }
        } else {
            // rational resampling with a small D: every phase was computed, keep the upsampled indices J = 0 (mod D).
            // J0 = global upsampled index of this call's first input, m_lo = global index of this call's first output.
            long long J = J0 + i0 * L;
            long long m = (J + D - 1) / D;                         // first kept output at or after J
            int gap = (int)(m * D - J);                            // its distance in upsampled samples
#pragma unroll
            for (int r = 0; r < IT_R; ++r) {
#pragma unroll
                for (int p = 0; p < L; ++p) {
                    if (gap == 0) {
                        if (i0 + r < n) y[m - m_lo] = acc[r][p];
                        ++m;
                        gap = D;
                    }
                    --gap;
                }
            }
        }
    }
}

// ---- Register-tiled polyphase resampler, any small (L, D) pair (interpolator: D == 1).
// Output m = aL + r' of period a reads inputs around q = aD + floor(r'D / L) with the taps of phase (r'D) mod L:
//     y[m] = sum_t h[p + tL] * c x[q - t].
// A thread owns RB periods = R = RB*L consecutive outputs (its first output is a multiple of L in absolute stream
// coordinates, so every phase p_r = (rD) mod L and input offset o_r = floor(rD / L) is a compile-time constant) and the
// RI = RB*D inputs they start from.  Per tap row t the R outputs need x[q0 + o_r - t]: a window that slides by one sample
// per row.  It lives in registers (a circular buffer, RI + C - 1 live samples for C rows), is refilled with C shared-memory loads per C rows,
// and feeds R multiply-adds per row; the taps are warp-uniform and come from the kernel-parameter constant bank as scalar
// operands.  The tile sits in shared memory TRANSPOSED, element e at (e mod RI) * NTP + e / RI: a window load is the same
// (row, column offset) for every thread plus its thread index, i.e. conflict-free for every (L, D).
// Only kept outputs are computed and only non-zero products: ceil(M / L) multiply-adds per output.
constexpr int RS_THREADS = 128;
constexpr int RS_C = 4;                       // tap rows per window refill
constexpr int RS_MAXT = 896;                  // taps incl. zero padding to Tt * L
constexpr int RS_NPOS = 168;                  // window positions: RI + Tt + 2C <= 20 + 132 + 8

__host__ __device__ constexpr int rs_mod(int a, int m) { return ((a % m) + m) % m; }

struct RsParams {
    float h[RS_MAXT];                         // h[t * L + p] = taps[p + t * L], zero padded
    long long c0, n;                          // absolute index of x[0], samples in this call
    long long m_lo, m_hi;                     // absolute output range of this call
    long long Mbase, ntiles;                  // first tile's first output (multiple of L, <= m_lo)
    int Tt, Hn, H, HB, NTP;                   // tap rows; history length; tile history (multiple of RI), H / RI; row pitch
    float c;
    unsigned short pos[RS_NPOS];              // pos[k] = shared-memory index of tile element H + RI - 1 - k (0 once that is negative)
};
static_assert(sizeof(RsParams) + 3 * sizeof(void*) <= 4096, "kernel parameters exceed 4 KB");

template <typename T, int L, int D, int RB>
__global__ void __launch_bounds__(RS_THREADS)
rs_poly_kernel(const T* __restrict__ x, const T* __restrict__ hist, T* __restrict__ y, const __grid_constant__ RsParams P) {
    constexpr int R = RB * L, RI = RB * D, C = RS_C, WN = RI + C - 1;
    constexpr int U = (WN + C + C - 1) / C, WP = U * C;      // circular window: WP >= WN + C
    extern __shared__ __align__(16) unsigned char rs_smem[];
    T* S = reinterpret_cast<T*>(rs_smem);
    const int tid = threadIdx.x;
    const int NTP = P.NTP, H = P.H;
    const int E = H + RS_THREADS * RI;
    const int nb = P.Tt / C;
    // A tile's E = H + 128 * RI elements (H <= 128, checked by the host) are fetched into KE registers per thread one tile
    // AHEAD: the loads of tile k+1 are in flight while tile k computes, so the global-memory latency is off the critical
    // path and the bytes in flight per SM do not depend on the occupancy (a load-stage-compute loop ran at 21-34 % of the HBM
    // roofline, latency-bound at 16 warps per SM).
    constexpr int KE = RI + 1;
    T pre[KE];
    auto fetch = [&](long long tile) {
        const long long lbase = ((P.Mbase + tile * (long long)(RS_THREADS * R)) / L) * D - H - P.c0;   // index into x of element 0
        const bool interior = lbase >= 0 && lbase + E <= P.n;
#pragma unroll
        for (int k = 0; k < KE; ++k) {
            const int e = tid + k * RS_THREADS;
            T v{};
            if (e < E) {
                const long long i = lbase + e;
                if (interior) v = __ldg(x + i);
                else if (i >= 0) { if (i < P.n) v = __ldg(x + i); }
                else if (P.Hn + i >= 0) v = __ldg(hist + (P.Hn + i));
            }
            pre[k] = v;
        }
    };
    long long tile = blockIdx.x;
    if (tile < P.ntiles) fetch(tile);
    for (; tile < P.ntiles; tile += gridDim.x) {
        const long long mt = P.Mbase + tile * (long long)(RS_THREADS * R);      // first output of the tile, multiple of L
        __syncthreads();                                                         // the previous tile's copy-out has read S
#pragma unroll
        for (int k = 0; k < KE; ++k) {
            const unsigned e = (unsigned)(tid + k * RS_THREADS);
            if (e < (unsigned)E) S[(e % RI) * NTP + e / RI] = scaled(pre[k], P.c);
        }
        __syncthreads();
        if (tile + gridDim.x < P.ntiles) fetch(tile + gridDim.x);
        // The window is a CIRCULAR register buffer of WP >= WN + C entries (WP a multiple of C): logical entry j of row block
        // tb lives at physical (j - tb*C) mod WP, so sliding the window by C moves nothing, and with the row-block loop unrolled
        // WP / C times every index is a compile-time constant.  The C entries of the NEXT block are loaded before this
        // block's multiply-adds into the slots the window has already left.
        T acc[R], W[WP];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = T{};
        const T* St = S + tid;
        // logical W[j] = element H + tid*RI + j - (C-1) - tb*C of the tile: rows t = tb*C + s read W[o_r - s + C - 1]
#pragma unroll
        for (int j = 0; j < WN; ++j) W[j] = St[P.pos[RI - 1 + C - 1 - j]];
#pragma unroll 1
        for (int tb0 = 0; tb0 < nb; tb0 += U) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int tb = tb0 + u;
                if (tb < nb) {                                   // warp-uniform
                    // unconditional (the table maps the positions past the last row block to a valid address): no inner
                    // branch, so the loads are scheduled ahead of this block's multiply-adds
                    const unsigned short* pk = P.pos + (RI - 1 + C - 1) + (tb + 1) * C;
#pragma unroll
                    for (int j = 0; j < C; ++j) W[rs_mod(j - (u + 1) * C, WP)] = St[pk[-j]];
                    const float* hb = P.h + tb * (C * L);
#pragma unroll
                    for (int s = 0; s < C; ++s) {
#pragma unroll
                        for (int r = 0; r < R; ++r)
                            acc[r] = fma_tap(acc[r], W[rs_mod((r * D) / L - s + C - 1 - u * C, WP)], hb[s * L + (r * D) % L]);
                    }
                }
            }
        }
        // Outputs leave through shared memory: a thread's R consecutive outputs are R * sizeof(T) apart from its neighbour's,
        // and storing them directly makes every warp store touch 32 sectors for 32 elements (measured: the x2 interpolator
        // ran at 21 % of the HBM roofline, store-bound).  Odd pitch RP: the per-thread writes are conflict-free, the copy-out
        // reads consecutive elements.
        constexpr int RP = R | 1;
        __syncthreads();                                                         // every window load of this tile is done
#pragma unroll
        for (int r = 0; r < R; ++r) S[tid * RP + r] = acc[r];
        __syncthreads();
        const long long ob = mt - P.m_lo;                                        // y index of the tile's first output
        if (mt >= P.m_lo && mt + RS_THREADS * R <= P.m_hi) {
#pragma unroll 4
            for (int o = tid; o < RS_THREADS * R; o += RS_THREADS) y[ob + o] = S[(o / R) * RP + o % R];
        } else {
            for (int o = tid; o < RS_THREADS * R; o += RS_THREADS) {
                const long long m = mt + o;
                if (m >= P.m_lo && m < P.m_hi) y[ob + o] = S[(o / R) * RP + o % R];
            }
        }
    }
}

// periods per thread for an instantiated (L, D), 0 otherwise
constexpr int rs_rb(int L, int D) {
    if (D == 1) return L == 2 ? 8 : (L <= 4 ? 4 : (L == 5 ? 3 : (L <= 8 ? 2 : 0)));
    if (L == 2 && (D == 3 || D == 5)) return 4;
    if (L == 3 && D == 2) return 4;
    if ((L == 3 && (D == 4 || D == 5)) || (L == 4 && (D == 3 || D == 5)) || (L == 5 && (D == 2 || D == 3 || D == 4))) return 3;
    if (L == 7 && D == 5) return 2;
    return 0;
}

struct RsGeom { int Tt, H, HB, NTP; size_t smem; };
RsGeom rs_geometry(int L, int D, int M, int elem) {
    const int RB = rs_rb(L, D), RI = RB * D;
    RsGeom g{};
    g.Tt = ((M + L - 1) / L + RS_C - 1) / RS_C * RS_C;
    g.HB = (g.Tt - 1 + RI - 1) / RI;
    if (g.HB < 1) g.HB = 1;
    g.H = g.HB * RI;
    const int banks = elem == 8 ? 16 : 32, k = (banks + RI - 1) / RI;       // consecutive elements of a staging store land k rows apart
    int ntp = g.HB + RS_THREADS + 1;
    while (ntp % banks != k % banks) ++ntp;
    g.NTP = ntp;
    const size_t tile_in = (size_t)RI * ntp, tile_out = (size_t)RS_THREADS * ((RB * L) | 1);     // the output staging reuses the tile
    g.smem = std::max(tile_in, tile_out) * elem;
    return g;
}

template <typename T, int L, int D>
int launch_rs(const RsParams& P, const void* x, const void* hist, void* y, size_t smem, cudaStream_t s) {
    constexpr int RB = rs_rb(L, D);
    auto k = rs_poly_kernel<T, L, D, RB>;
    static int per_sm_dev[LRB_MAX_DEVICES] = {0};
    static size_t smem_dev[LRB_MAX_DEVICES] = {0};
    const int dv = ctx().device & (LRB_MAX_DEVICES - 1);
    if (per_sm_dev[dv] == 0 || smem_dev[dv] != smem) {                        // resident CTAs per SM (registers, shared memory)
        int fit = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, k, RS_THREADS, smem) != cudaSuccess || fit < 1) fit = 1;
        per_sm_dev[dv] = std::min(fit, 8);
        smem_dev[dv] = smem;
    }
    const int per_sm = per_sm_dev[dv];
    const long long cap = (long long)ctx().sm_count * per_sm;
    const unsigned g = (unsigned)std::min<long long>(P.ntiles, cap);
    k<<<g, RS_THREADS, smem, s>>>((const T*)x, (const T*)hist, (T*)y, P);
    return 0;
}

int grid_for(long long n) {
    long long b = (n + 255) / 256;
    const long long cap = (long long)ctx().sm_count * 16;
    return (int)std::max<long long>(1, std::min(b, cap));
}

}  // namespace

// ---------------------------------------------------------------------------------------------
ScaleBlock::ScaleBlock(float re, float im, bool cdata, bool cconst, bool dev) : cre(re), cim(im), complex_data(cdata), complex_const(cconst) {
    name = "mulconst";
    in_size = out_size = cdata ? 8 : 4;
    dev_ptrs = dev;
}
int ScaleBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = n;
    consumed += n;
    if (n == 0) return 0;
    const int g = grid_for((long long)n);
    if (complex_data && complex_const) scale_kernel<true, true><<<g, 256, 0, s>>>(dx, dy, (long long)n, cre, cim);
    else if (complex_data) scale_kernel<true, false><<<g, 256, 0, s>>>(dx, dy, (long long)n, cre, cim);
    else scale_kernel<false, false><<<g, 256, 0, s>>>(dx, dy, (long long)n, cre, cim);
    count_launch();
    LRB_CHECK(cudaGetLastError());
    return 0;
}

UpsampleBlock::UpsampleBlock(unsigned factor, unsigned elem, bool dev) {
    name = "upsample";
    in_size = out_size = elem;
    dev_ptrs = dev;
    L = (int)factor;
}
int UpsampleBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    const long long no = (long long)n * L;
    *n_out = (size_t)no;
    consumed += n;
    if (n == 0) return 0;
    if (in_size == 8) upsample_kernel<float2><<<grid_for(no), 256, 0, s>>>((const float2*)dx, (float2*)dy, no, L);
    else upsample_kernel<float><<<grid_for(no), 256, 0, s>>>((const float*)dx, (float*)dy, no, L);
    count_launch();
    LRB_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------
InterpFirBlock::InterpFirBlock(bool cdata, const float* taps_host, int ntaps, int interp, int decim, bool has_scale_, float scale_, bool dev)
    : complex_data(cdata), L(interp), D(decim), M(ntaps), has_scale(has_scale_), scale(scale_) {
    label = std::string(has_scale ? "mulconst+" : "") + "upsample+fir" + (D > 1 ? "+down" : "") + "(" + std::to_string(M) + ",x" +
            std::to_string(L) + (D > 1 ? "/" + std::to_string(D) : "") + ")";
    name = label.c_str();
    in_size = out_size = cdata ? 8 : 4;
    dev_ptrs = dev;
    h_taps.assign(taps_host, taps_host + ntaps);
    Hn = (M + L - 1) / L;
}
InterpFirBlock::~InterpFirBlock() {
    cudaFree(d_taps);
    cudaFree(d_taps_tp);
}
int InterpFirBlock::init() {
    LRB_CHECK(cudaMalloc(&d_taps, sizeof(float) * (size_t)M));
    LRB_CHECK(cudaMemcpy(d_taps, h_taps.data(), sizeof(float) * (size_t)M, cudaMemcpyHostToDevice));
    Tt = ((M + L - 1) / L + IT_R - 1) / IT_R * IT_R;
    if (D <= 4 && L >= 2 && L <= 8 && (size_t)Tt * L * sizeof(float) + (size_t)(Tt + IT_TILE) * in_size + 16 <= 48 * 1024) {
        std::vector<float> tp((size_t)Tt * L, 0.0f);
        for (int k = 0; k < M; ++k) tp[(size_t)(k / L) * L + (k % L)] = h_taps[k];
        LRB_CHECK(cudaMalloc(&d_taps_tp, sizeof(float) * tp.size()));
        LRB_CHECK(cudaMemcpy(d_taps_tp, tp.data(), sizeof(float) * tp.size(), cudaMemcpyHostToDevice));
        if (Hn < Tt) Hn = Tt;                     // the tile staging reads Tt samples of history
    }
    // the register-tiled (L, D) kernel when the pair is instantiated and the padded taps fit the parameter bank
    if (rs_rb(L, D) > 0) {
        const RsGeom g = rs_geometry(L, D, M, (int)in_size);
        if (g.Tt * L <= RS_MAXT && g.smem <= 48 * 1024 && g.H <= RS_THREADS && rs_rb(L, D) * D + g.Tt + 2 * RS_C <= RS_NPOS) {
            rs_ok = true;
            if (Hn < g.Tt) Hn = g.Tt;
        }
    }
    return carry(hist, in_size * (size_t)Hn);
}
uint64_t InterpFirBlock::outputs_before(uint64_t idx) const { return (idx * (uint64_t)L + (uint64_t)D - 1) / (uint64_t)D; }
size_t InterpFirBlock::max_output(size_t n) const { return (size_t)(((unsigned long long)n * L) / D + 2); }
int InterpFirBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    const long long m_lo = (long long)outputs_before(consumed), m_hi = (long long)outputs_before(consumed + n);
    const long long no = m_hi - m_lo;
    *n_out = (size_t)no;
    if (n == 0) return 0;
    if (no > 0 && rs_ok) {
        const RsGeom g = rs_geometry(L, D, M, (int)in_size);
        RsParams P;
        for (int i = 0; i < g.Tt * L; ++i) P.h[i] = i < M ? h_taps[i] : 0.0f;      // h[t*L + p] = taps[p + t*L]: natural order
        P.c0 = (long long)consumed; P.n = (long long)n; P.m_lo = m_lo; P.m_hi = m_hi;
        P.Mbase = (m_lo / L) * L;
        const long long TO = (long long)RS_THREADS * rs_rb(L, D) * L;
        P.ntiles = (m_hi - P.Mbase + TO - 1) / TO;
        P.Tt = g.Tt; P.Hn = Hn; P.H = g.H; P.HB = g.HB; P.NTP = g.NTP;
        {
            const int RI = rs_rb(L, D) * D;
            for (int k = 0; k < RS_NPOS; ++k) {
                const int ep = g.H + RI - 1 - k;
                P.pos[k] = ep >= 0 ? (unsigned short)((ep % RI) * g.NTP + ep / RI) : (unsigned short)0;
            }
        }
        P.c = has_scale ? scale : 1.0f;
#define LRB_RS(LL, DD) case (LL) * 32 + (DD): \
            if (complex_data) launch_rs<float2, LL, DD>(P, dx, hist.in(), dy, g.smem, s); \
            else launch_rs<float, LL, DD>(P, dx, hist.in(), dy, g.smem, s); \
            break;
        switch (L * 32 + D) {
            LRB_RS(2, 1) LRB_RS(3, 1) LRB_RS(4, 1) LRB_RS(5, 1) LRB_RS(6, 1) LRB_RS(7, 1) LRB_RS(8, 1)
            LRB_RS(2, 3) LRB_RS(2, 5) LRB_RS(3, 2) LRB_RS(3, 4) LRB_RS(3, 5) LRB_RS(4, 3) LRB_RS(4, 5)
            LRB_RS(5, 2) LRB_RS(5, 3) LRB_RS(5, 4) LRB_RS(7, 5)
            default: set_error("resampler: no kernel for this (L, D)"); return -1;
        }
#undef LRB_RS
        count_launch();
        LRB_CHECK(cudaGetLastError());
    } else if (no > 0 && d_taps_tp) {
        const long long ntiles = ((long long)n + IT_TILE - 1) / IT_TILE;
        const int g = (int)std::min<long long>(ntiles, (long long)ctx().sm_count * 8);
        const size_t smem = (((size_t)Tt * L * sizeof(float) + 15) & ~(size_t)15) + (size_t)(Tt + IT_TILE) * in_size;
#define LRB_IT2(T, LL, S) interp_tiled_kernel<T, LL, S><<<g, IT_THREADS, smem, s>>>((const T*)dx, (const T*)hist.in(), (T*)dy, d_taps_tp, (long long)n, Hn, Tt, scale, D, (long long)consumed * L, m_lo)
#define LRB_IT(LL) \
        if (complex_data) { if (has_scale) LRB_IT2(float2, LL, true); else LRB_IT2(float2, LL, false); } \
        else { if (has_scale) LRB_IT2(float, LL, true); else LRB_IT2(float, LL, false); }
        switch (L) {
            case 2: LRB_IT(2); break;
            case 3: LRB_IT(3); break;
            case 4: LRB_IT(4); break;
            case 5: LRB_IT(5); break;
            case 6: LRB_IT(6); break;
            case 7: LRB_IT(7); break;
            default: LRB_IT(8); break;
        }
#undef LRB_IT
#undef LRB_IT2
        count_launch();
        LRB_CHECK(cudaGetLastError());
    } else if (no > 0) {
        const int g = grid_for(no);
#define LRB_IF(T, S) interp_fir_kernel<T, S><<<g, 256, 0, s>>>((const T*)dx, (const T*)hist.in(), (T*)dy, d_taps, no, m_lo, (long long)consumed, Hn, L, D, M, scale)
        if (complex_data) { if (has_scale) LRB_IF(float2, true); else LRB_IF(float2, false); }
        else { if (has_scale) LRB_IF(float, true); else LRB_IF(float, false); }
#undef LRB_IF
        count_launch();
        LRB_CHECK(cudaGetLastError());
    }
    if (launch_hist_update(dx, (long long)n, hist.in(), hist.out(), Hn, (int)in_size, s) != 0) return -1;
    hist.flip();
    consumed += n;
    return 0;
}

}  // namespace lrb
