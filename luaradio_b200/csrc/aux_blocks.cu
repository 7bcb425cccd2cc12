// Blocks either side of the hot path (SURVEY.md 8f rows 3 and 4): the two-input element-wise blocks and DelayBlock that
// the WBFM-stereo / AM-synchronous chains add to it, and the power spectral density of the spectrum sinks.
//
//   MultiplyBlock / MultiplyConjugateBlock / AddBlock / SubtractBlock
//       radio/blocks/signal/multiply.lua, multiplyconjugate.lua:26-51, add.lua, subtract.lua
//       (volk_32fc_x2_multiply_32fc / volk_32fc_x2_multiply_conjugate_32fc / volk_32f_x2_add_32f ... or Lua loops)
//   DelayBlock   radio/blocks/signal/delay.lua:26-60: y[n] = x[n - D], D zeros first, state of D samples carried
//   PSD          radio/utilities/spectrum_utils.lua:524-642: window -> DFT -> |X_k|^2 / (rate * window energy) [-> 10 log10]
//
// All HBM-streaming kernels (128-bit accesses where the pointers allow); the PSD runs one CTA per frame with the
// transform in shared memory (frames of up to 4096 points, power of two).
#include "../../include/lrb200.h"
#include "common.cuh"
#include "blocks.h"
#include "fft32_gen.cuh"

#include <cmath>
#include <new>
#include <string>
#include <vector>

namespace lrb {

namespace {

constexpr int AX_THREADS = 256;

inline int ax_grid(long long items) {
    long long blocks = (items + AX_THREADS - 1) / AX_THREADS;
    long long cap = (long long)ctx().sm_count * 16;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

enum BinOp { BIN_MUL = 0, BIN_MULCONJ = 1, BIN_ADD = 2, BIN_SUB = 3 };

template <int OP>
__device__ __forceinline__ float2 bin_c(float2 a, float2 b) {
    if constexpr (OP == BIN_MUL) return cmul(a, b);
    if constexpr (OP == BIN_MULCONJ) return cmul(a, make_float2(b.x, -b.y));
    if constexpr (OP == BIN_ADD) return __fadd2_rn(a, b);
    return __fadd2_rn(a, make_float2(-b.x, -b.y));
}
template <int OP>
__device__ __forceinline__ float bin_r(float a, float b) {
    if constexpr (OP == BIN_MUL || OP == BIN_MULCONJ) return a * b;
    if constexpr (OP == BIN_ADD) return a + b;
    return a - b;
}

// complex: two samples per thread per step (128-bit); real: four
template <int OP>
__global__ void __launch_bounds__(AX_THREADS)
binary_c_kernel(const float2* __restrict__ a, const float2* __restrict__ b, float2* __restrict__ y, long long n, int vec_ok) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec_ok) {
        const long long np = n >> 1;
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(b);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (; p < np; p += stride) {
            const float4 u = __ldcs(a4 + p), v = __ldcs(b4 + p);
            const float2 r0 = bin_c<OP>(make_float2(u.x, u.y), make_float2(v.x, v.y));
            const float2 r1 = bin_c<OP>(make_float2(u.z, u.w), make_float2(v.z, v.w));
            __stcs(y4 + p, make_float4(r0.x, r0.y, r1.x, r1.y));
        }
        if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) y[n - 1] = bin_c<OP>(a[n - 1], b[n - 1]);
    } else {
        for (; p < n; p += stride) y[p] = bin_c<OP>(a[p], b[p]);
    }
}
template <int OP>
__global__ void __launch_bounds__(AX_THREADS)
binary_r_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ y, long long n, int vec_ok) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec_ok) {
        const long long nq = n >> 2;
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(b);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (; p < nq; p += stride) {
            const float4 u = __ldcs(a4 + p), v = __ldcs(b4 + p);
            __stcs(y4 + p, make_float4(bin_r<OP>(u.x, v.x), bin_r<OP>(u.y, v.y), bin_r<OP>(u.z, v.z), bin_r<OP>(u.w, v.w)));
        }
        if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
            const long long i = (nq << 2) + threadIdx.x;
            y[i] = bin_r<OP>(a[i], b[i]);
        }
    } else {
        for (; p < n; p += stride) y[p] = bin_r<OP>(a[p], b[p]);
    }
}

// delay.lua:36-60 on 4-byte words (a complex sample is two words): y[i] = i < Dw ? state[i] : x[i - Dw];
// new_state[j] = logical(n - Dw + j) over [state | x]
__global__ void __launch_bounds__(AX_THREADS)
delay_kernel(const uint32_t* __restrict__ x, const uint32_t* __restrict__ st_in, uint32_t* __restrict__ st_out,
             uint32_t* __restrict__ y, long long nw, long long Dw) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += stride)
        y[i] = i < Dw ? st_in[i] : x[i - Dw];
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < Dw; j += stride) {
        const long long l = nw + j;                       // logical index into [state | x], minus Dw
        st_out[j] = l < Dw ? st_in[l] : x[l - Dw];
    }
}

// ---- PSD: one CTA per frame of N points (power of two, <= 4096): window, radix-2 FFT in shared memory, |X|^2 / scale
__global__ void __launch_bounds__(256)
psd_kernel(const void* __restrict__ xv, const float* __restrict__ window, float* __restrict__ y, int N, int logN,
           int complex_in, float inv_scale, int logarithmic, const float2* __restrict__ tw /* W_N^k, k < N/2 */) {
    extern __shared__ float2 sm[];
    const long long frame = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    // load in bit-reversed order with the window applied (spectrum_utils.lua:598-606)
    for (int i = tid; i < N; i += nt) {
        const int r = (int)(__brev((unsigned)i) >> (32 - logN));
        const float w = window[i];
        float2 v;
        if (complex_in) {
            v = reinterpret_cast<const float2*>(xv)[frame * N + i];
            v = make_float2(v.x * w, v.y * w);
        } else {
            v = make_float2(reinterpret_cast<const float*>(xv)[frame * N + i] * w, 0.f);
        }
        sm[r] = v;
    }
    __syncthreads();
    for (int s = 1; s <= logN; ++s) {
        const int half = 1 << (s - 1);
        for (int k = tid; k < N / 2; k += nt) {
            const int j = k & (half - 1);
            const int i0 = ((k >> (s - 1)) << s) + j;
            const float2 wv = tw[j << (logN - s)];        // W_N^(j * N / 2^s), forward sign
            const float2 a = sm[i0], b = cmul(sm[i0 + half], wv);
            sm[i0] = __fadd2_rn(a, b);
            sm[i0 + half] = __fadd2_rn(a, make_float2(-b.x, -b.y));
        }
        __syncthreads();
    }
    for (int i = tid; i < N; i += nt) {
        const float2 v = sm[i];
        float p = fmaf(v.x, v.x, v.y * v.y) * inv_scale;
        if (logarithmic) p = 10.0f * log10f(p);
        y[frame * N + i] = p;
    }
}

// ---- PSD of 1024-point frames (the spectrum sinks' default size): one WARP per frame on the register-resident 32 x 32
// transform of fir_fft.cu -- window at the load, DFT32 over n1, twiddle, one warp-private transpose, DFT32 over n2, and
// |X_k|^2 / scale written lane-contiguously (k = lane + 32 k2).  No CTA barrier in the frame loop.
constexpr int PS_WARPS = 4;
constexpr int PS_XSTRIDE = 33;
__global__ void __launch_bounds__(PS_WARPS * 32)
psd1024_kernel(const void* __restrict__ xv, const float* __restrict__ window, float* __restrict__ y, long long frames,
               int complex_in, float inv_scale, int logarithmic, const float2* __restrict__ tw) {
    extern __shared__ __align__(16) float2 psm[];
    float2* s_tw = psm;                                            // [k1][n2] W1024^(k1 n2)
    float* s_win = reinterpret_cast<float*>(psm + 1024);           // 1024 floats
    float2* xch = psm + 1024 + 512 + (threadIdx.x >> 5) * (32 * PS_XSTRIDE);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 1024; i += PS_WARPS * 32) { s_tw[i] = tw[i]; s_win[i] = window[i]; }
    __syncthreads();
    const long long wstride = (long long)gridDim.x * PS_WARPS;
    for (long long f = (long long)blockIdx.x * PS_WARPS + warp; f < frames; f += wstride) {
        float2 v[32];
        if (complex_in) {
            const float2* xb = reinterpret_cast<const float2*>(xv) + f * 1024 + lane;
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const float2 t = __ldcs(xb + 32 * r);
                const float w = s_win[32 * r + lane];
                v[r] = make_float2(t.x * w, t.y * w);
            }
        } else {
            const float* xb = reinterpret_cast<const float*>(xv) + f * 1024 + lane;
#pragma unroll
            for (int r = 0; r < 32; ++r) v[r] = make_float2(__ldcs(xb + 32 * r) * s_win[32 * r + lane], 0.f);
        }
        fft32_nat2br<false>(v);
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; ++k1) {
            float2 t = v[bitrev5(k1)];
            if (k1 > 0) t = cmul(t, s_tw[k1 * 32 + lane]);
            xch[k1 * PS_XSTRIDE + lane] = t;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 32; ++r) v[r] = xch[lane * PS_XSTRIDE + r];
        fft32_nat2br<false>(v);
        float* yb = y + f * 1024 + lane;
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2) {
            const float2 t = v[bitrev5(k2)];
            float p = fmaf(t.x, t.x, t.y * t.y) * inv_scale;
            if (logarithmic) p = 10.0f * log10f(p);
            __stcs(yb + 32 * k2, p);
        }
    }
}

// ---- PLLBlock (radio/blocks/signal/pll.lua:140-170): a NONLINEAR recurrence -- phase detector atan2f(x conj(vco)),
// second-order loop filter, frequency clamp, phase wrap -- restated operation by operation (Lua numbers are doubles; the
// VCO output, the phase-detector product and the error are rounded to float32 where the reference stores them in
// ComplexFloat32 / Float32 cells).  One thread runs the stream in order: exact for any input, locked or not, at a few
// MS/s (the reference's Lua loop: 5 MS/s on its i5).  state = {phi_locked, phi_multiplied, freq_locked}.
struct PllParams { double alpha, beta, fmin, fmax, mult; };
__global__ void pll_kernel(const float2* __restrict__ x, long long n, float2* __restrict__ out, float* __restrict__ err,
                           double* __restrict__ state, PllParams P) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    double phi = state[0], phim = state[1], freq = state[2];
    const double two_pi = 6.283185307179586476925286766559;
    for (long long i = 0; i < n; ++i) {
        double s, c, sm_, cm_;
        sincos(phi, &s, &c);
        sincos(phim, &sm_, &cm_);
        const float vr = (float)c, vi = (float)s;
        out[i] = make_float2((float)cm_, (float)sm_);
        const float2 xv = x[i];
        // x * conj(vco), each component computed in double and stored as float32 (complexfloat32.lua:79-81)
        const float pr = (float)((double)xv.x * (double)vr - (double)xv.y * (double)(-vi));
        const float pi = (float)((double)xv.x * (double)(-vi) + (double)xv.y * (double)vr);
        const float e = atan2f(pi, pr);
        err[i] = e;
        freq = freq + P.beta * (double)e;
        phi = phi + freq + P.alpha * (double)e;
        phim = phim + freq * P.mult + P.alpha * (double)e;
        freq = freq > P.fmax ? P.fmax : freq;
        freq = freq < P.fmin ? P.fmin : freq;
        phi = phi > two_pi ? phi - two_pi : phi;
        phi = phi < -two_pi ? phi + two_pi : phi;
        phim = phim > two_pi ? phim - two_pi : phim;
        phim = phim < -two_pi ? phim + two_pi : phim;
    }
    state[0] = phi; state[1] = phim; state[2] = freq;
}

// ---- chunk-parallel PLL (opt-in, lrb200_pll_set_mode(q, 1)).  Valid while the loop is LOCKED: from a phase guess
// arg(x) and the centre frequency the second-order loop converges to the stream's own (phi_locked, freq_locked)
// trajectory within W = 24 / (zeta * loop bandwidth) samples, so every chunk can be simulated by its own thread after a
// W-sample lead-in (chunk 0 starts from the carried state and is exact).  phi_multiplied is NOT a function of the locked
// state (it integrates multiplier * freq + alpha * error over the whole past), so it is rebuilt exactly from prefix sums
// over the chunks: with A[i] = sum_{k<i} (freq'_k + alpha e_k) and E[i] = sum_{k<i} e_k,
//     phi_multiplied[i] = phi_multiplied[0] + m A[i] + (1 - m) alpha E[i]     (mod 2 pi).
struct PllChunk { double freq0, dA, dE, phi_end, freq_end, A0, E0; };

__device__ __forceinline__ float pll_step(float2 xv, double& phi, double& freq, const PllParams& P, double& inc) {
    const double two_pi = 6.283185307179586476925286766559;
    double s, c;
    sincos(phi, &s, &c);
    const float vr = (float)c, vi = (float)s;
    const float pr = (float)((double)xv.x * (double)vr - (double)xv.y * (double)(-vi));
    const float pi = (float)((double)xv.x * (double)(-vi) + (double)xv.y * (double)vr);
    const float e = atan2f(pi, pr);
    freq = freq + P.beta * (double)e;
    inc = freq + P.alpha * (double)e;
    phi = phi + inc;
    freq = freq > P.fmax ? P.fmax : freq;
    freq = freq < P.fmin ? P.fmin : freq;
    phi = phi > two_pi ? phi - two_pi : phi;
    phi = phi < -two_pi ? phi + two_pi : phi;
    return e;
}

__global__ void __launch_bounds__(128)
pll_sim_kernel(const float2* __restrict__ x, long long n, float* __restrict__ err, long long L, long long W, int nchunks,
               const double* __restrict__ state, PllParams P, PllChunk* __restrict__ chunks) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    const long long start = (long long)c * L, end = start + L < n ? start + L : n;
    double phi, freq, inc;
    if (c == 0) {
        phi = state[0];
        freq = state[2];
    } else {
        const long long begin = start - W;                       // L >= W, so begin >= 0
        const float2 x0 = x[begin];
        phi = (double)atan2f(x0.y, x0.x);
        freq = 0.5 * (P.fmin + P.fmax);
        for (long long i = begin; i < start; ++i) pll_step(x[i], phi, freq, P, inc);
    }
    PllChunk r;
    r.freq0 = freq;
    double dA = 0.0, dE = 0.0;
    for (long long i = start; i < end; ++i) {
        const float e = pll_step(x[i], phi, freq, P, inc);
        err[i] = e;
        dA += inc;
        dE += (double)e;
    }
    r.dA = dA; r.dE = dE; r.phi_end = phi; r.freq_end = freq; r.A0 = 0.0; r.E0 = 0.0;
    chunks[c] = r;
}

__global__ void pll_prefix_kernel(PllChunk* chunks, int nchunks, double* state, PllParams P) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const double two_pi = 6.283185307179586476925286766559;
    double A = 0.0, E = 0.0;
    for (int c = 0; c < nchunks; ++c) {
        chunks[c].A0 = A; chunks[c].E0 = E;
        A += chunks[c].dA; E += chunks[c].dE;
    }
    // carried state for the next call; state[3] keeps this call's phi_multiplied[0] for the output kernel
    state[3] = state[1];
    state[0] = chunks[nchunks - 1].phi_end;
    state[2] = chunks[nchunks - 1].freq_end;
    state[1] = fmod(state[1] + P.mult * A + (1.0 - P.mult) * P.alpha * E, two_pi);
}

__global__ void __launch_bounds__(128)
pll_out_kernel(const float* __restrict__ err, long long n, float2* __restrict__ out, long long L, int nchunks,
               const double* __restrict__ state, PllParams P, const PllChunk* __restrict__ chunks) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    const long long start = (long long)c * L, end = start + L < n ? start + L : n;
    const double phim0 = state[3];
    double A = chunks[c].A0, E = chunks[c].E0, freq = chunks[c].freq0;
    const double two_pi = 6.283185307179586476925286766559;
    for (long long i = start; i < end; ++i) {
        double ph = phim0 + P.mult * A + (1.0 - P.mult) * P.alpha * E;
        ph -= two_pi * floor(ph / two_pi);                  // keep sincos in its accurate range
        double s, cc;
        sincos(ph, &s, &cc);
        out[i] = make_float2((float)cc, (float)s);
        const double e = (double)err[i];
        freq = freq + P.beta * e;
        A += freq + P.alpha * e;
        E += e;
        freq = freq > P.fmax ? P.fmax : freq;
        freq = freq < P.fmin ? P.fmin : freq;
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
struct PllBlock : Block {
    PllParams P;
    double init_freq;
    double* d_state = nullptr;      // phi_locked, phi_multiplied, freq_locked, (scratch) phi_multiplied at call start
    int mode = 0;                   // 0 = exact sequential, 1 = chunk-parallel (locked loop)
    long long warm = 0;             // lead-in of the chunk-parallel form
    PllChunk* d_chunks = nullptr;
    int chunk_cap = 0;
    PllBlock(double loop_bw_hz, double fmin_hz, double fmax_hz, double multiplier, double rate, bool dev) {
        name = "pll";
        in_size = 8;
        out_size = 8;
        dev_ptrs = dev;
        num_outputs = 2;
        // pll.lua:113-131
        double bw = 2 * M_PI * (loop_bw_hz / rate);
        P.fmin = 2 * M_PI * (fmin_hz / rate);
        P.fmax = 2 * M_PI * (fmax_hz / rate);
        const double damping = std::sqrt(2.0) / 2;
        bw = bw / (damping + 1 / (4 * damping));
        const double denom = 1 + 2 * damping * bw + bw * bw;
        P.alpha = (4 * damping * bw) / denom;
        P.beta = (4 * bw * bw) / denom;
        P.mult = multiplier;
        init_freq = (P.fmin + P.fmax) / 2.0;
        warm = (long long)std::ceil(24.0 / (damping * bw));
    }
    ~PllBlock() override { cudaFree(d_state); cudaFree(d_chunks); }
    size_t out_size_of(int port) const override { return port == 0 ? 8 : 4; }
    long long memory_in() const override { return -1; }        // the multiplied phase integrates the whole past
    int set_state(cudaStream_t s) {
        const double h[3] = {0.0, 0.0, init_freq};
        LRB_CHECK(cudaMemcpyAsync(d_state, h, sizeof(h), cudaMemcpyHostToDevice, s));
        return 0;
    }
    int init() override {
        LRB_CHECK(cudaMalloc(&d_state, 4 * sizeof(double)));
        if (set_state(ctx().stream) != 0) return -1;
        LRB_CHECK(cudaStreamSynchronize(ctx().stream));
        return 0;
    }
    // the one block whose reset state is not zero (the loop starts at the middle of its frequency range), so d_state is
    // not carried state: reset rewrites it here instead of zeroing it
    void reset_host() override { consumed = 0; set_state(ctx().stream); cudaStreamSynchronize(ctx().stream); }
    int run(const void*, size_t, void*, size_t*, cudaStream_t) override {
        set_error("pll has two outputs (out, error): use lrb200_block_execute_multi");
        return -1;
    }
    int run_multi(const void* const* dx, int nin, size_t n, void* const* dy, int nout, size_t* n_out, cudaStream_t s) override {
        if (nin != 1 || nout != 2) { set_error("pll: expected 1 input and 2 outputs"); return -1; }
        *n_out = n;
        if (n == 0) return 0;
        const long long L = warm * 4 > 16384 ? warm * 4 : 16384;
        if (mode == 1 && (long long)n >= 2 * L) {
            const int nchunks = (int)(((long long)n + L - 1) / L);
            if (nchunks > chunk_cap) {
                LRB_CHECK(cudaStreamSynchronize(s));
                cudaFree(d_chunks);
                d_chunks = nullptr;
                LRB_CHECK(cudaMalloc(&d_chunks, sizeof(PllChunk) * (size_t)nchunks));
                chunk_cap = nchunks;
            }
            const int blocks = (nchunks + 127) / 128;
            pll_sim_kernel<<<blocks, 128, 0, s>>>((const float2*)dx[0], (long long)n, (float*)dy[1], L, warm, nchunks, d_state, P, d_chunks);
            pll_prefix_kernel<<<1, 32, 0, s>>>(d_chunks, nchunks, d_state, P);
            pll_out_kernel<<<blocks, 128, 0, s>>>((const float*)dy[1], (long long)n, (float2*)dy[0], L, nchunks, d_state, P, d_chunks);
            count_launch(3);
            LRB_CHECK(cudaGetLastError());
            consumed += n;
            return 0;
        }
        pll_kernel<<<1, 32, 0, s>>>((const float2*)dx[0], (long long)n, (float2*)dy[0], (float*)dy[1], d_state, P);
        count_launch();
        LRB_CHECK(cudaGetLastError());
        consumed += n;
        return 0;
    }
};

struct BinaryBlock : Block {
    int op;
    bool cplx;
    std::string label;
    BinaryBlock(int op_, bool cplx_, bool dev) : op(op_), cplx(cplx_) {
        static const char* names[] = {"multiply", "multiplyconjugate", "add", "subtract"};
        label = std::string(names[op]) + (cplx ? "_cc" : "_rr");
        name = label.c_str();
        in_size = out_size = cplx ? 8 : 4;
        dev_ptrs = dev;
        num_inputs = 2;
    }
    int run(const void*, size_t, void*, size_t*, cudaStream_t) override {
        set_error("%s needs two inputs: use lrb200_block_execute_multi", name);
        return -1;
    }
    int run_multi(const void* const* dx, int nin, size_t n, void* const* dy, int nout, size_t* n_out, cudaStream_t s) override {
        if (nin != 2 || nout != 1) { set_error("%s: expected 2 inputs and 1 output", name); return -1; }
        *n_out = n;
        if (n == 0) return 0;
        const int vec = ((reinterpret_cast<uintptr_t>(dx[0]) | reinterpret_cast<uintptr_t>(dx[1]) | reinterpret_cast<uintptr_t>(dy[0])) & 15) == 0;
        const int grid = ax_grid((long long)n / (cplx ? 2 : 4) + 1);
#define LRB_BIN(OP)                                                                                                        \
        if (cplx) binary_c_kernel<OP><<<grid, AX_THREADS, 0, s>>>((const float2*)dx[0], (const float2*)dx[1], (float2*)dy[0], (long long)n, vec); \
        else binary_r_kernel<OP><<<grid, AX_THREADS, 0, s>>>((const float*)dx[0], (const float*)dx[1], (float*)dy[0], (long long)n, vec);
        switch (op) {
            case BIN_MUL: LRB_BIN(BIN_MUL) break;
            case BIN_MULCONJ: LRB_BIN(BIN_MULCONJ) break;
            case BIN_ADD: LRB_BIN(BIN_ADD) break;
            default: LRB_BIN(BIN_SUB) break;
        }
#undef LRB_BIN
        count_launch();
        LRB_CHECK(cudaGetLastError());
        consumed += n;
        return 0;
    }
};

struct DelayBlock : Block {
    long long D;
    Carried state;                  // last D inputs
    DelayBlock(unsigned num_samples, unsigned elem, bool dev) : D(num_samples) {
        name = "delay";
        in_size = out_size = elem;
        dev_ptrs = dev;
    }
    int init() override { return carry(state, (size_t)D * in_size); }
    long long memory_in() const override { return D; }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override {
        *n_out = n;
        if (n == 0) return 0;
        const long long wpe = (long long)in_size / 4;
        const long long nw = (long long)n * wpe, Dw = D * wpe;
        delay_kernel<<<ax_grid(nw > Dw ? nw : Dw), AX_THREADS, 0, s>>>((const uint32_t*)dx, (const uint32_t*)state.in(),
                                                                        (uint32_t*)state.out(), (uint32_t*)dy, nw, Dw);
        count_launch();
        LRB_CHECK(cudaGetLastError());
        state.flip();
        consumed += n;
        return 0;
    }
};

struct PsdBlock : Block {
    int N, logN;
    bool cplx, logarithmic;
    float inv_scale;
    std::vector<float> h_window;
    float* d_window = nullptr;
    float2* d_tw = nullptr;
    float2* d_tw1024 = nullptr;      // N == 1024: inter-pass twiddles of the register-resident transform
    PsdBlock(int N_, const float* window, double scale, bool log_, bool cplx_, bool dev)
        : N(N_), cplx(cplx_), logarithmic(log_), inv_scale((float)(1.0 / scale)) {
        name = "psd";
        in_size = cplx ? 8 : 4;
        out_size = 4;
        dev_ptrs = dev;
        logN = 0;
        while ((1 << logN) < N) ++logN;
        h_window.assign(window, window + N);
    }
    ~PsdBlock() override { cudaFree(d_window); cudaFree(d_tw); cudaFree(d_tw1024); }
    int init() override {
        std::vector<float2> tw((size_t)N / 2 + 1);
        for (int k = 0; k < N / 2; ++k)
            tw[(size_t)k] = make_float2((float)std::cos(2 * M_PI * k / N), (float)(-std::sin(2 * M_PI * k / N)));
        LRB_CHECK(cudaMalloc(&d_window, sizeof(float) * (size_t)N));
        LRB_CHECK(cudaMalloc(&d_tw, sizeof(float2) * ((size_t)N / 2 + 1)));
        LRB_CHECK(cudaMemcpy(d_window, h_window.data(), sizeof(float) * (size_t)N, cudaMemcpyHostToDevice));
        LRB_CHECK(cudaMemcpy(d_tw, tw.data(), sizeof(float2) * ((size_t)N / 2 + 1), cudaMemcpyHostToDevice));
        if (N == 1024) {
            std::vector<float2> t2(1024);
            for (int a = 0; a < 32; ++a)
                for (int c = 0; c < 32; ++c) {
                    const int e = (a * c) % 1024;
                    t2[(size_t)a * 32 + c] = make_float2((float)std::cos(2 * M_PI * e / 1024.0), (float)(-std::sin(2 * M_PI * e / 1024.0)));
                }
            LRB_CHECK(cudaMalloc(&d_tw1024, sizeof(float2) * 1024));
            LRB_CHECK(cudaMemcpy(d_tw1024, t2.data(), sizeof(float2) * 1024, cudaMemcpyHostToDevice));
        }
        return 0;
    }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override {
        if (n % (size_t)N) { set_error("psd: the input must be a whole number of %d-sample frames (got %zu samples)", N, n); return -1; }
        *n_out = n;
        if (n == 0) return 0;
        const size_t frames = n / (size_t)N;
        if (frames > 2147483647u) { set_error("psd: too many frames in one call"); return -1; }
        if (N == 1024) {
            constexpr size_t smem = sizeof(float2) * (1024 + 512 + PS_WARPS * 32 * PS_XSTRIDE);
            long long ctas = ((long long)frames + PS_WARPS - 1) / PS_WARPS;
            const long long cap = (long long)ctx().sm_count * 4;
            if (ctas > cap) ctas = cap;
            psd1024_kernel<<<(unsigned)ctas, PS_WARPS * 32, smem, s>>>(dx, d_window, (float*)dy, (long long)frames, cplx ? 1 : 0, inv_scale,
                                                                        logarithmic ? 1 : 0, d_tw1024);
            count_launch();
            LRB_CHECK(cudaGetLastError());
            consumed += n;
            return 0;
        }
        psd_kernel<<<(unsigned)frames, 256, sizeof(float2) * (size_t)N, s>>>(dx, d_window, (float*)dy, N, logN, cplx ? 1 : 0,
                                                                              inv_scale, logarithmic ? 1 : 0, d_tw);
        count_launch();
        LRB_CHECK(cudaGetLastError());
        consumed += n;
        return 0;
    }
};

}  // namespace lrb

using namespace lrb;

extern "C" {

lrb200_block_t* lrb200_binary_create(const char* op, unsigned complex_data, unsigned flags) {
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    const std::string o = op ? op : "";
    int code = o == "multiply" ? BIN_MUL : o == "multiplyconjugate" ? BIN_MULCONJ : o == "add" ? BIN_ADD : o == "subtract" ? BIN_SUB : -1;
    if (code < 0) { set_error("binary: unknown operation \"%s\" (multiply, multiplyconjugate, add, subtract)", o.c_str()); return nullptr; }
    if (code == BIN_MULCONJ && !complex_data) { set_error("binary: multiplyconjugate needs complex data"); return nullptr; }
    return wrap(make_block<BinaryBlock>(code, complex_data != 0, (flags & LRB200_DEVICE) != 0));
}

lrb200_block_t* lrb200_pll_create(double loop_bandwidth, double frequency_min, double frequency_max, double multiplier,
                                  double rate, unsigned flags) {
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    if (!(rate > 0.0) || !(loop_bandwidth > 0.0) || !std::isfinite(multiplier)) { set_error("pll: rate and loop bandwidth must be positive"); return nullptr; }
    if (!(frequency_min <= frequency_max)) { set_error("pll: frequency_min must not exceed frequency_max"); return nullptr; }
    return wrap(make_block<PllBlock>(loop_bandwidth, frequency_min, frequency_max, multiplier, rate, (flags & LRB200_DEVICE) != 0));
}

int lrb200_pll_set_mode(lrb200_block_t* q, int mode) {
    PllBlock* p = q && q->impl ? dynamic_cast<PllBlock*>(q->impl) : nullptr;
    if (!p) { set_error("not a PLL handle"); return -1; }
    if (mode != 0 && mode != 1) { set_error("pll: mode must be 0 (exact, sequential) or 1 (chunk-parallel, locked loop)"); return -1; }
    p->mode = mode;
    return 0;
}

lrb200_block_t* lrb200_delay_create(unsigned num_samples, unsigned elem_size, unsigned flags) {
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    if (num_samples == 0) { set_error("delay: number of samples must be greater than 0"); return nullptr; }
    if (elem_size != 4 && elem_size != 8) { set_error("delay: elem_size must be 4 or 8"); return nullptr; }
    return wrap(make_block<DelayBlock>(num_samples, elem_size, (flags & LRB200_DEVICE) != 0));
}

lrb200_block_t* lrb200_psd_create(unsigned num_samples, const float32_t* window, double scale, unsigned logarithmic,
                                  unsigned complex_data, unsigned flags) {
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    if (num_samples < 2 || num_samples > 4096 || (num_samples & (num_samples - 1))) {
        set_error("psd: the frame length must be a power of two in 2..4096 (got %u)", num_samples);
        return nullptr;
    }
    if (!window) { set_error("psd: missing window"); return nullptr; }
    if (!(scale > 0.0)) { set_error("psd: scale (sample rate * window energy) must be positive"); return nullptr; }
    return wrap(make_block<PsdBlock>((int)num_samples, (const float*)window, scale, logarithmic != 0, complex_data != 0,
                                     (flags & LRB200_DEVICE) != 0));
}

}  // extern "C"
