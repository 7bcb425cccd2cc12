// Source boundary (SURVEY.md 8f row 1): IQFileSource sample formats -> ComplexFloat32 on the device, so that a
// host-fed graph moves the file's own bytes over PCIe (2 B/sample for RTL-SDR style u8 IQ instead of 8).
//
// Reference: radio/blocks/sources/iqfile.lua:96-108 (byte swap loop, then (value - offset) / scale per component) with
// the table radio/utilities/format_utils.lua:82-97.  The reference computes in double and stores float32; here
// 8/16-bit formats use correctly rounded float32 (operands exact, one division), 32-bit and f64 formats double.
#include "common.cuh"
#include "blocks.h"

#include <algorithm>
#include <cstring>
#include <string>
#include <new>

namespace lrb {

namespace {

enum IqFmt { F_U8, F_S8, F_U16, F_S16, F_U32, F_S32, F_F32, F_F64 };

__device__ __forceinline__ uint16_t bswap16(uint16_t v) { return (uint16_t)((v >> 8) | (v << 8)); }
__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
__device__ __forceinline__ uint64_t bswap64(uint64_t v) {
    return ((uint64_t)bswap32((uint32_t)v) << 32) | bswap32((uint32_t)(v >> 32));
}

// n / 127.5 for the 8-bit formats: quotient estimate + one FMA residual correction (3 instructions instead of the IEEE
// division sequence).  Equal to the reference's double-precision (v - offset) / scale rounded to float32 for all 512
// possible inputs (checked exhaustively; tests/test_gpu_golden.py::test_iqconv_8bit_all_values_bit_exact).
__device__ __forceinline__ float div127p5(float n) {
    const float r = 1.0f / 127.5f;
    const float q = n * r;
    return fmaf(fmaf(-q, 127.5f, n), r, q);
}

// same scheme for the 16-bit formats (n / 32767.5; all 2 x 65536 inputs checked against the double-precision result)
__device__ __forceinline__ float div32767p5(float n) {
    const float r = 1.0f / 32767.5f;
    const float q = n * r;
    return fmaf(fmaf(-q, 32767.5f, n), r, q);
}

template <int FMT, bool SWAP>
__device__ __forceinline__ float conv16(uint32_t h) {          // h: the 16 raw bits in the low half
    uint16_t v = (uint16_t)h;
    if (SWAP) v = bswap16(v);
    return FMT == F_U16 ? div32767p5((float)v - 32767.5f) : div32767p5((float)(int16_t)v);
}

template <int FMT, bool SWAP>
__device__ __forceinline__ float conv_one(const unsigned char* p) {
    if constexpr (FMT == F_U8) return div127p5((float)p[0] - 127.5f);
    if constexpr (FMT == F_S8) return div127p5((float)(signed char)p[0]);
    if constexpr (FMT == F_U16 || FMT == F_S16) {
        uint16_t v = *reinterpret_cast<const uint16_t*>(p);
        if (SWAP) v = bswap16(v);
        return FMT == F_U16 ? div32767p5((float)v - 32767.5f) : div32767p5((float)(int16_t)v);
    }
    if constexpr (FMT == F_U32 || FMT == F_S32) {
        uint32_t v = *reinterpret_cast<const uint32_t*>(p);
        if (SWAP) v = bswap32(v);
        const double d = FMT == F_U32 ? ((double)v - 2147483647.5) : (double)(int32_t)v;
        return (float)(d / 2147483647.5);
    }
    if constexpr (FMT == F_F32) {
        uint32_t v = *reinterpret_cast<const uint32_t*>(p);
        if (SWAP) v = bswap32(v);
        return __uint_as_float(v);
    }
    if constexpr (FMT == F_F64) {
        uint64_t v = *reinterpret_cast<const uint64_t*>(p);
        if (SWAP) v = bswap64(v);
        return (float)__longlong_as_double((long long)v);
    }
    return 0.f;
}

template <int FMT, bool SWAP, int BYTES>
__global__ void __launch_bounds__(256)
iqconv_kernel(const unsigned char* __restrict__ x, float2* __restrict__ y, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned char* p = x + i * (2 * BYTES);
        y[i] = make_float2(conv_one<FMT, SWAP>(p), conv_one<FMT, SWAP>(p + BYTES));
    }
}

// u8 IQ (the RTL-SDR wire format): one 32-bit load (two I/Q samples) and one 128-bit store per thread and iteration, so
// both the loads and the stores of a warp are contiguous (128 B in, 512 B out); four iterations in flight per thread.
__global__ void __launch_bounds__(256)
iqconv_u8_vec_kernel(const uint32_t* __restrict__ x, float4* __restrict__ y, long long n2) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n2; i += 4 * stride) {
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = __ldcs(x + i + k * stride);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float4 o;
            o.x = div127p5((float)(w[k] & 0xff) - 127.5f);
            o.y = div127p5((float)((w[k] >> 8) & 0xff) - 127.5f);
            o.z = div127p5((float)((w[k] >> 16) & 0xff) - 127.5f);
            o.w = div127p5((float)(w[k] >> 24) - 127.5f);
            __stcs(y + i + k * stride, o);
        }
    }
    for (; i < n2; i += stride) {
        const uint32_t w = __ldcs(x + i);
        float4 o;
        o.x = div127p5((float)(w & 0xff) - 127.5f);
        o.y = div127p5((float)((w >> 8) & 0xff) - 127.5f);
        o.z = div127p5((float)((w >> 16) & 0xff) - 127.5f);
        o.w = div127p5((float)(w >> 24) - 127.5f);
        __stcs(y + i, o);
    }
}

// 16-bit I/Q: one 64-bit load (two samples) and one 128-bit store per thread and iteration, warp-contiguous both ways
template <int FMT, bool SWAP>
__global__ void __launch_bounds__(256)
iqconv16_vec_kernel(const uint2* __restrict__ x, float4* __restrict__ y, long long n2) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n2; i += 4 * stride) {
        uint2 w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = __ldcs(x + i + k * stride);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            __stcs(y + i + k * stride, make_float4(conv16<FMT, SWAP>(w[k].x), conv16<FMT, SWAP>(w[k].x >> 16),
                                                   conv16<FMT, SWAP>(w[k].y), conv16<FMT, SWAP>(w[k].y >> 16)));
    }
    for (; i < n2; i += stride) {
        const uint2 w = __ldcs(x + i);
        __stcs(y + i, make_float4(conv16<FMT, SWAP>(w.x), conv16<FMT, SWAP>(w.x >> 16), conv16<FMT, SWAP>(w.y), conv16<FMT, SWAP>(w.y >> 16)));
    }
}

struct FmtInfo { const char* name; int fmt; int bytes; bool big_endian; };
const FmtInfo FORMATS[] = {
    {"u8", F_U8, 1, false}, {"s8", F_S8, 1, false},
    {"u16le", F_U16, 2, false}, {"u16be", F_U16, 2, true}, {"s16le", F_S16, 2, false}, {"s16be", F_S16, 2, true},
    {"u32le", F_U32, 4, false}, {"u32be", F_U32, 4, true}, {"s32le", F_S32, 4, false}, {"s32be", F_S32, 4, true},
    {"f32le", F_F32, 4, false}, {"f32be", F_F32, 4, true}, {"f64le", F_F64, 8, false}, {"f64be", F_F64, 8, true},
};

struct IqConvBlock : Block {
    FmtInfo info;
    std::string label;
    explicit IqConvBlock(const FmtInfo& f, bool dev) : info(f) {
        label = std::string("iqconv(") + f.name + ")";
        name = label.c_str();
        in_size = (size_t)2 * f.bytes;
        out_size = 8;
        dev_ptrs = dev;
    }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override {
        *n_out = n;
        consumed += n;
        if (n == 0) return 0;
        const unsigned char* x = (const unsigned char*)dx;
        float2* y = (float2*)dy;
        const long long nn = (long long)n;
        int blocks = (int)((nn + 255) / 256);
        const int cap = ctx().sm_count * 16;
        if (blocks > cap) blocks = cap;
        const bool sw = info.big_endian;          // device is little endian
#define LRB_CONV(F, B) \
        if (sw) iqconv_kernel<F, true, B><<<blocks, 256, 0, s>>>(x, y, nn); else iqconv_kernel<F, false, B><<<blocks, 256, 0, s>>>(x, y, nn)
        switch (info.fmt) {
            case F_U8:
                if ((reinterpret_cast<uintptr_t>(x) & 3) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 && nn >= 2) {
                    const long long n2 = nn / 2;
                    int vb = (int)((n2 + 255) / 256);
                    if (vb > cap) vb = cap;
                    iqconv_u8_vec_kernel<<<vb, 256, 0, s>>>((const uint32_t*)x, (float4*)y, n2);
                    if (nn % 2) { iqconv_kernel<F_U8, false, 1><<<1, 32, 0, s>>>(x + n2 * 4, y + n2 * 2, 1); count_launch(); }
                } else {
                    iqconv_kernel<F_U8, false, 1><<<blocks, 256, 0, s>>>(x, y, nn);
                }
                break;
            case F_S8: iqconv_kernel<F_S8, false, 1><<<blocks, 256, 0, s>>>(x, y, nn); break;
            case F_U16:
            case F_S16:
                if ((reinterpret_cast<uintptr_t>(x) & 7) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 && nn >= 2) {
                    const long long n2 = nn / 2;
                    int vb = (int)((n2 + 255) / 256);
                    if (vb > cap) vb = cap;
                    const uint2* x2 = (const uint2*)x;
                    float4* y4 = (float4*)y;
                    if (info.fmt == F_U16) { if (sw) iqconv16_vec_kernel<F_U16, true><<<vb, 256, 0, s>>>(x2, y4, n2); else iqconv16_vec_kernel<F_U16, false><<<vb, 256, 0, s>>>(x2, y4, n2); }
                    else { if (sw) iqconv16_vec_kernel<F_S16, true><<<vb, 256, 0, s>>>(x2, y4, n2); else iqconv16_vec_kernel<F_S16, false><<<vb, 256, 0, s>>>(x2, y4, n2); }
                    if (nn % 2) {
                        const unsigned char* xt = x + n2 * 8;
                        float2* yt = y + n2 * 2;
                        if (info.fmt == F_U16) { if (sw) iqconv_kernel<F_U16, true, 2><<<1, 32, 0, s>>>(xt, yt, 1); else iqconv_kernel<F_U16, false, 2><<<1, 32, 0, s>>>(xt, yt, 1); }
                        else { if (sw) iqconv_kernel<F_S16, true, 2><<<1, 32, 0, s>>>(xt, yt, 1); else iqconv_kernel<F_S16, false, 2><<<1, 32, 0, s>>>(xt, yt, 1); }
                        count_launch();
                    }
                } else if (info.fmt == F_U16) { LRB_CONV(F_U16, 2); } else { LRB_CONV(F_S16, 2); }
                break;
            case F_U32: LRB_CONV(F_U32, 4); break;
            case F_S32: LRB_CONV(F_S32, 4); break;
            case F_F32: LRB_CONV(F_F32, 4); break;
            default: LRB_CONV(F_F64, 8); break;
        }
#undef LRB_CONV
        count_launch();
        LRB_CHECK(cudaGetLastError());
        return 0;
    }
};


// ---- RealFileSource (radio/blocks/sources/realfile.lua:86-104): the same per-component map, one component per sample
template <int FMT, bool SWAP, int BYTES>
__global__ void __launch_bounds__(256)
realconv_kernel(const unsigned char* __restrict__ x, float* __restrict__ y, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        y[i] = conv_one<FMT, SWAP>(x + i * BYTES);
}

// ---- Sink boundary: Float32 / ComplexFloat32 -> file sample format, on the device, so that the D2H copy carries the
// file's bytes (2 B/sample for 16-bit WAV instead of 4).  Reference: IQFileSink:process (radio/blocks/sinks/iqfile.lua:
// 66-80), RealFileSink (sinks/realfile.lua), WAVFileSink:process (sinks/wavfile.lua:170-186): raw = x*scale + offset in
// double, stored into the C integer type (truncation toward zero), then the byte swap.  Values outside [-1, 1] are
// undefined behaviour in the reference's double -> integer store; here they saturate.
template <int BYTES> struct RawT;
template <> struct RawT<1> { typedef uint8_t type; };
template <> struct RawT<2> { typedef uint16_t type; };
template <> struct RawT<4> { typedef uint32_t type; };
template <> struct RawT<8> { typedef uint64_t type; };

template <int FMT, bool SWAP>
__device__ __forceinline__ typename RawT<(FMT == F_U8 || FMT == F_S8) ? 1 : (FMT == F_U16 || FMT == F_S16) ? 2 : (FMT == F_F64 ? 8 : 4)>::type
sink_one(float xf) {
    constexpr double scale = (FMT == F_U8 || FMT == F_S8) ? 127.5 : (FMT == F_U16 || FMT == F_S16) ? 32767.5
                             : (FMT == F_U32 || FMT == F_S32) ? 2147483647.5 : 1.0;
    constexpr double offset = FMT == F_U8 ? 127.5 : FMT == F_U16 ? 32767.5 : FMT == F_U32 ? 2147483647.5 : 0.0;
    const double v = __dadd_rn(__dmul_rn((double)xf, scale), offset);
    if constexpr (FMT == F_F32) { uint32_t b = __float_as_uint((float)v); return SWAP ? bswap32(b) : b; }
    else if constexpr (FMT == F_F64) { uint64_t b = (uint64_t)__double_as_longlong(v); return SWAP ? bswap64(b) : b; }
    else {
        long long t = __double2ll_rz(v);
        constexpr long long lo = FMT == F_S8 ? -128LL : FMT == F_S16 ? -32768LL : FMT == F_S32 ? -2147483648LL : 0LL;
        constexpr long long hi = FMT == F_U8 ? 255LL : FMT == F_S8 ? 127LL : FMT == F_U16 ? 65535LL : FMT == F_S16 ? 32767LL
                                 : FMT == F_U32 ? 4294967295LL : 2147483647LL;
        t = t < lo ? lo : (t > hi ? hi : t);
        if constexpr (FMT == F_U8 || FMT == F_S8) return (uint8_t)t;
        else if constexpr (FMT == F_U16 || FMT == F_S16) { uint16_t b = (uint16_t)t; return SWAP ? bswap16(b) : b; }
        else { uint32_t b = (uint32_t)t; return SWAP ? bswap32(b) : b; }
    }
}

template <int BYTES> struct alignas(4 * BYTES) Raw4 { typename RawT<BYTES>::type v[4]; };

// four components per thread: one 128-bit load, one 4*BYTES store; VEC = false: any alignment, one component per thread
template <int FMT, bool SWAP, int BYTES, bool VEC>
__global__ void __launch_bounds__(256)
sinkconv_kernel(const float* __restrict__ x, unsigned char* __restrict__ y, long long n) {
    typedef typename RawT<BYTES>::type T;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (VEC) {
        const long long n4 = n / 4;
        for (long long i = tid; i < n4; i += stride) {
            const float4 v = __ldcs(reinterpret_cast<const float4*>(x) + i);
            Raw4<BYTES> o;
            o.v[0] = sink_one<FMT, SWAP>(v.x);
            o.v[1] = sink_one<FMT, SWAP>(v.y);
            o.v[2] = sink_one<FMT, SWAP>(v.z);
            o.v[3] = sink_one<FMT, SWAP>(v.w);
            reinterpret_cast<Raw4<BYTES>*>(y)[i] = o;
        }
        if (tid < n - n4 * 4) reinterpret_cast<T*>(y)[n4 * 4 + tid] = sink_one<FMT, SWAP>(x[n4 * 4 + tid]);
    } else {
        for (long long i = tid; i < n; i += stride) {
            const T b = sink_one<FMT, SWAP>(x[i]);
            memcpy(y + i * BYTES, &b, BYTES);
        }
    }
}

// direction / arity of the three other file-format blocks
struct FileConvBlock : Block {
    FmtInfo info;
    bool to_file;             // true: float -> raw (sinks); false: raw -> float (RealFileSource)
    int comps;                // components per sample (1 real, 2 complex)
    std::string label;
    FileConvBlock(const FmtInfo& f, bool to_file_, int comps_, bool dev) : info(f), to_file(to_file_), comps(comps_) {
        label = std::string(to_file ? (comps == 2 ? "iqsink(" : "realsink(") : "realconv(") + f.name + ")";
        name = label.c_str();
        in_size = to_file ? 4 * (size_t)comps : (size_t)f.bytes * comps;
        out_size = to_file ? (size_t)f.bytes * comps : 4 * (size_t)comps;
        dev_ptrs = dev;
    }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override {
        *n_out = n;
        consumed += n;
        if (n == 0) return 0;
        const long long nc = (long long)n * comps;
        const int cap = ctx().sm_count * 16;
        const bool sw = info.big_endian;
        if (!to_file) {
            int blocks = (int)std::min<long long>((nc + 255) / 256, cap);
            const unsigned char* x = (const unsigned char*)dx;
            float* y = (float*)dy;
#define LRB_RC(F, B) \
            if (sw) realconv_kernel<F, true, B><<<blocks, 256, 0, s>>>(x, y, nc); else realconv_kernel<F, false, B><<<blocks, 256, 0, s>>>(x, y, nc)
            switch (info.fmt) {
                case F_U8: realconv_kernel<F_U8, false, 1><<<blocks, 256, 0, s>>>(x, y, nc); break;
                case F_S8: realconv_kernel<F_S8, false, 1><<<blocks, 256, 0, s>>>(x, y, nc); break;
                case F_U16: LRB_RC(F_U16, 2); break;
                case F_S16: LRB_RC(F_S16, 2); break;
                case F_U32: LRB_RC(F_U32, 4); break;
                case F_S32: LRB_RC(F_S32, 4); break;
                case F_F32: LRB_RC(F_F32, 4); break;
                default: LRB_RC(F_F64, 8); break;
            }
#undef LRB_RC
        } else {
            const float* x = (const float*)dx;
            unsigned char* y = (unsigned char*)dy;
            const bool vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) % (4 * info.bytes)) == 0;
            const long long threads = vec ? std::max<long long>(nc / 4, 4) : nc;
            int blocks = (int)std::min<long long>((threads + 255) / 256, cap);
#define LRB_SK2(F, SW, B) \
            if (vec) sinkconv_kernel<F, SW, B, true><<<blocks, 256, 0, s>>>(x, y, nc); else sinkconv_kernel<F, SW, B, false><<<blocks, 256, 0, s>>>(x, y, nc)
#define LRB_SK(F, B) \
            if (sw) { LRB_SK2(F, true, B); } else { LRB_SK2(F, false, B); }
            switch (info.fmt) {
                case F_U8: LRB_SK2(F_U8, false, 1); break;
                case F_S8: LRB_SK2(F_S8, false, 1); break;
                case F_U16: LRB_SK(F_U16, 2); break;
                case F_S16: LRB_SK(F_S16, 2); break;
                case F_U32: LRB_SK(F_U32, 4); break;
                case F_S32: LRB_SK(F_S32, 4); break;
                case F_F32: LRB_SK(F_F32, 4); break;
                default: LRB_SK(F_F64, 8); break;
            }
#undef LRB_SK
#undef LRB_SK2
        }
        count_launch();
        LRB_CHECK(cudaGetLastError());
        return 0;
    }
};

}  // namespace

Block* make_iqconv(const char* format, bool dev) {
    if (!format) { set_error("iqconv: format is NULL"); return nullptr; }
    for (const FmtInfo& f : FORMATS)
        if (std::strcmp(f.name, format) == 0) {
            return make_block<IqConvBlock>(f, dev);
        }
    set_error("Unsupported format (\"%s\")", format);     // iqfile.lua:46
    return nullptr;
}

Block* make_fileconv(const char* format, bool to_file, int comps, bool dev) {
    if (!format) { set_error("fileconv: format is NULL"); return nullptr; }
    for (const FmtInfo& f : FORMATS)
        if (std::strcmp(f.name, format) == 0) {
            return make_block<FileConvBlock>(f, to_file, comps, dev);
        }
    set_error("Unsupported format (\"%s\")", format);
    return nullptr;
}

}  // namespace lrb
