// C ABI of libluaradio_b200.so (include/lrb200.h): context, block objects with their carried
// streaming state, and the single-stream GPU flow graph.  No CPU fallback: every entry point needs a
// CUDA device and fails loudly (return code + lrb200_last_error) without one.
#include "../../include/lrb200.h"
#include "common.cuh"
#include "blocks.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <new>

namespace lrb {

static thread_local char g_err[512] = "";
static Ctx g_ctx;

Ctx& ctx() { return g_ctx; }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

bool cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return false;
}

cudaStream_t side_fork(cudaStream_t s) {
    Ctx& c = g_ctx;
    if (!c.side) {
        if (cudaStreamCreateWithFlags(&c.side, cudaStreamNonBlocking) != cudaSuccess) { c.side = nullptr; return s; }
        cudaEventCreateWithFlags(&c.ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&c.ev_join, cudaEventDisableTiming);
    }
    if (cudaEventRecord(c.ev_fork, s) != cudaSuccess || cudaStreamWaitEvent(c.side, c.ev_fork, 0) != cudaSuccess) return s;
    return c.side;
}

void side_join(cudaStream_t s, cudaStream_t side) {
    if (side == s) return;
    cudaEventRecord(g_ctx.ev_join, side);
    cudaStreamWaitEvent(s, g_ctx.ev_join, 0);
}

static int ensure_init() {
    if (g_ctx.device >= 0) return 0;
    return lrb200_init(0);
}

// ---------------------------------------------------------------------------------------------
// Block base: host-pointer (drop-in) mode stages through grow-only device buffers in chunks.
// ---------------------------------------------------------------------------------------------
static constexpr size_t HOST_CHUNK = (size_t)1 << 24;   // samples per staged chunk in host mode

Block::~Block() {
    for (void* p : staging) cudaFree(p);
}

int Block::carry(Carried& c, size_t bytes, int slots) {
    for (int i = 0; i < slots; ++i) {
        LRB_CHECK(cudaMalloc(&c.slot[i], bytes));
        LRB_CHECK(cudaMemset(c.slot[i], 0, bytes));
    }
    c.bytes = bytes;
    carried.push_back(&c);
    return 0;
}

int Block::execute_multi(const void* const* x, int nin, size_t n, void* const* y, int nout, size_t* n_out) {
    cudaStream_t s = ctx().stream;
    if (nin != num_inputs || nout != num_outputs) {
        set_error("%s: expected %d input(s) and %d output(s), got %d and %d", name, num_inputs, num_outputs, nin, nout);
        return -1;
    }
    size_t produced = 0;
    if (dev_ptrs) {
        if (run_multi(x, nin, n, y, nout, &produced, s) != 0) return -1;
        if (n_out) *n_out = produced;
        return 0;
    }
    if (staging.empty()) { staging.assign((size_t)(nin + nout), nullptr); staging_cap.assign((size_t)(nin + nout), 0); }
    size_t done = 0;
    std::vector<const void*> din((size_t)nin);
    std::vector<void*> dout((size_t)nout);
    while (done < n) {
        const size_t nc = n - done < HOST_CHUNK ? n - done : HOST_CHUNK;
        const size_t mo = max_output(nc);
        for (int i = 0; i < nin; ++i) {
            if (reserve(&staging[(size_t)i], &staging_cap[(size_t)i], nc * in_size) != 0) return -1;
            LRB_CHECK(cudaMemcpyAsync(staging[(size_t)i], (const char*)x[i] + done * in_size, nc * in_size, cudaMemcpyHostToDevice, s));
            din[(size_t)i] = staging[(size_t)i];
        }
        for (int o = 0; o < nout; ++o) {
            if (reserve(&staging[(size_t)(nin + o)], &staging_cap[(size_t)(nin + o)], (mo ? mo : 1) * out_size_of(o)) != 0) return -1;
            dout[(size_t)o] = staging[(size_t)(nin + o)];
        }
        size_t no = 0;
        if (run_multi(din.data(), nin, nc, dout.data(), nout, &no, s) != 0) return -1;
        for (int o = 0; o < nout; ++o)
            if (no) LRB_CHECK(cudaMemcpyAsync((char*)y[o] + produced * out_size_of(o), dout[(size_t)o], no * out_size_of(o), cudaMemcpyDeviceToHost, s));
        // the staging buffers are reused by the next chunk: drain before overwriting them
        LRB_CHECK(cudaStreamSynchronize(s));
        produced += no;
        done += nc;
    }
    if (n_out) *n_out = produced;
    return 0;
}

int Block::reserve(void** p, size_t* cap, size_t bytes) {
    if (bytes <= *cap) return 0;
    cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    LRB_CHECK(cudaMalloc(p, bytes));
    *cap = bytes;
    return 0;
}

int Block::reset() {
    reset_host();
    std::vector<std::pair<void*, size_t>> segs;
    state_buffers(segs);
    for (auto& sg : segs) LRB_CHECK(cudaMemsetAsync(sg.first, 0, sg.second, ctx().stream));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// FIR (+ Hilbert)
// ---------------------------------------------------------------------------------------------
FirBlock::FirBlock(FirKind k, const void* taps_host, unsigned ntaps, unsigned decim, bool dev, bool rot, double turns_per_sample) {
    kind = k;
    M = (int)ntaps;
    D = (int)decim;
    dev_ptrs = dev;
    const bool cin = (k == FIR_CRCF || k == FIR_CCCF);
    in_size = cin ? 8 : 4;
    out_size = (cin || k == FIR_HILBERT) ? 8 : 4;
    tap_size = (k == FIR_CCCF) ? 8 : 4;
    name = k == FIR_CRCF ? "fir_crcf" : k == FIR_CCCF ? "fir_cccf" : k == FIR_RRRF ? "fir_rrrf" : "hilbert";
    h_taps.assign((const char*)taps_host, (const char*)taps_host + (size_t)M * tap_size);
    rotate = rot;
    rot_turns = turns_per_sample;
    rot_fix = turns_to_fix(turns_per_sample);
}

int FirBlock::init() {
    LRB_CHECK(cudaMalloc(&d_taps, (size_t)M * tap_size));
    LRB_CHECK(cudaMemcpy(d_taps, h_taps.data(), (size_t)M * tap_size, cudaMemcpyHostToDevice));
    if (carry(hist, (size_t)(M > 1 ? M - 1 : 1) * in_size) != 0) return -1;
    return fast_init();
}

int FirBlock::set_pole(float c) {
    if (carry(pole, sizeof(float)) != 0) return -1;
    has_pole = true;
    pole_c = c;
    return 0;
}

FirBlock::~FirBlock() {
    cudaFree(d_taps);
    fast_free();
}

static long long decay_samples(double c) {        // samples until |c|^k < 1e-12; < 0 if it never gets there
    const double a = std::fabs(c);
    if (a == 0.0) return 0;
    if (a >= 1.0) return -1;
    return (long long)std::ceil(std::log(1e-12) / std::log(a)) + 1;
}

long long FirBlock::memory_in() const {
    long long m = M - 1;
    if (has_pole) {
        const long long w = decay_samples((double)pole_c);
        if (w < 0) return -1;
        m += w * D;
    }
    return m;
}
long long IirBlock::memory_in() const {
    const long long w = decay_samples((double)c);
    return w < 0 ? -1 : w + nb;
}

int FirBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    const auto [first, no] = plan(n);
    *n_out = (size_t)no;
    if (n == 0) return 0;
    // the history for the next call depends only on x and the old history: side stream, concurrent with the filter
    // (short calls -- the reference's 8192-sample vectors -- are launch-latency bound: no fork/join events for them)
    cudaStream_t side = s;
    if (M > 1) {
        if (n >= SIDE_STREAM_MIN) side = side_fork(s);
        if (launch_hist_update(dx, (long long)n, hist.in(), hist.out(), M - 1, (int)in_size, side) != 0) return -1;
    }
    int rc = fast_run(dx, n, dy, first, no, s);
    if (rc == 0) rc = launch_fir_generic(kind, dx, hist.in(), d_taps, M, D, first, no, dy, s) == 0 ? 1 : -1;
    side_join(s, side);
    if (rc < 0) return -1;
    if (M > 1) hist.flip();
    if (has_pole && no > 0) pole.flip();
    consumed += n;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// FrequencyTranslator
// ---------------------------------------------------------------------------------------------
RotatorBlock::RotatorBlock(double turns_per_sample, bool dev) {
    name = "rotator";
    in_size = out_size = 8;
    dev_ptrs = dev;
    turns = turns_per_sample;
    turns_fix = turns_to_fix(turns_per_sample);
}

int RotatorBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = n;
    if (launch_rotator((const float2*)dx, (float2*)dy, (long long)n, turns_fix, consumed, s) != 0) return -1;
    consumed += n;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// FrequencyDiscriminator
// ---------------------------------------------------------------------------------------------
DiscrimBlock::DiscrimBlock(float gain_, bool dev) {
    name = "discrim";
    in_size = 8;
    out_size = 4;
    dev_ptrs = dev;
    gain = gain_;
}
int DiscrimBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = n;
    if (n == 0) return 0;
    if (launch_discrim((const float2*)dx, (const float2*)prev.in(), (float*)dy, (long long)n, 1.0f / gain, s) != 0) return -1;
    if (launch_copy_last(dx, (long long)n, prev.out(), 8, s) != 0) return -1;
    consumed += n;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Downsampler
// ---------------------------------------------------------------------------------------------
DownsampleBlock::DownsampleBlock(unsigned factor, unsigned elem, bool dev) {
    name = "downsample";
    in_size = out_size = elem;
    dev_ptrs = dev;
    D = (int)factor;
}
int DownsampleBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    const auto [first, no] = plan(n);
    *n_out = (size_t)no;
    if (launch_downsample(dx, dy, first, no, D, (int)in_size, s) != 0) return -1;
    consumed += n;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// IIR (single pole: na <= 2)
// ---------------------------------------------------------------------------------------------
IirBlock::IirBlock(bool cplx, const float* b_, unsigned nb_, const float* a_, unsigned na_, bool dev) {
    name = cplx ? "iir_crcf" : "iir_rrrf";
    in_size = out_size = cplx ? 8 : 4;
    dev_ptrs = dev;
    complex_data = cplx;
    nb = (int)nb_;
    double a0 = a_[0];
    for (int j = 0; j < nb; ++j) b[j] = (float)((double)b_[j] / a0);
    c = (na_ >= 2) ? (float)(-(double)a_[1] / a0) : 0.0f;
}
int IirBlock::init() {
    if (carry(xhist, (size_t)(nb > 1 ? nb - 1 : 1) * in_size) != 0 || carry(ystate, in_size) != 0) return -1;
    return iir_work_alloc(&work, (int)in_size);
}
IirBlock::~IirBlock() { iir_work_free(&work); }
int IirBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = (size_t)plan(n).n_out;
    const long long maxn = iir_max_per_launch(work);
    size_t done = 0, produced = 0;
    while (done < n) {
        long long nc = (long long)(n - done) < maxn ? (long long)(n - done) : maxn;
        const auto [first, no] = plan((size_t)nc);
        if (launch_iir1(complex_data, (const char*)dx + done * in_size, nc, (char*)dy + produced * out_size, b, nb, c,
                        xhist.in(), xhist.out(), ystate.in(), ystate.out(), first, D, &work, s) != 0)
            return -1;
        xhist.flip();
        ystate.flip();
        consumed += (uint64_t)nc;
        done += (size_t)nc;
        produced += (size_t)no;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// IIR of any order
// ---------------------------------------------------------------------------------------------
IirGeneralBlock::IirGeneralBlock(bool cplx, const float* b_, unsigned nb_, const float* a_, unsigned na_, bool dev) {
    name = cplx ? "iir_crcf(general)" : "iir_rrrf(general)";
    in_size = out_size = cplx ? 8 : 4;
    dev_ptrs = dev;
    complex_data = cplx;
    nb = (int)nb_;
    na = (int)na_;
    const double a0 = a_[0];
    for (int j = 0; j < nb; ++j) b[j] = (float)((double)b_[j] / a0);
    for (int j = 0; j < na; ++j) a[j] = (float)((double)a_[j] / a0);
    // impulse response of 1/A(z) in float64: last index where |h| >= 1e-10 * peak
    const int limit = 1 << 16;
    std::vector<double> h(limit);
    double peak = 0.0;
    long long last = 0;
    for (int i = 0; i < limit; ++i) {
        double v = (i == 0) ? 1.0 : 0.0;
        for (int j = 1; j < na && j <= i; ++j) v -= (double)a[j] * h[i - j];
        h[i] = v;
        if (std::fabs(v) > peak) peak = std::fabs(v);
        if (!std::isfinite(v)) { last = limit; break; }
        if (std::fabs(v) >= 1e-10 * peak) last = i;
    }
    warm = (last + na + nb >= limit - 1) ? -1 : last + na + nb;
}
int IirGeneralBlock::init() { return carry(xhist, 10 * in_size) != 0 ? -1 : carry(yhist, 10 * in_size); }
int IirGeneralBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = n;
    if (n == 0) return 0;
    if (launch_iir_general(complex_data, dx, (long long)n, dy, b, nb, a, na, xhist.in(), yhist.in(), warm, s) != 0) return -1;
    // carried state: last nb-1 inputs of [xhist | x], last na-1 outputs of [yhist | y] (oldest first)
    if (nb > 1 && launch_hist_update(dx, (long long)n, xhist.in(), xhist.out(), nb - 1, (int)in_size, s) != 0) return -1;
    if (na > 1 && launch_hist_update(dy, (long long)n, yhist.in(), yhist.out(), na - 1, (int)in_size, s) != 0) return -1;
    xhist.flip();
    yhist.flip();
    consumed += n;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// ComplexMagnitude / ComplexToReal
// ---------------------------------------------------------------------------------------------
C2fBlock::C2fBlock(int op_, bool dev) {
    op = op_;
    name = op == 0 ? "cmag" : "c2r";
    in_size = 8;
    out_size = 4;
    dev_ptrs = dev;
}
int C2fBlock::run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
    *n_out = n;
    consumed += n;
    return op == 0 ? launch_cmag((const float2*)dx, (float*)dy, (long long)n, s)
                   : launch_c2r((const float2*)dx, (float*)dy, (long long)n, s);
}

}  // namespace lrb

// =============================================================================================
// extern "C" surface
// =============================================================================================
using namespace lrb;

lrb200_block_t* lrb::wrap(Block* b) {
    if (!b) return nullptr;
    lrb200_block_t* h = new (std::nothrow) lrb200_block_s{b};
    if (!h) { delete b; set_error("out of memory"); }
    return h;
}

extern "C" {

int lrb200_init(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        set_error("no CUDA device available (%s); libluaradio_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return -1;
    }
    if (device < 0 || device >= count) { set_error("device %d out of range (0..%d)", device, count - 1); return -1; }
    LRB_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    LRB_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return -1;
    }
    if (g_ctx.device != device) {
        // switching devices: the library stream, the side stream and its events belong to the old device.  Handles
        // created on the old device keep their buffers there and must not be used while another device is current.
        if (g_ctx.own_stream && g_ctx.stream) cudaStreamDestroy(g_ctx.stream);
        g_ctx.stream = nullptr;
        g_ctx.own_stream = false;
        if (g_ctx.side) cudaStreamDestroy(g_ctx.side);
        if (g_ctx.ev_fork) cudaEventDestroy(g_ctx.ev_fork);
        if (g_ctx.ev_join) cudaEventDestroy(g_ctx.ev_join);
        g_ctx.side = nullptr;
        g_ctx.ev_fork = g_ctx.ev_join = nullptr;
    }
    g_ctx.device = device;
    g_ctx.sm_count = prop.multiProcessorCount;
    if (!g_ctx.stream) {
        LRB_CHECK(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
        g_ctx.own_stream = true;
    }
    return 0;
}

int lrb200_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
    return count;
}

int lrb200_current_device(void) { return g_ctx.device; }

const char* lrb200_last_error(void) { return g_err; }
const char* lrb200_version(void) { return "luaradio_b200 0.1.0 (sm_100a)"; }

int lrb200_set_stream(void* cuda_stream) {
    if (ensure_init() != 0) return -1;
    if (g_ctx.own_stream && g_ctx.stream) cudaStreamDestroy(g_ctx.stream);
    g_ctx.own_stream = false;
    g_ctx.stream = (cudaStream_t)cuda_stream;
    if (!cuda_stream) {
        LRB_CHECK(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
        g_ctx.own_stream = true;
    }
    return 0;
}
void* lrb200_get_stream(void) { return (void*)g_ctx.stream; }

int lrb200_sync(void) {
    if (ensure_init() != 0) return -1;
    LRB_CHECK(cudaStreamSynchronize(g_ctx.stream));
    return 0;
}

uint64_t lrb200_launch_count(void) { return g_ctx.launches.load(); }

void* lrb200_malloc(size_t bytes) {
    if (ensure_init() != 0) return nullptr;
    void* p = nullptr;
    if (!cuda_ok(cudaMalloc(&p, bytes ? bytes : 1), "cudaMalloc")) return nullptr;
    return p;
}
void lrb200_free(void* p) { if (p) cudaFree(p); }
void* lrb200_host_alloc(size_t bytes) {
    if (ensure_init() != 0) return nullptr;
    void* p = nullptr;
    if (!cuda_ok(cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault), "cudaHostAlloc")) return nullptr;
    return p;
}
void lrb200_host_free(void* p) { if (p) cudaFreeHost(p); }
int lrb200_memcpy_h2d(void* dst, const void* src, size_t bytes) {
    if (ensure_init() != 0) return -1;
    LRB_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream));
    return 0;
}
int lrb200_memcpy_d2h(void* dst, const void* src, size_t bytes) {
    if (ensure_init() != 0) return -1;
    LRB_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_ctx.stream));
    return 0;
}
// ---- peer access for time-chunk sharding with one process per GPU: the left neighbour's tail is copied by the copy
// engine over NVLink (no SM, no collective kernel competing with the persistent compute kernels)
int lrb200_ipc_export(void* dptr, void* handle_out64) {
    if (ensure_init() != 0) return -1;
    if (!dptr || !handle_out64) { set_error("ipc_export: null pointer"); return -1; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    LRB_CHECK(cudaIpcGetMemHandle(&h, dptr));
    memcpy(handle_out64, &h, sizeof(h));
    return 0;
}
void* lrb200_ipc_import(const void* handle64) {
    if (ensure_init() != 0) return nullptr;
    if (!handle64) { set_error("ipc_import: null handle"); return nullptr; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    void* p = nullptr;
    if (!cuda_ok(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle")) return nullptr;
    return p;
}
int lrb200_ipc_close(void* imported) {
    if (!imported) return 0;
    LRB_CHECK(cudaIpcCloseMemHandle(imported));
    return 0;
}
int lrb200_memcpy_d2d(void* dst, const void* src, size_t bytes, void* cuda_stream) {
    if (ensure_init() != 0) return -1;
    LRB_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, cuda_stream ? (cudaStream_t)cuda_stream : g_ctx.stream));
    return 0;
}
int lrb200_memset(void* p, int value, size_t bytes) {
    if (ensure_init() != 0) return -1;
    LRB_CHECK(cudaMemsetAsync(p, value, bytes, g_ctx.stream));
    return 0;
}

// ---- generic block ---------------------------------------------------------------------------
int lrb200_block_execute(lrb200_block_t* q, const void* x, size_t n, void* y, size_t* n_out) {
    if (!q || !q->impl) { set_error("null block handle"); return -1; }
    if (n > 0 && (!x || !y)) { set_error("%s: null sample buffer", q->impl->name); return -1; }
    return q->impl->execute(x, n, y, n_out);
}
int lrb200_block_execute_multi(lrb200_block_t* q, const void* const* x, unsigned num_inputs, size_t n, void* const* y,
                               unsigned num_outputs, size_t* n_out) {
    if (!q || !q->impl) { set_error("null block handle"); return -1; }
    if (!x || !y) { set_error("%s: null port array", q->impl->name); return -1; }
    for (unsigned i = 0; i < num_inputs; ++i) if (n > 0 && !x[i]) { set_error("%s: null sample buffer", q->impl->name); return -1; }
    for (unsigned i = 0; i < num_outputs; ++i) if (n > 0 && !y[i]) { set_error("%s: null sample buffer", q->impl->name); return -1; }
    return q->impl->execute_multi(x, (int)num_inputs, n, y, (int)num_outputs, n_out);
}
unsigned lrb200_block_num_inputs(const lrb200_block_t* q) { return q && q->impl ? (unsigned)q->impl->num_inputs : 0; }
unsigned lrb200_block_num_outputs(const lrb200_block_t* q) { return q && q->impl ? (unsigned)q->impl->num_outputs : 0; }
size_t lrb200_block_max_output(const lrb200_block_t* q, size_t n) { return q && q->impl ? q->impl->max_output(n) : 0; }
size_t lrb200_block_in_size(const lrb200_block_t* q) { return q && q->impl ? q->impl->in_size : 0; }
size_t lrb200_block_out_size(const lrb200_block_t* q) { return q && q->impl ? q->impl->out_size : 0; }
int lrb200_block_reset(lrb200_block_t* q) {
    if (!q || !q->impl) { set_error("null block handle"); return -1; }
    return q->impl->reset();
}
int lrb200_block_seek(lrb200_block_t* q, uint64_t idx) {
    if (!q || !q->impl) { set_error("null block handle"); return -1; }
    return q->impl->seek(idx);
}
void lrb200_block_destroy(lrb200_block_t* q) {
    if (!q) return;
    delete q->impl;
    delete q;
}
const char* lrb200_block_name(const lrb200_block_t* q) { return q && q->impl ? q->impl->name : ""; }

// ---- FIR ---------------------------------------------------------------------------------------
static lrb200_block_t* fir_create(FirKind k, const void* taps, unsigned ntaps, unsigned decim, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (!taps || ntaps == 0) { set_error("fir: taps must be non-empty"); return nullptr; }
    if (decim == 0) { set_error("fir: decimation must be >= 1"); return nullptr; }
    if (k == FIR_HILBERT && (ntaps % 2) == 0) { set_error("hilbert: number of taps must be odd"); return nullptr; }
    return wrap(make_block<FirBlock>(k, taps, ntaps, decim, (flags & LRB200_DEVICE) != 0));
}
lrb200_fir_t* lrb200_fir_create_crcf(const float32_t* taps, unsigned ntaps, unsigned decim, unsigned flags) { return fir_create(FIR_CRCF, taps, ntaps, decim, flags); }
lrb200_fir_t* lrb200_fir_create_cccf(const complex_float32_t* taps, unsigned ntaps, unsigned decim, unsigned flags) { return fir_create(FIR_CCCF, taps, ntaps, decim, flags); }
lrb200_fir_t* lrb200_fir_create_rrrf(const float32_t* taps, unsigned ntaps, unsigned decim, unsigned flags) { return fir_create(FIR_RRRF, taps, ntaps, decim, flags); }
int lrb200_fir_execute(lrb200_fir_t* q, const void* x, size_t n, void* y, size_t* n_out) { return lrb200_block_execute(q, x, n, y, n_out); }
int lrb200_fir_reset(lrb200_fir_t* q) { return lrb200_block_reset(q); }
void lrb200_fir_destroy(lrb200_fir_t* q) { lrb200_block_destroy(q); }
int lrb200_fir_set_algorithm(lrb200_fir_t* q, int algo) {
    FirBlock* f = q && q->impl ? dynamic_cast<FirBlock*>(q->impl) : nullptr;
    if (!f) { set_error("not a FIR handle"); return -1; }
    return f->set_algorithm(algo);
}
int lrb200_fir_get_algorithm(const lrb200_fir_t* q) {
    FirBlock* f = q && q->impl ? dynamic_cast<FirBlock*>(q->impl) : nullptr;
    if (!f) { set_error("not a FIR handle"); return -1; }
    return f->effective_algorithm();
}

lrb200_hilbert_t* lrb200_hilbert_create(const float32_t* taps, unsigned ntaps, unsigned flags) { return fir_create(FIR_HILBERT, taps, ntaps, 1, flags); }

lrb200_rotator_t* lrb200_rotator_create(double turns_per_sample, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (!std::isfinite(turns_per_sample)) { set_error("rotator: turns_per_sample is not finite"); return nullptr; }
    return wrap(make_block<RotatorBlock>(turns_per_sample, (flags & LRB200_DEVICE) != 0));
}

lrb200_discrim_t* lrb200_discrim_create(float gain, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (!(gain != 0.0f) || !std::isfinite(gain)) { set_error("discrim: gain must be finite and non-zero"); return nullptr; }
    return wrap(make_block<DiscrimBlock>(gain, (flags & LRB200_DEVICE) != 0));
}

lrb200_downsample_t* lrb200_downsample_create(unsigned factor, unsigned elem_size, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (factor == 0) { set_error("downsample: factor must be >= 1"); return nullptr; }
    if (elem_size != 4 && elem_size != 8) { set_error("downsample: elem_size must be 4 or 8"); return nullptr; }
    return wrap(make_block<DownsampleBlock>(factor, elem_size, (flags & LRB200_DEVICE) != 0));
}

static lrb200_block_t* iir_create(bool cplx, const float32_t* b, unsigned nb, const float32_t* a, unsigned na, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (!b || nb == 0 || !a || na == 0) { set_error("iir: b and a taps must be non-empty"); return nullptr; }
    if (nb > 10 || na > 10) { set_error("iir: at most 10 feed-forward and 10 feedback taps"); return nullptr; }
    if (a[0].value == 0.0f) { set_error("iir: a[0] must be non-zero"); return nullptr; }
    if (na > 2 || nb > 9)
        return wrap(make_block<IirGeneralBlock>(cplx, (const float*)b, nb, (const float*)a, na, (flags & LRB200_DEVICE) != 0));
    return wrap(make_block<IirBlock>(cplx, (const float*)b, nb, (const float*)a, na, (flags & LRB200_DEVICE) != 0));
}
lrb200_iir_t* lrb200_iir_create_rrrf(const float32_t* b, unsigned nb, const float32_t* a, unsigned na, unsigned flags) { return iir_create(false, b, nb, a, na, flags); }
lrb200_iir_t* lrb200_iir_create_crcf(const float32_t* b, unsigned nb, const float32_t* a, unsigned na, unsigned flags) { return iir_create(true, b, nb, a, na, flags); }

lrb200_block_t* lrb200_cmag_create(unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_block<C2fBlock>(0, (flags & LRB200_DEVICE) != 0));
}
lrb200_block_t* lrb200_c2r_create(unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_block<C2fBlock>(1, (flags & LRB200_DEVICE) != 0));
}

lrb200_block_t* lrb200_mulconst_create(float re, float im, unsigned complex_data, unsigned complex_constant, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (complex_constant && !complex_data) { set_error("mulconst: a complex constant needs complex data"); return nullptr; }
    return wrap(make_block<ScaleBlock>(re, im, complex_data != 0, complex_constant != 0, (flags & LRB200_DEVICE) != 0));
}
lrb200_block_t* lrb200_upsample_create(unsigned factor, unsigned elem_size, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    if (factor == 0) { set_error("upsample: factor must be >= 1"); return nullptr; }
    if (elem_size != 4 && elem_size != 8) { set_error("upsample: elem_size must be 4 or 8"); return nullptr; }
    return wrap(make_block<UpsampleBlock>(factor, elem_size, (flags & LRB200_DEVICE) != 0));
}

lrb200_block_t* lrb200_iqconv_create(const char* format, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_iqconv(format, (flags & LRB200_DEVICE) != 0));
}

lrb200_block_t* lrb200_realconv_create(const char* format, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_fileconv(format, false, 1, (flags & LRB200_DEVICE) != 0));
}
lrb200_block_t* lrb200_iqsink_create(const char* format, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_fileconv(format, true, 2, (flags & LRB200_DEVICE) != 0));
}
lrb200_block_t* lrb200_realsink_create(const char* format, unsigned flags) {
    if (ensure_init() != 0) return nullptr;
    return wrap(make_fileconv(format, true, 1, (flags & LRB200_DEVICE) != 0));
}

// ---- synthetic sources -------------------------------------------------------------------------
int lrb200_synth_white_iq(complex_float32_t* dst, uint64_t n0, size_t n, uint32_t seed) {
    if (ensure_init() != 0) return -1;
    return launch_synth_white((float2*)dst, n0, (long long)n, seed, g_ctx.stream);
}
int lrb200_synth_fm_iq(complex_float32_t* dst, uint64_t n0, size_t n, uint32_t seed, double rate, double carrier,
                       double deviation, float amp, float noise) {
    if (ensure_init() != 0) return -1;
    return launch_synth_fm((float2*)dst, n0, (long long)n, seed, rate, carrier, deviation, amp, noise, g_ctx.stream);
}

}  // extern "C"
