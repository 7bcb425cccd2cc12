// Block objects behind the opaque C handles (internal).
#pragma once
#include "common.cuh"
#include <vector>
#include <string>
#include <new>
#include <utility>

namespace lrb {

// One device buffer of carried state: the part of a block's state that one call reads and writes for the next (FIR
// history, IIR state, a previous sample, a delay line).  Two slots ping-pong: a call reads in() and writes out(), then
// flip()s; one slot is read and written in place.  Block::carry allocates and zero-fills it and records it for reset().
struct Carried {
    void* slot[2] = {nullptr, nullptr};
    size_t bytes = 0;
    int idx = 0;
    Carried() = default;
    Carried(const Carried&) = delete;
    Carried& operator=(const Carried&) = delete;
    ~Carried() { cudaFree(slot[0]); cudaFree(slot[1]); }
    void* in() const { return slot[idx]; }
    void* out() const { return slot[1] ? slot[idx ^ 1] : slot[0]; }
    void flip() { idx ^= 1; }
};

struct Block {
    const char* name = "block";
    size_t in_size = 8, out_size = 8;
    bool dev_ptrs = false;
    uint64_t consumed = 0;            // global index of the next input sample

    virtual ~Block();
    virtual int init() { return 0; }
    virtual size_t max_output(size_t n) const { return n; }
    int num_inputs = 1, num_outputs = 1;
    // device pointers in/out, asynchronous on s; consumes n, produces *n_out, advances the carried state
    virtual int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) = 0;
    // blocks with several input / output ports (all inputs the same length n and element size in_size, block.lua:516-532)
    virtual int run_multi(const void* const* dx, int nin, size_t n, void* const* dy, int nout, size_t* n_out, cudaStream_t s) {
        if (nin != 1 || nout != 1) { set_error("%s has one input and one output", name); return -1; }
        return run(dx[0], n, dy[0], n_out, s);
    }
    // host pointers (staged through grow-only device buffers, like Vector:resize) or device pointers (dev_ptrs)
    int execute_multi(const void* const* x, int nin, size_t n, void* const* y, int nout, size_t* n_out);
    int execute(const void* x, size_t n, void* y, size_t* n_out) { return execute_multi(&x, 1, n, &y, 1, n_out); }
    virtual size_t out_size_of(int port) const { (void)port; return out_size; }    // element size of output port `port`
    std::vector<void*> staging;       // host mode: nin + nout device buffers
    std::vector<size_t> staging_cap;
    // reset = host-side bookkeeping + zeroing the carried state; a graph zeroes every stage's buffers with ONE
    // kernel (a 256 Mi-sample chain step is ~1 ms: a dozen cudaMemsetAsync nodes per step were 1.5 % of it)
    std::vector<Carried*> carried;    // recorded by carry()
    int carry(Carried& c, size_t bytes, int slots = 2);
    virtual void reset_host() { consumed = 0; for (Carried* c : carried) c->idx = 0; }
    void state_buffers(std::vector<std::pair<void*, size_t>>& segs) const {
        for (const Carried* c : carried)
            for (void* p : c->slot) if (p) segs.push_back({p, c->bytes});
    }
    int reset();
    virtual int seek(uint64_t idx) { consumed = idx; return 0; }
    // number of outputs this block has produced once `idx` inputs are consumed (for graph seek)
    virtual uint64_t outputs_before(uint64_t idx) const { return idx; }
    // time-chunk sharding (SURVEY.md 8e): how many INPUT samples of left context a cold start needs before this block's
    // outputs equal the streaming ones to float32 resolution (FIR history, IIR decay to 1e-12, ...); < 0 = unbounded
    virtual long long memory_in() const { return 0; }
    // output rate / input rate = up / down
    virtual void rate(unsigned* up, unsigned* down) const { *up = 1; *down = 1; }
    // sharded runs: can this block's launch keep the launches that read the first Ctx::lead_samples inputs behind
    // Ctx::lead_event while everything else starts at once?  (else the whole stream waits for the neighbour exchange)
    virtual bool supports_lead_wait() const { return false; }
    // is all carried state (history, previous output, pole state) read ONLY by launches this block puts on the side
    // stream for a long call (edge tiles, history update)?  Then a short call may run entirely on the side stream and the
    // next long call's interior kernel need not wait for it (run_shard's split of the last stage).
    virtual bool state_only_on_side_stream() const { return false; }
    static int reserve(void** p, size_t* cap, size_t bytes);
};

// Keeps the inputs at global index == 0 (mod D) (downsampler.lua:45-53 in global-index form).
struct DecimatingBlock : Block {
    int D = 1;
    struct Plan { long long first, n_out; };   // output j of the call is input first + j*D of the call
    Plan plan(size_t n) const {
        const long long f = (long long)(((uint64_t)D - consumed % (uint64_t)D) % (uint64_t)D);
        return {f, (long long)n > f ? ((long long)n - f + D - 1) / D : 0};
    }
    size_t max_output(size_t n) const override { return D == 1 ? n : n / D + 1; }
    uint64_t outputs_before(uint64_t idx) const override { return (idx + D - 1) / D; }
    void rate(unsigned* up, unsigned* down) const override { *up = 1; *down = (unsigned)D; }
};

// construct, init(), delete on failure: nullptr (with the error set) or a ready block
template <typename B, typename... A>
B* make_block(A&&... args) {
    B* b = new (std::nothrow) B(std::forward<A>(args)...);
    if (!b) { set_error("out of memory"); return nullptr; }
    if (b->init() != 0) { delete b; return nullptr; }
    return b;
}

struct FirFast;   // overlap-save plan (fir_fft.cu)
struct PolyTaps;  // polyphase decimator taps (tuner.cu)

struct FirBlock : DecimatingBlock {
    FirKind kind;
    int M = 0;
    size_t tap_size = 4;
    std::vector<char> h_taps;
    void* d_taps = nullptr;
    Carried hist;                     // last M-1 inputs
    int algo = 0;                     // LRB200_FIR_AUTO / DIRECT / FFT
    bool rotate = false;              // fused FrequencyTranslator in front (graph fusion; FFT path only)
    double rot_turns = 0.0;
    uint64_t rot_fix = 0;
    FirFast* fast = nullptr;
    PolyTaps* poly = nullptr;
    bool gen_poly = false;            // poly_generic.cu covers this (kind, M, D)
    std::string label;                // owns `name` when a graph rewrite renames the block
    // output-rate pole fused behind a real polyphase decimator (graph rewrite of FIR -> IIR1 -> Downsampler)
    bool has_pole = false;
    float pole_c = 0.f;
    Carried pole;
    int set_pole(float c);

    // rotate: fused FrequencyTranslator(turns_per_sample) in front
    FirBlock(FirKind k, const void* taps_host, unsigned ntaps, unsigned decim, bool dev, bool rotate = false,
             double turns_per_sample = 0.0);
    ~FirBlock() override;
    int init() override;
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
    long long memory_in() const override;
    bool supports_lead_wait() const override { return poly != nullptr && algo != 2 /* LRB200_FIR_FFT */ && !rotate; }
    bool state_only_on_side_stream() const override { return poly != nullptr && algo != 2 && !rotate; }
    // fast paths (fir_fft.cu): fast_run returns 1 if it handled the call, 0 to fall back, <0 on error
    int fast_init();
    void fast_free();
    int fast_run(const void* dx, size_t n, void* dy, long long first, long long n_out, cudaStream_t s);
    int set_algorithm(int a);
    int effective_algorithm() const;
};

struct RotatorBlock : Block {
    double turns = 0;
    uint64_t turns_fix = 0;
    RotatorBlock(double turns_per_sample, bool dev);
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
};

struct DiscrimBlock : Block {
    float gain = 1.f;
    Carried prev;                     // previous input sample, read and written in place
    DiscrimBlock(float gain, bool dev);
    int init() override { return carry(prev, sizeof(float2), 1); }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
    long long memory_in() const override { return 1; }
};

struct DownsampleBlock : DecimatingBlock {
    DownsampleBlock(unsigned factor, unsigned elem, bool dev);
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
};

struct IirBlock : DecimatingBlock {     // D > 1: fused Downsampler behind the filter (graph fusion)
    bool complex_data = false;
    float b[9] = {0};
    int nb = 1;
    float c = 0.f;
    Carried xhist, ystate;
    IirScanWork work;
    IirBlock(bool cplx, const float* b, unsigned nb, const float* a, unsigned na, bool dev);
    ~IirBlock() override;
    int init() override;
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
    long long memory_in() const override;
};

// IIRFilterBlock of any order (na > 2): direct form I, time-parallel chunks with a measured warm-up
struct IirGeneralBlock : Block {
    bool complex_data = false;
    float b[10] = {0}, a[10] = {0};
    int nb = 1, na = 1;
    long long warm = -1;               // samples until the impulse response of 1/A(z) is below 1e-10 of its peak
    Carried xhist, yhist;
    IirGeneralBlock(bool cplx, const float* b, unsigned nb, const float* a, unsigned na, bool dev);
    int init() override;
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
    long long memory_in() const override { return warm < 0 ? -1 : warm + nb; }
};

struct C2fBlock : Block {
    int op = 0;                       // 0 = magnitude, 1 = real part
    C2fBlock(int op, bool dev);
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
};

// resample.cu ---------------------------------------------------------------------------------
struct ScaleBlock : Block {           // MultiplyConstantBlock
    float cre, cim;
    bool complex_data, complex_const;
    ScaleBlock(float re, float im, bool cdata, bool cconst, bool dev);
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
};

struct UpsampleBlock : Block {        // UpsamplerBlock
    int L = 1;
    UpsampleBlock(unsigned factor, unsigned elem, bool dev);
    size_t max_output(size_t n) const override { return n * (size_t)L; }
    uint64_t outputs_before(uint64_t idx) const override { return idx * (uint64_t)L; }
    void rate(unsigned* up, unsigned* down) const override { *up = (unsigned)L; *down = 1; }
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
};

struct InterpFirBlock : Block {       // [MultiplyConstant ->] Upsampler -> FIR(real taps) [-> Downsampler], fused
    bool complex_data;
    int L, D, M, Hn = 0;
    bool has_scale;
    float scale;
    std::vector<float> h_taps;
    float* d_taps = nullptr;
    float* d_taps_tp = nullptr;          // [t][phase] layout for the register-tiled interpolator (D == 1, L <= 8)
    int Tt = 0;
    bool rs_ok = false;                  // the register-tiled (L, D) polyphase kernel covers this shape (resample.cu)
    Carried hist;                        // last Hn inputs
    std::string label;
    InterpFirBlock(bool cdata, const float* taps_host, int ntaps, int interp, int decim, bool has_scale, float scale, bool dev);
    ~InterpFirBlock() override;
    int init() override;
    size_t max_output(size_t n) const override;
    uint64_t outputs_before(uint64_t idx) const override;
    int run(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) override;
    long long memory_in() const override { return Hn + 1; }
    void rate(unsigned* up, unsigned* down) const override { *up = (unsigned)L; *down = (unsigned)D; }
};

}  // namespace lrb

// the opaque public handle
struct lrb200_block_s { lrb::Block* impl; };

namespace lrb {
// hands a ready block (or nullptr from make_block) to the caller as a new handle; nullptr with the error set on failure
lrb200_block_s* wrap(Block* b);
}  // namespace lrb

namespace lrb {
// tuner.cu: register-tiled polyphase decimating FIR (complex in, real taps), optional fused rotator.
// Returns 1 if the (M, D) shape is supported and the launch was enqueued, 0 if unsupported, <0 on error.
PolyTaps* polyphase_prepare(const float* taps, int M, int D, double turns_per_sample, bool phasor_table = false,
                            bool real_data = false);
void polyphase_release(PolyTaps* p);
int launch_polyphase_crcf(const PolyTaps* p, const float2* x, const float2* hist, long long n, float2* y,
                          long long first, long long n_out, bool rotate, uint64_t turns_fix, uint64_t g0,
                          cudaStream_t s);
// real input, real taps, decimating (x / hist / y are float32)
// z_in != nullptr additionally fuses the output-rate pole z[m] = pole_c z[m-1] + w[m] (state carried in z_in -> z_out)
int launch_polyphase_rrrf(const PolyTaps* p, const float* x, const float* hist, long long n, float* y,
                          long long first, long long n_out, cudaStream_t s, float pole_c = 0.f,
                          const float* z_in = nullptr, float* z_out = nullptr);
bool polyphase_pole_ok(float c);     // the pole's memory fits the kernel's warm-up
// iqconv.cu: IQFileSource sample format -> ComplexFloat32 (nullptr + error for an unknown format)
Block* make_iqconv(const char* format, bool dev);
// RealFileSource (to_file = false, comps = 1), RealFileSink/WAVFileSink (true, 1), IQFileSink (true, 2)
Block* make_fileconv(const char* format, bool to_file, int comps, bool dev);
// tuner.cu: fused FrequencyTranslator -> FIR(crcf) -> Downsampler; returns nullptr (with the error set) on failure
// disc_gain != 0 additionally fuses a FrequencyDiscriminator(gain) behind it (float output)
Block* make_tuner(double turns_per_sample, const float* taps, int ntaps, int decim, float disc_gain);
}  // namespace lrb
