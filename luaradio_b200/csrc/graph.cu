// Single-stream GPU flow graph: a connected chain of GPU blocks sharing device-resident buffers.
//
// Replaces, for a run of connected GPU blocks, the reference's fork-per-block scheduler and socketpair
// pipes (radio/core/composite.lua:568-636, radio/core/pipe.lua:53-88): intermediate sample vectors stay
// in a two-slot device ring; host<->device traffic exists only at the two ends, double-buffered on
// separate copy streams so chunk i+1 uploads while chunk i computes and chunk i-1 downloads.
// commit(fuse=1) rewrites adjacent blocks into fused kernels:
//   Rotator -> FIR(crcf) -> Downsampler [-> Discriminator]  =>  tuner kernel (composites/tuner.lua:40-47)
//   FIR -> Downsampler                    =>  decimating FIR    (composites/decimator.lua:34-41)
//   IIR -> Downsampler                    =>  scan with strided store
//   [MultiplyConstant ->] Upsampler -> FIR [-> Downsampler]  =>  polyphase interpolating FIR
#include "../../include/lrb200.h"
#include "common.cuh"
#include "blocks.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

namespace lrb {

struct Graph {
    std::vector<Block*> blocks;      // as appended (owned)
    std::vector<Block*> fused;       // blocks created by fusion (owned)
    std::vector<Block*> stages;      // execution order after commit (not owned)
    bool committed = false;
    void* ring[2] = {nullptr, nullptr};
    size_t ring_cap[2] = {0, 0};
    // host-mode double buffering
    void* d_in[2] = {nullptr, nullptr};  size_t d_in_cap[2] = {0, 0};
    void* d_out[2] = {nullptr, nullptr}; size_t d_out_cap[2] = {0, 0};
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    size_t host_chunk = (size_t)1 << 23;   // input samples per pipelined chunk
    std::string desc;
    // super-chunk mode (SURVEY.md 8e "streaming mode"): small host vectors are packed into pinned slots of `sc` samples;
    // a full slot is processed asynchronously while the next one fills, and its outputs are handed back when that next
    // slot is submitted (or at flush) -- the per-vector cost is one host memcpy instead of copies + launches + a sync
    size_t sc = 0;
    char* sc_hin[2] = {nullptr, nullptr};
    char* sc_hout[2] = {nullptr, nullptr};
    void* sc_din[2] = {nullptr, nullptr};
    void* sc_dout[2] = {nullptr, nullptr};
    cudaEvent_t sc_done[2] = {nullptr, nullptr};
    bool sc_pending[2] = {false, false};
    size_t sc_nout[2] = {0, 0};
    size_t sc_fill = 0, sc_outcap = 0;
    int sc_cur = 0;
    // time-chunk sharding (run_shard): scratch for the outputs that belong to the halo
    void* head_out = nullptr; size_t head_out_cap = 0;
    // optional per-stage timing
    bool timing = false;
    std::vector<std::vector<cudaEvent_t>> tev;   // per stage: [start0, stop0, start1, stop1, ...]
    std::vector<int> tcount;

    cudaEvent_t timing_event(size_t stage, size_t idx) {
        if (tev.size() < stages.size()) { tev.resize(stages.size()); tcount.assign(stages.size(), 0); }
        auto& v = tev[stage];
        while (v.size() <= idx) { cudaEvent_t e; cudaEventCreate(&e); v.push_back(e); }
        return v[idx];
    }

    ~Graph() {
        for (auto& v : tev) for (cudaEvent_t e : v) cudaEventDestroy(e);
        for (Block* b : blocks) delete b;
        for (Block* b : fused) delete b;
        for (int i = 0; i < 2; ++i) {
            cudaFree(ring[i]); cudaFree(d_in[i]); cudaFree(d_out[i]);
            if (ev_h2d[i]) cudaEventDestroy(ev_h2d[i]);
            if (ev_comp[i]) cudaEventDestroy(ev_comp[i]);
            if (ev_d2h[i]) cudaEventDestroy(ev_d2h[i]);
        }
        if (s_h2d) cudaStreamDestroy(s_h2d);
        if (s_d2h) cudaStreamDestroy(s_d2h);
        free_superchunk();
        cudaFree(head_out);
    }

    void free_superchunk() {
        for (int i = 0; i < 2; ++i) {
            if (sc_hin[i]) cudaFreeHost(sc_hin[i]);
            if (sc_hout[i]) cudaFreeHost(sc_hout[i]);
            cudaFree(sc_din[i]); cudaFree(sc_dout[i]);
            if (sc_done[i]) cudaEventDestroy(sc_done[i]);
            sc_hin[i] = sc_hout[i] = nullptr; sc_din[i] = sc_dout[i] = nullptr; sc_done[i] = nullptr;
            sc_pending[i] = false; sc_nout[i] = 0;
        }
        sc = 0; sc_fill = 0; sc_cur = 0;
    }

    size_t max_output(size_t n) const {
        for (Block* b : stages) n = b->max_output(n);
        return n;
    }

    int commit(int fuse) {
        stages.clear();
        for (Block* b : fused) delete b;
        fused.clear();
        desc.clear();
        size_t i = 0;
        while (i < blocks.size()) {
            Block* b = blocks[i];
            Block* st = b;
            Block* st2 = nullptr;        // a rewrite may turn a run of blocks into two stages
            size_t used = 1;
            if (fuse) {
                RotatorBlock* rot = dynamic_cast<RotatorBlock*>(b);
                FirBlock* fir = dynamic_cast<FirBlock*>(b);
                IirBlock* iir = dynamic_cast<IirBlock*>(b);
                if (rot && i + 1 < blocks.size()) {
                    FirBlock* f2 = dynamic_cast<FirBlock*>(blocks[i + 1]);
                    DownsampleBlock* d3 = (i + 2 < blocks.size()) ? dynamic_cast<DownsampleBlock*>(blocks[i + 2]) : nullptr;
                    if (d3 && d3->in_size != 8) d3 = nullptr;
                    const bool fir_ok = f2 && (f2->kind == FIR_CRCF || f2->kind == FIR_CCCF) && f2->D == 1;
                    if (fir_ok && d3 && f2->kind == FIR_CRCF) {
                        DiscrimBlock* d4 = (i + 3 < blocks.size()) ? dynamic_cast<DiscrimBlock*>(blocks[i + 3]) : nullptr;
                        Block* t = make_tuner(rot->turns, (const float*)f2->h_taps.data(), f2->M, d3->D, d4 ? d4->gain : 0.0f);
                        if (t) { fused.push_back(t); st = t; used = d4 ? 4 : 3; }
                    }
                    if (used == 1 && fir_ok && f2->M <= 513) {
                        // translator folded into the overlap-save kernel (any taps, complex taps included)
                        // (the fused translator forces the overlap-save path: algo is moot)
                        FirBlock* nf = make_block<FirBlock>(f2->kind, f2->h_taps.data(), (unsigned)f2->M, (unsigned)(d3 ? d3->D : 1), true,
                                                            true, rot->turns);
                        if (!nf) return -1;
                        nf->name = f2->kind == FIR_CCCF ? "rot+fir_cccf" : "rot+fir_crcf";
                        fused.push_back(nf); st = nf; used = d3 ? 3 : 2;
                    }
                }
                {
                    // [MultiplyConstant(real c) ->] Upsampler(L) -> FIR(real taps) [-> Downsampler(D)]  =>  polyphase
                    // interpolating FIR (composites/interpolator.lua:31-41, composites/rationalresampler.lua:33-46)
                    size_t j = i;
                    ScaleBlock* sc = dynamic_cast<ScaleBlock*>(blocks[j]);
                    if (sc && !sc->complex_const) ++j; else sc = nullptr;
                    UpsampleBlock* up = j < blocks.size() ? dynamic_cast<UpsampleBlock*>(blocks[j]) : nullptr;
                    FirBlock* f2 = (up && j + 1 < blocks.size()) ? dynamic_cast<FirBlock*>(blocks[j + 1]) : nullptr;
                    if (up && f2 && f2->D == 1 && (f2->kind == FIR_CRCF || f2->kind == FIR_RRRF) && f2->in_size == up->out_size) {
                        DownsampleBlock* d3 = (j + 2 < blocks.size()) ? dynamic_cast<DownsampleBlock*>(blocks[j + 2]) : nullptr;
                        if (d3 && d3->in_size != f2->out_size) d3 = nullptr;
                        InterpFirBlock* nb = make_block<InterpFirBlock>(f2->kind == FIR_CRCF, (const float*)f2->h_taps.data(), f2->M,
                                                                        up->L, d3 ? d3->D : 1, sc != nullptr, sc ? sc->cre : 1.0f, true);
                        if (!nb) return -1;
                        fused.push_back(nb); st = nb; used = (j - i) + 2 + (d3 ? 1 : 0);
                    }
                }
                if (used == 1 && fir && fir->D == 1 && fir->kind == FIR_RRRF && i + 2 < blocks.size()) {
                    // FIR(h) -> single-pole IIR (b, c) -> Downsampler(D), all real (the chain's audio tail,
                    // examples/rtlsdr_wbfm_mono.lua:15-18; iirfilter.lua:147-179; downsampler.lua:45-53).
                    // y[n] = c y[n-1] + v[n], v = b * u, u = h * x.  Unrolling the recurrence D times:
                    //     y[n] = c^D y[n-D] + sum_{i<D} c^i v[n-i]
                    // so the kept samples z[m] = y[mD] obey  z[m] = c^D z[m-1] + w[mD]  with  w = (h * b * [1, c, .., c^(D-1)]) * x:
                    // ONE decimating FIR with M + nb + D - 2 taps (only kept outputs computed) and a pole c^D at the
                    // output rate, instead of a full-rate FIR and a full-rate recurrence that both compute D times more
                    // samples than the Downsampler keeps.  Zero initial state on both sides, so the streams are equal
                    // from the first sample; the taps are designed in float64 from the float32 coefficients.
                    IirBlock* i2 = dynamic_cast<IirBlock*>(blocks[i + 1]);
                    DownsampleBlock* d3 = dynamic_cast<DownsampleBlock*>(blocks[i + 2]);
                    if (i2 && !i2->complex_data && i2->D == 1 && d3 && d3->in_size == 4 && d3->D > 1) {
                        const int Dd = d3->D, nbb = i2->nb;
                        std::vector<double> g((size_t)(nbb + Dd - 1), 0.0);
                        double cp = 1.0;
                        for (int k = 0; k < Dd; ++k) {
                            for (int j = 0; j < nbb; ++j) g[(size_t)(k + j)] += cp * (double)i2->b[j];
                            cp *= (double)i2->c;
                        }
                        const float* h = (const float*)fir->h_taps.data();
                        const int Mc = fir->M + (int)g.size() - 1;
                        std::vector<float> hc((size_t)Mc);
                        for (int t = 0; t < Mc; ++t) {
                            double acc = 0.0;
                            for (int k = 0; k < (int)g.size(); ++k)
                                if (t - k >= 0 && t - k < fir->M) acc += g[(size_t)k] * (double)h[t - k];
                            hc[(size_t)t] = (float)acc;
                        }
                        FirBlock* nf = make_block<FirBlock>(FIR_RRRF, hc.data(), (unsigned)Mc, (unsigned)Dd, true);
                        if (!nf) return -1;
                        nf->set_algorithm(fir->algo);
                        if (nf->poly && nf->algo != LRB200_FIR_FFT && polyphase_pole_ok((float)cp)) {
                            // the pole's memory (|c^D|^64 <= 1e-8) fits the kernel's own warm-up: ONE stage
                            if (nf->set_pole((float)cp) != 0) { delete nf; return -1; }
                            nf->label = "fir*iir1_rrrf(" + std::to_string(Mc) + ",/" + std::to_string(Dd) + ")+pole";
                            nf->name = nf->label.c_str();
                            fused.push_back(nf);
                            st = nf; used = 3;
                        } else if (nf->poly) {      // only worth it when the polyphase kernel has this shape
                            const float one = 1.0f, a2[2] = {1.0f, (float)(-cp)};     // cp == c^D
                            IirBlock* ni = make_block<IirBlock>(false, &one, 1, a2, 2, true);
                            if (!ni) { delete nf; return -1; }
                            nf->label = "fir*iir1_rrrf(" + std::to_string(Mc) + ",/" + std::to_string(Dd) + ")";
                            nf->name = nf->label.c_str();
                            ni->name = "pole_rrrf";
                            fused.push_back(nf); fused.push_back(ni);
                            st = nf; st2 = ni; used = 3;
                        } else {
                            delete nf;
                        }
                    }
                }
                if (used == 1 && fir && fir->D == 1 && fir->kind != FIR_HILBERT && i + 1 < blocks.size()) {
                    DownsampleBlock* d2 = dynamic_cast<DownsampleBlock*>(blocks[i + 1]);
                    if (d2 && d2->in_size == fir->out_size) {
                        FirBlock* nf = make_block<FirBlock>(fir->kind, fir->h_taps.data(), (unsigned)fir->M, (unsigned)d2->D, true);
                        if (!nf) return -1;
                        nf->set_algorithm(fir->algo);      // FIRFilterBlock(taps, use_fft) survives the fusion
                        fused.push_back(nf); st = nf; used = 2;
                    }
                }
                if (used == 1 && iir && iir->D == 1 && i + 1 < blocks.size()) {
                    DownsampleBlock* d2 = dynamic_cast<DownsampleBlock*>(blocks[i + 1]);
                    if (d2 && d2->in_size == iir->out_size) {
                        float a[2] = {1.0f, -iir->c};
                        IirBlock* ni = make_block<IirBlock>(iir->complex_data, iir->b, (unsigned)iir->nb, a, 2, true);
                        if (!ni) return -1;
                        ni->D = d2->D;
                        fused.push_back(ni); st = ni; used = 2;
                    }
                }
            }
            stages.push_back(st);
            if (!desc.empty()) desc += " | ";
            desc += st->name;
            if (used > 1) { desc += "[fused x"; desc += std::to_string(used); desc += "]"; }
            if (st2) { stages.push_back(st2); desc += " | "; desc += st2->name; }
            i += used;
        }
        for (size_t k = 0; k + 1 < stages.size(); ++k) {
            if (stages[k]->out_size != stages[k + 1]->in_size) {
                set_error("graph: %s (out %zu B) cannot feed %s (in %zu B)", stages[k]->name, stages[k]->out_size,
                          stages[k + 1]->name, stages[k + 1]->in_size);
                return -1;
            }
        }
        committed = true;
        return 0;
    }

    // device in/out, asynchronous on s
    int run_device(const void* dx, size_t n, void* dy, size_t* n_out, cudaStream_t s) {
        if (!committed && commit(1) != 0) return -1;
        if (stages.empty()) { set_error("graph: no blocks"); return -1; }
        // size the ring for this n
        size_t m = n;
        for (size_t k = 0; k + 1 < stages.size(); ++k) {
            m = stages[k]->max_output(m);
            size_t bytes = (m ? m : 1) * stages[k]->out_size;
            int slot = (int)(k & 1);
            if (bytes > ring_cap[slot]) {
                // a stage still in flight may be reading the old buffer
                LRB_CHECK(cudaStreamSynchronize(s));
                if (Block::reserve(&ring[slot], &ring_cap[slot], bytes) != 0) return -1;
            }
        }
        const void* in = dx;
        size_t cnt = n;
        for (size_t k = 0; k < stages.size(); ++k) {
            void* out = (k + 1 == stages.size()) ? dy : ring[k & 1];
            size_t no = 0;
            if (timing) {
                if (tcount.size() < stages.size()) { tev.resize(stages.size()); tcount.assign(stages.size(), 0); }
                cudaEventRecord(timing_event(k, 2 * (size_t)tcount[k]), s);
            }
            if (stages[k]->run(in, cnt, out, &no, s) != 0) return -1;
            if (timing) { cudaEventRecord(timing_event(k, 2 * (size_t)tcount[k] + 1), s); tcount[k]++; }
            in = out;
            cnt = no;
        }
        *n_out = cnt;
        return 0;
    }

    int ensure_host_pipeline() {
        if (s_h2d) return 0;
        LRB_CHECK(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
        LRB_CHECK(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            LRB_CHECK(cudaEventCreateWithFlags(&ev_h2d[i], cudaEventDisableTiming));
            LRB_CHECK(cudaEventCreateWithFlags(&ev_comp[i], cudaEventDisableTiming));
            LRB_CHECK(cudaEventCreateWithFlags(&ev_d2h[i], cudaEventDisableTiming));
        }
        return 0;
    }

    // host in/out: pipelined H2D | kernels | D2H over two slots
    int run_host(const void* x, size_t n, void* y, size_t* n_out) {
        if (!committed && commit(1) != 0) return -1;
        if (stages.empty()) { set_error("graph: no blocks"); return -1; }
        cudaStream_t s = ctx().stream;
        const size_t isz = stages.front()->in_size, osz = stages.back()->out_size;
        if (sc) return run_accumulate(x, n, y, n_out);
        if (n <= host_chunk) {
            // one chunk (every call of the reference's per-vector regime, pipe.lua:73): copy, kernels and copy back in
            // order on ONE stream with ONE synchronize -- no cross-stream events, nothing to overlap anyway
            const size_t mo = max_output(n);
            if (n * isz > d_in_cap[0] || (mo ? mo : 1) * osz > d_out_cap[0]) {
                LRB_CHECK(cudaStreamSynchronize(s));
                if (Block::reserve(&d_in[0], &d_in_cap[0], (n ? n : 1) * isz) != 0) return -1;
                if (Block::reserve(&d_out[0], &d_out_cap[0], (mo ? mo : 1) * osz) != 0) return -1;
            }
            size_t no = 0;
            if (n) LRB_CHECK(cudaMemcpyAsync(d_in[0], x, n * isz, cudaMemcpyHostToDevice, s));
            if (run_device(d_in[0], n, d_out[0], &no, s) != 0) return -1;
            if (no) LRB_CHECK(cudaMemcpyAsync(y, d_out[0], no * osz, cudaMemcpyDeviceToHost, s));
            LRB_CHECK(cudaStreamSynchronize(s));
            *n_out = no;
            return 0;
        }
        if (ensure_host_pipeline() != 0) return -1;
        size_t done = 0, produced = 0;
        int it = 0;
        while (done < n) {
            const int slot = it & 1;
            size_t nc = n - done < host_chunk ? n - done : host_chunk;
            size_t mo = max_output(nc);
            if (nc * isz > d_in_cap[slot] || (mo ? mo : 1) * osz > d_out_cap[slot]) {
                LRB_CHECK(cudaDeviceSynchronize());
                if (Block::reserve(&d_in[slot], &d_in_cap[slot], nc * isz) != 0) return -1;
                if (Block::reserve(&d_out[slot], &d_out_cap[slot], (mo ? mo : 1) * osz) != 0) return -1;
            }
            if (it >= 2) LRB_CHECK(cudaStreamWaitEvent(s_h2d, ev_comp[slot], 0));     // d_in[slot] free again
            LRB_CHECK(cudaMemcpyAsync(d_in[slot], (const char*)x + done * isz, nc * isz, cudaMemcpyHostToDevice, s_h2d));
            LRB_CHECK(cudaEventRecord(ev_h2d[slot], s_h2d));
            LRB_CHECK(cudaStreamWaitEvent(s, ev_h2d[slot], 0));
            if (it >= 2) LRB_CHECK(cudaStreamWaitEvent(s, ev_d2h[slot], 0));          // d_out[slot] drained
            size_t no = 0;
            if (run_device(d_in[slot], nc, d_out[slot], &no, s) != 0) return -1;
            LRB_CHECK(cudaEventRecord(ev_comp[slot], s));
            LRB_CHECK(cudaStreamWaitEvent(s_d2h, ev_comp[slot], 0));
            if (no) LRB_CHECK(cudaMemcpyAsync((char*)y + produced * osz, d_out[slot], no * osz, cudaMemcpyDeviceToHost, s_d2h));
            LRB_CHECK(cudaEventRecord(ev_d2h[slot], s_d2h));
            produced += no;
            done += nc;
            ++it;
        }
        // the last download is behind every upload and every kernel (event chain), so one synchronize drains all three
        LRB_CHECK(cudaStreamSynchronize(s_d2h));
        LRB_CHECK(cudaStreamSynchronize(s));     // (returns at once; keeps the compute stream's error state observable)
        *n_out = produced;
        return 0;
    }

    // ---- super-chunk mode -------------------------------------------------------------------------------------
    int set_superchunk(size_t samples) {
        if (!committed && commit(1) != 0) return -1;
        if (stages.empty()) { set_error("graph: no blocks"); return -1; }
        if (sc_pending[0] || sc_pending[1] || sc_fill) { set_error("graph: flush before changing the super-chunk size"); return -1; }
        free_superchunk();
        if (samples == 0) return 0;
        const size_t isz = stages.front()->in_size, osz = stages.back()->out_size;
        sc_outcap = max_output(samples) + 1;
        for (int i = 0; i < 2; ++i) {
            LRB_CHECK(cudaHostAlloc((void**)&sc_hin[i], samples * isz, cudaHostAllocDefault));
            LRB_CHECK(cudaHostAlloc((void**)&sc_hout[i], sc_outcap * osz, cudaHostAllocDefault));
            LRB_CHECK(cudaMalloc(&sc_din[i], samples * isz));
            LRB_CHECK(cudaMalloc(&sc_dout[i], sc_outcap * osz));
            LRB_CHECK(cudaEventCreateWithFlags(&sc_done[i], cudaEventDisableTiming));
        }
        sc = samples;
        return 0;
    }
    size_t sc_collect(int slot, char* y) {
        if (!sc_pending[slot]) return 0;
        if (!cuda_ok(cudaEventSynchronize(sc_done[slot]), "cudaEventSynchronize")) return (size_t)-1;
        const size_t osz = stages.back()->out_size;
        if (sc_nout[slot]) memcpy(y, sc_hout[slot], sc_nout[slot] * osz);
        sc_pending[slot] = false;
        return sc_nout[slot];
    }
    int sc_submit(int slot, size_t count) {
        cudaStream_t s = ctx().stream;
        const size_t isz = stages.front()->in_size, osz = stages.back()->out_size;
        size_t no = 0;
        LRB_CHECK(cudaMemcpyAsync(sc_din[slot], sc_hin[slot], count * isz, cudaMemcpyHostToDevice, s));
        if (run_device(sc_din[slot], count, sc_dout[slot], &no, s) != 0) return -1;
        if (no) LRB_CHECK(cudaMemcpyAsync(sc_hout[slot], sc_dout[slot], no * osz, cudaMemcpyDeviceToHost, s));
        LRB_CHECK(cudaEventRecord(sc_done[slot], s));
        sc_nout[slot] = no;
        sc_pending[slot] = true;
        return 0;
    }
    int run_accumulate(const void* x, size_t n, void* y, size_t* n_out) {
        const size_t isz = stages.front()->in_size, osz = stages.back()->out_size;
        const char* xp = (const char*)x;
        char* yp = (char*)y;
        size_t produced = 0;
        while (n > 0) {
            const size_t take = n < sc - sc_fill ? n : sc - sc_fill;
            memcpy(sc_hin[sc_cur] + sc_fill * isz, xp, take * isz);
            sc_fill += take; xp += take * isz; n -= take;
            if (sc_fill == sc) {
                // the other slot was submitted one super-chunk ago: its results are (long) ready
                const size_t got = sc_collect(sc_cur ^ 1, yp + produced * osz);
                if (got == (size_t)-1) return -1;
                produced += got;
                if (sc_submit(sc_cur, sc) != 0) return -1;
                sc_cur ^= 1;
                sc_fill = 0;
            }
        }
        *n_out = produced;
        return 0;
    }
    int flush(void* y, size_t* n_out) {
        *n_out = 0;
        if (!sc) return 0;
        const size_t osz = stages.back()->out_size;
        char* yp = (char*)y;
        size_t produced = 0;
        size_t got = sc_collect(sc_cur ^ 1, yp);
        if (got == (size_t)-1) return -1;
        produced += got;
        if (sc_fill) {
            if (sc_submit(sc_cur, sc_fill) != 0) return -1;
            got = sc_collect(sc_cur, yp + produced * osz);
            if (got == (size_t)-1) return -1;
            produced += got;
            sc_fill = 0;
        }
        *n_out = produced;
        return 0;
    }

    int reset(cudaStream_t s) {
        std::vector<std::pair<void*, size_t>> segs;
        for (Block* b : blocks) { b->reset_host(); b->state_buffers(segs); }
        for (Block* b : fused) { b->reset_host(); b->state_buffers(segs); }
        if (segs.empty()) return 0;
        std::vector<void*> ptrs;
        std::vector<size_t> bytes;
        for (auto& sg : segs) { ptrs.push_back(sg.first); bytes.push_back(sg.second); }
        return launch_zero_segments(ptrs.data(), bytes.data(), (int)ptrs.size(), s);
    }
    int reset() { return reset(ctx().stream); }

    // ---- time-chunk sharding (SURVEY.md 8e) -------------------------------------------------------------------
    // total rate change in lowest terms: outputs per input = up / down
    void total_rate(unsigned long long* up, unsigned long long* down) const {
        unsigned long long u = 1, d = 1;
        for (Block* b : stages) {
            unsigned bu, bd;
            b->rate(&bu, &bd);
            u *= bu; d *= bd;
            unsigned long long a = u, c = d;
            while (c) { unsigned long long t = a % c; a = c; c = t; }
            u /= a; d /= a;
        }
        *up = u; *down = d;
    }
    // input samples of left context a cold start needs so that the outputs equal the streaming ones to float32
    // resolution, rounded up to a whole number of output periods; < 0 when a stage's memory is unbounded
    long long halo() {
        if (!committed && commit(1) != 0) return -1;
        double need = 0.0;                                   // at the input rate of the stage being visited
        for (size_t k = stages.size(); k-- > 0;) {
            unsigned bu, bd;
            stages[k]->rate(&bu, &bd);
            const long long mem = stages[k]->memory_in();
            if (mem < 0) { set_error("graph: %s has unbounded memory, the stream cannot be cut", stages[k]->name); return -1; }
            need = std::ceil(need * (double)bd / (double)bu) + (double)mem + 1.0;
        }
        unsigned long long up, down;
        total_rate(&up, &down);
        // whole output periods, and a multiple of 4 samples so that a chunk placed `halo` samples into a 16-byte aligned
        // buffer stays 16-byte aligned (float32 and complex streams alike): the vectorised interior kernels need that
        const long long q = 4 * (long long)down;
        long long h = (long long)need;
        h = ((h + q - 1) / q) * q;
        return h;
    }

    // One time chunk of a sharded stream.  dx -> [halo samples of the left neighbour | n samples of this chunk], the chunk
    // starting at global input index `start` (a multiple of the output period, like halo).  The stream is run COLD from
    // start - halo over halo + n samples -- every stage's memory has died out by `start` (halo()) -- and the halo's outputs
    // are dropped.  Only what reads the neighbour's samples waits for `halo_ready`: the first stage keeps the few tiles
    // that touch dx[0, halo) out of its interior kernel and runs them as edge tiles on the side stream behind the event
    // (Ctx::lead_samples / lead_event); everything else starts at once, so the exchange overlaps the chunk's kernels.
    // A first stage that cannot do that makes the compute stream wait for the event (the exchange is then serial).
    // The last stage runs as two streaming calls -- the inputs that belong to the halo (their outputs go to a scratch
    // buffer), then the rest straight into dy -- so dy receives exactly the chunk's outputs.  `head` is unused (kept in
    // the C ABI for callers that built a second graph for the former head-piece scheme).
    int run_shard(Graph& head, const void* dx, size_t halo_n, size_t n, uint64_t start, void* dy, size_t* n_out, cudaEvent_t halo_ready) {
        (void)head;
        if (!committed && commit(1) != 0) return -1;
        if (stages.empty()) { set_error("graph: no blocks"); return -1; }
        cudaStream_t s = ctx().stream;
        const size_t isz = stages.front()->in_size, osz = stages.back()->out_size;
        unsigned long long up, down;
        total_rate(&up, &down);
        if (halo_n % down || start % down) { set_error("graph: halo and start must be multiples of %llu input samples", down); return -1; }
        if (halo_n == 0 || start == 0) {                     // the stream's first chunk: nothing to its left
            if (reset(s) != 0 || seek(start) != 0) return -1;
            return run_device((const char*)dx + halo_n * isz, n, dy, n_out, s);
        }
        if (start < halo_n) { set_error("graph: chunk starts inside the halo"); return -1; }
        if (reset(s) != 0 || seek(start - halo_n) != 0) return -1;
        const size_t K = stages.size();
        // inputs of every stage that belong to the halo: lead[k] = (stage-k input index of `start`) - (that of start - halo)
        std::vector<size_t> lead(K + 1);
        {
            uint64_t a = start - halo_n, b = start;
            for (size_t k = 0; k < K; ++k) {
                lead[k] = (size_t)(b - a);
                a = stages[k]->outputs_before(a);
                b = stages[k]->outputs_before(b);
            }
            lead[K] = (size_t)(b - a);                       // outputs of the halo: dropped
        }
        const size_t ho = lead[K];
        if ((ho + 1) * osz > head_out_cap) {
            LRB_CHECK(cudaStreamSynchronize(s));
            if (Block::reserve(&head_out, &head_out_cap, (ho + 1) * osz) != 0) return -1;
        }
        // ring for halo + n inputs
        const size_t n_tot = halo_n + n;
        size_t m = n_tot;
        for (size_t k = 0; k + 1 < K; ++k) {
            m = stages[k]->max_output(m);
            const size_t bytes = (m ? m : 1) * stages[k]->out_size;
            const int slot = (int)(k & 1);
            if (bytes > ring_cap[slot]) {
                LRB_CHECK(cudaStreamSynchronize(s));
                if (Block::reserve(&ring[slot], &ring_cap[slot], bytes) != 0) return -1;
            }
        }
        const bool overlap = halo_ready && K >= 2 && stages[0]->supports_lead_wait();
        if (halo_ready && !overlap) LRB_CHECK(cudaStreamWaitEvent(s, halo_ready, 0));
        const void* in = dx;
        size_t cnt = n_tot;
        int rc = 0;
        for (size_t k = 0; k < K && rc == 0; ++k) {
            const bool last = k + 1 == K;
            if (timing) {
                if (tcount.size() < K) { tev.resize(K); tcount.assign(K, 0); }
                cudaEventRecord(timing_event(k, 2 * (size_t)tcount[k]), s);
            }
            if (k == 0 && overlap) { ctx().lead_samples = (long long)halo_n; ctx().lead_event = halo_ready; ctx().reserve_ctas = 4; }
            size_t no = 0;
            if (!last) {
                void* out = ring[k & 1];
                rc = stages[k]->run(in, cnt, out, &no, s);
                in = out;
                cnt = no;
            } else {
                // two streaming calls: the halo's share of the inputs -> scratch, the chunk's -> dy
                // (the short first call goes to the side stream when the stage keeps every state access there: the second
                // call's interior kernel then starts without waiting for the first call's latency-bound edge kernel)
                size_t no1 = 0;
                const size_t m1 = lead[k] < cnt ? lead[k] : cnt;
                cudaStream_t s1 = (stages[k]->state_only_on_side_stream() && cnt - m1 >= SIDE_STREAM_MIN) ? side_fork(s) : s;
                rc = stages[k]->run(in, m1, head_out, &no1, s1);
                if (rc == 0 && no1 != ho) { set_error("graph: halo produced %zu outputs, expected %zu", no1, ho); rc = -1; }
                if (rc == 0) rc = stages[k]->run((const char*)in + m1 * stages[k]->in_size, cnt - m1, dy, &no, s);
                side_join(s, s1);
                cnt = no;
            }
            if (k == 0) { ctx().lead_samples = 0; ctx().lead_event = nullptr; ctx().reserve_ctas = 0; }
            if (timing) { cudaEventRecord(timing_event(k, 2 * (size_t)tcount[k] + 1), s); tcount[k]++; }
        }
        if (rc != 0) return -1;
        *n_out = cnt;
        return 0;
    }

    int seek(uint64_t idx) {
        if (!committed && commit(1) != 0) return -1;
        for (Block* b : stages) {
            if (b->seek(idx) != 0) return -1;
            idx = b->outputs_before(idx);
        }
        return 0;
    }
};

// ---------------------------------------------------------------------------------------------------------------------
// Device DAG: fan-out / fan-in between GPU nodes without host hops.  A node is a multi-port block (MultiplyConjugate, Add,
// Subtract, PLL, ...), a single block, or a committed LINEAR flow graph (so the fused kernels keep doing the work inside
// every linear run).  Nodes are added in topological order; an input reference is (producer node, output port) or the
// DAG's own input.  Every edge is a grow-only device buffer; all inputs of a node must deliver the same number of samples
// per call (true whenever the converging paths have the same rate changes -- every block here is zero-latency; the
// reference's PipeMux would buffer a surplus instead, radio/core/pipe.lua:495-615).  Host in, host out(s): one upload,
// the node launches in order on the library stream, one download per output, one synchronize.
// This is what composites/wbfmstereodemodulator.lua:22-64 and amsynchronousdemodulator.lua:25-45 need on the device.
// ---------------------------------------------------------------------------------------------------------------------
void destroy_graph_handle(void* holder);      // delete (lrb200_graph_t*) -- defined behind the handle type below

struct DagNode {
    Block* blk = nullptr;          // owned
    Graph* sub = nullptr;          // a committed linear run: lives inside `holder` (the caller's former handle, owned)
    void* holder = nullptr;
    std::vector<int> in_refs;      // producer node * 4 + port, or -1 for the DAG input
    std::vector<void*> out_buf;
    std::vector<size_t> out_cap, out_cnt;
    int nout() const { return sub ? 1 : blk->num_outputs; }
    size_t out_size(int port) const { return sub ? sub->stages.back()->out_size : blk->out_size_of(port); }
    size_t in_size() const { return sub ? sub->stages.front()->in_size : blk->in_size; }
    const char* name() const { return sub ? sub->desc.c_str() : blk->name; }
};

struct Dag {
    std::vector<DagNode> nodes;
    std::vector<int> outputs;
    void* d_in = nullptr; size_t d_in_cap = 0;
    size_t in_size = 0;
    std::string desc;

    ~Dag() {
        for (DagNode& nd : nodes) {
            delete nd.blk;
            if (nd.holder) destroy_graph_handle(nd.holder);
            for (void* p : nd.out_buf) cudaFree(p);
        }
        cudaFree(d_in);
    }

    int add(Block* blk, Graph* sub, void* holder, const int* refs, unsigned nin) {
        DagNode nd;
        nd.blk = blk; nd.sub = sub; nd.holder = holder;
        const int want = sub ? 1 : blk->num_inputs;
        if ((int)nin != want) { set_error("dag: %s takes %d input(s), got %u", nd.name(), want, nin); return -1; }
        for (unsigned i = 0; i < nin; ++i) {
            const int r = refs[i];
            size_t esz;
            if (r == -1) {
                if (in_size && in_size != nd.in_size()) { set_error("dag: the input feeds nodes of different sample sizes"); return -1; }
                in_size = nd.in_size();
                esz = in_size;
            } else {
                const int pn = r >> 2, pp = r & 3;
                if (r < 0 || pn >= (int)nodes.size() || pp >= nodes[(size_t)pn].nout()) { set_error("dag: bad input reference %d", r); return -1; }
                esz = nodes[(size_t)pn].out_size(pp);
            }
            if (esz != nd.in_size()) { set_error("dag: %zu-byte samples cannot feed %s (%zu-byte input)", esz, nd.name(), nd.in_size()); return -1; }
            nd.in_refs.push_back(r);
        }
        nd.out_buf.assign((size_t)nd.nout(), nullptr);
        nd.out_cap.assign((size_t)nd.nout(), 0);
        nd.out_cnt.assign((size_t)nd.nout(), 0);
        nodes.push_back(nd);
        if (!desc.empty()) desc += " ; ";
        desc += nd.name();
        return (int)nodes.size() - 1;
    }

    int reset() {
        for (DagNode& nd : nodes) {
            if (nd.sub) { if (nd.sub->reset() != 0) return -1; }
            else if (nd.blk->reset() != 0) return -1;
        }
        return 0;
    }

    int run_host(const void* x, size_t n, void* const* y, size_t* n_out) {
        if (nodes.empty() || outputs.empty()) { set_error("dag: no nodes / no outputs"); return -1; }
        cudaStream_t s = ctx().stream;
        if (n * in_size > d_in_cap) {
            LRB_CHECK(cudaStreamSynchronize(s));
            if (Block::reserve(&d_in, &d_in_cap, n * in_size) != 0) return -1;
        }
        if (n) LRB_CHECK(cudaMemcpyAsync(d_in, x, n * in_size, cudaMemcpyHostToDevice, s));
        for (DagNode& nd : nodes) {
            std::vector<const void*> ins;
            size_t cnt = 0;
            for (size_t i = 0; i < nd.in_refs.size(); ++i) {
                const int r = nd.in_refs[i];
                const void* p = r == -1 ? d_in : nodes[(size_t)(r >> 2)].out_buf[(size_t)(r & 3)];
                const size_t c = r == -1 ? n : nodes[(size_t)(r >> 2)].out_cnt[(size_t)(r & 3)];
                if (i && c != cnt) { set_error("dag: %s received inputs of different lengths (%zu, %zu)", nd.name(), cnt, c); return -1; }
                cnt = c;
                ins.push_back(p);
            }
            const size_t mo = nd.sub ? nd.sub->max_output(cnt) : nd.blk->max_output(cnt);
            for (int o = 0; o < nd.nout(); ++o) {
                const size_t bytes = (mo ? mo : 1) * nd.out_size(o);
                if (bytes > nd.out_cap[(size_t)o]) {
                    LRB_CHECK(cudaStreamSynchronize(s));
                    if (Block::reserve(&nd.out_buf[(size_t)o], &nd.out_cap[(size_t)o], bytes) != 0) return -1;
                }
            }
            size_t no = 0;
            if (nd.sub) {
                if (nd.sub->run_device(ins[0], cnt, nd.out_buf[0], &no, s) != 0) return -1;
            } else {
                if (nd.blk->run_multi(ins.data(), (int)ins.size(), cnt, nd.out_buf.data(), nd.nout(), &no, s) != 0) return -1;
            }
            for (int o = 0; o < nd.nout(); ++o) nd.out_cnt[(size_t)o] = no;
        }
        for (size_t k = 0; k < outputs.size(); ++k) {
            const DagNode& nd = nodes[(size_t)(outputs[k] >> 2)];
            const int port = outputs[k] & 3;
            const size_t c = nd.out_cnt[(size_t)port];
            if (c) LRB_CHECK(cudaMemcpyAsync(y[k], nd.out_buf[(size_t)port], c * nd.out_size(port), cudaMemcpyDeviceToHost, s));
            n_out[k] = c;
        }
        LRB_CHECK(cudaStreamSynchronize(s));
        return 0;
    }
};

}  // namespace lrb

using namespace lrb;

struct lrb200_graph_s { Graph g; };
struct lrb200_dag_s { Dag d; };
namespace lrb { void destroy_graph_handle(void* holder) { delete static_cast<lrb200_graph_s*>(holder); } }

extern "C" {

lrb200_graph_t* lrb200_graph_create(void) {
    if (lrb200_device_count() <= 0) { set_error("no CUDA device available; libluaradio_b200 has no CPU fallback"); return nullptr; }
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    lrb200_graph_t* g = new (std::nothrow) lrb200_graph_s();
    if (!g) set_error("out of memory");
    return g;
}

int lrb200_graph_append(lrb200_graph_t* g, lrb200_block_t* q) {
    if (!g || !q || !q->impl) { set_error("graph_append: null handle"); return -1; }
    if (!q->impl->dev_ptrs) { set_error("graph_append: block %s was not created with LRB200_DEVICE", q->impl->name); return -1; }
    if (!g->g.blocks.empty() && g->g.blocks.back()->out_size != q->impl->in_size) {
        set_error("graph_append: %s (out %zu B) cannot feed %s (in %zu B)", g->g.blocks.back()->name,
                  g->g.blocks.back()->out_size, q->impl->name, q->impl->in_size);
        return -1;
    }
    g->g.blocks.push_back(q->impl);
    g->g.committed = false;
    q->impl = nullptr;          // ownership moves to the graph
    delete q;
    return 0;
}

int lrb200_graph_commit(lrb200_graph_t* g, int fuse) {
    if (!g) { set_error("null graph"); return -1; }
    return g->g.commit(fuse);
}

int lrb200_graph_execute(lrb200_graph_t* g, const void* x, size_t n, void* y, size_t* n_out) {
    if (!g) { set_error("null graph"); return -1; }
    size_t no = 0;
    int rc = g->g.run_host(x, n, y, &no);
    if (n_out) *n_out = no;
    return rc;
}

int lrb200_graph_execute_device(lrb200_graph_t* g, const void* dx, size_t n, void* dy, size_t* n_out) {
    if (!g) { set_error("null graph"); return -1; }
    size_t no = 0;
    int rc = g->g.run_device(dx, n, dy, &no, ctx().stream);
    if (n_out) *n_out = no;
    return rc;
}

size_t lrb200_graph_max_output(const lrb200_graph_t* g, size_t n) {
    if (!g) return 0;
    lrb200_graph_t* gg = const_cast<lrb200_graph_t*>(g);
    if (!gg->g.committed && gg->g.commit(1) != 0) return 0;
    // super-chunk mode: one call may hand back the results of the slots completed while n samples were appended
    if (gg->g.sc) return (n / gg->g.sc + 2) * gg->g.sc_outcap;
    return gg->g.max_output(n);
}

int lrb200_graph_set_superchunk(lrb200_graph_t* g, size_t samples) {
    if (!g) { set_error("null graph"); return -1; }
    return g->g.set_superchunk(samples);
}

int lrb200_graph_flush(lrb200_graph_t* g, void* y, size_t* n_out) {
    if (!g) { set_error("null graph"); return -1; }
    size_t no = 0;
    int rc = g->g.flush(y, &no);
    if (n_out) *n_out = no;
    return rc;
}

long long lrb200_graph_halo(lrb200_graph_t* g) {
    if (!g) { set_error("null graph"); return -1; }
    return g->g.halo();
}

int lrb200_graph_execute_shard(lrb200_graph_t* g, lrb200_graph_t* g_head, const void* dx, size_t halo, size_t n,
                               uint64_t start, void* dy, size_t* n_out, void* halo_ready_event) {
    if (!g) { set_error("null graph"); return -1; }
    size_t no = 0;
    int rc = g->g.run_shard(g_head ? g_head->g : g->g, dx, halo, n, start, dy, &no, (cudaEvent_t)halo_ready_event);
    if (n_out) *n_out = no;
    return rc;
}

int lrb200_graph_reset(lrb200_graph_t* g) {
    if (!g) { set_error("null graph"); return -1; }
    return g->g.reset();
}

int lrb200_graph_seek(lrb200_graph_t* g, uint64_t sample_index) {
    if (!g) { set_error("null graph"); return -1; }
    return g->g.seek(sample_index);
}

int lrb200_graph_num_stages(const lrb200_graph_t* g) {
    if (!g) return 0;
    lrb200_graph_t* gg = const_cast<lrb200_graph_t*>(g);
    if (!gg->g.committed && gg->g.commit(1) != 0) return -1;
    return (int)gg->g.stages.size();
}

const char* lrb200_graph_describe(const lrb200_graph_t* g) {
    if (!g) return "";
    lrb200_graph_t* gg = const_cast<lrb200_graph_t*>(g);
    if (!gg->g.committed && gg->g.commit(1) != 0) return "";
    return gg->g.desc.c_str();
}

const char* lrb200_graph_stage_name(const lrb200_graph_t* g, int stage) {
    if (!g) return "";
    lrb200_graph_t* gg = const_cast<lrb200_graph_t*>(g);
    if (!gg->g.committed && gg->g.commit(1) != 0) return "";
    if (stage < 0 || stage >= (int)gg->g.stages.size()) return "";
    return gg->g.stages[stage]->name;
}

int lrb200_graph_set_timing(lrb200_graph_t* g, int enable) {
    if (!g) { set_error("null graph"); return -1; }
    g->g.timing = enable != 0;
    return 0;
}

double lrb200_graph_stage_time_ms(lrb200_graph_t* g, int stage, int* executions) {
    if (executions) *executions = 0;
    if (!g || stage < 0 || stage >= (int)g->g.tcount.size()) return 0.0;
    if (cudaStreamSynchronize(ctx().stream) != cudaSuccess) return 0.0;
    double total = 0.0;
    int cnt = g->g.tcount[stage];
    for (int i = 0; i < cnt; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, g->g.tev[stage][2 * i], g->g.tev[stage][2 * i + 1]) == cudaSuccess) total += ms;
    }
    if (executions) *executions = cnt;
    g->g.tcount[stage] = 0;
    return total;
}

void lrb200_graph_destroy(lrb200_graph_t* g) { delete g; }

// ---- device DAG ------------------------------------------------------------------------------------------------------
lrb200_dag_t* lrb200_dag_create(void) {
    if (lrb200_device_count() <= 0) { set_error("no CUDA device available; libluaradio_b200 has no CPU fallback"); return nullptr; }
    if (ctx().device < 0 && lrb200_init(0) != 0) return nullptr;
    lrb200_dag_t* d = new (std::nothrow) lrb200_dag_s();
    if (!d) set_error("out of memory");
    return d;
}

int lrb200_dag_add_block(lrb200_dag_t* d, lrb200_block_t* q, const int* inputs, unsigned num_inputs) {
    if (!d || !q || !q->impl || (!inputs && num_inputs)) { set_error("dag_add_block: null argument"); return -1; }
    if (!q->impl->dev_ptrs) { set_error("dag_add_block: block %s was not created with LRB200_DEVICE", q->impl->name); return -1; }
    const int id = d->d.add(q->impl, nullptr, nullptr, inputs, num_inputs);
    if (id < 0) return -1;
    q->impl = nullptr;          // ownership moves to the DAG
    delete q;
    return id;
}

int lrb200_dag_add_graph(lrb200_dag_t* d, lrb200_graph_t* g, int input) {
    if (!d || !g) { set_error("dag_add_graph: null argument"); return -1; }
    if (!g->g.committed && g->g.commit(1) != 0) return -1;
    if (g->g.stages.empty()) { set_error("dag_add_graph: empty graph"); return -1; }
    return d->d.add(nullptr, &g->g, g, &input, 1);       // on success the handle belongs to the DAG
}

int lrb200_dag_set_outputs(lrb200_dag_t* d, const int* outputs, unsigned num_outputs) {
    if (!d || !outputs || !num_outputs) { set_error("dag_set_outputs: null argument"); return -1; }
    for (unsigned k = 0; k < num_outputs; ++k) {
        const int r = outputs[k];
        if (r < 0 || (r >> 2) >= (int)d->d.nodes.size() || (r & 3) >= d->d.nodes[(size_t)(r >> 2)].nout()) { set_error("dag_set_outputs: bad reference %d", r); return -1; }
    }
    d->d.outputs.assign(outputs, outputs + num_outputs);
    return 0;
}

int lrb200_dag_execute(lrb200_dag_t* d, const void* x, size_t n, void* const* y, size_t* n_out) {
    if (!d || !y || !n_out || (n && !x)) { set_error("dag_execute: null argument"); return -1; }
    return d->d.run_host(x, n, y, n_out);
}

size_t lrb200_dag_max_output(const lrb200_dag_t* d, unsigned output, size_t n) {
    if (!d || output >= d->d.outputs.size()) return 0;
    // conservative: no node here produces more samples than its input times the interpolation factors on the way
    size_t m = n;
    for (const DagNode& nd : d->d.nodes) { const size_t c = nd.sub ? nd.sub->max_output(n) : nd.blk->max_output(n); if (c > m) m = c; }
    return m;
}

int lrb200_dag_reset(lrb200_dag_t* d) {
    if (!d) { set_error("null dag"); return -1; }
    return d->d.reset();
}

const char* lrb200_dag_describe(const lrb200_dag_t* d) { return d ? d->d.desc.c_str() : ""; }

void lrb200_dag_destroy(lrb200_dag_t* d) { delete d; }

}  // extern "C"
