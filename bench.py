#!/usr/bin/env python3
"""bench.py -- WBFM-mono chain throughput on B200 (BASELINE.json metric), roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload wbfm_mono_256Mi|wbfm_mono_8Gi]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (default config.workload = "wbfm_mono_256Mi", BASELINE.json configs[2]): the full
examples/rtlsdr_wbfm_mono.lua flow graph  Tuner(-250e3, 200e3, 5) -> FrequencyDiscriminator(1.25) ->
Lowpass(128, 15e3) -> FMDeemphasis(75e-6) -> Downsampler(5)  on 256 Mi complex-float32 samples of synthetic
FM IQ at 1.1025 MS/s per GPU (weak scaling).  A "step" is one pass of the chain over one rank's chunk.
--workload wbfm_mono_8Gi is BASELINE.json configs[4] as written: ONE 8 Gi-sample stream cut into N time chunks
(strong scaling, 8 Gi / N samples per rank; N = 1 needs 64 GiB of HBM for the input).

  value     : whole-job M input-samples/s, inputs resident in HBM (device-generated synthetic IQ), CUDA events on the
              launching stream, max over ranks.  Per-stage times are measured in a SEPARATE pass after the timed loop.
  e2e       : same metric through the C ABI with HOST buffers (lrb200_graph_execute: pinned host in, host out,
              H2D + kernels + D2H pipelined inside the timed call).
  e2e_small : the same call in the reference's per-vector regime: pageable host vectors of 8192 / 32768 / 131072
              samples (radio/core/pipe.lua:73, radio/blocks/sources/zero.lua:30), synchronous per call and in
              super-chunk mode (lrb200_graph_set_superchunk).
  N > 1     : the stream is sharded by time chunk.  Each step rank r sends the last HALO input samples of its chunk to
              rank r+1 (copy engine through a CUDA-IPC peer pointer, or NCCL P2P with --halo nccl; on its own stream) while
              every rank already runs its stream cold from HALO samples early; only the first stage's few tiles that read
              the neighbour's samples wait for them (lrb200_graph_execute_shard).  HALO = lrb200_graph_halo().
  check     : every rank re-computes windows of its output with the numpy oracle run cold from HALO samples before the
              window (the first window straddles the rank's left chunk boundary) and the run FAILS on a mismatch.
  --dump-outputs DIR : after the timed steps, what the last one computed (the chain's audio output) goes to DIR/audio.npy
              (float32; DIR/audio_rank<r>.npy per rank for N > 1).  Inputs are seeded, so two builds run with the same
              arguments can be compared output for output.  Beyond DUMP_BYTES in all, a fixed, seeded sample of the outputs is
              written instead, with the sampled output indices beside it (<name>_index.npy, float64).
  --impl reference : the C restatement of the reference's CPU path (oracle/lr_oracle.c: VOLK dot-product FIRs and the
              overlap-save FIRs the reference defaults to with FFTW; the faster one is timed) on all usable host
              cores -- the reference stack (LuaJIT/VOLK/liquid/FFTW) is not installable here.  Does not load the
              GPU library.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # write nothing into the tree, which may be read-only (oracle/cbuild.py: the same for the native build)

RATE = 1102500.0
TUNE_OFFSET = -250e3
BANDWIDTH = 200e3
HALO = 4000            # tests: a lead-in that covers lrb200_graph_halo() of the chain with margin
ORACLE_LEAD = HALO     # cold-start lead-in of the oracle windows (multiple of 25; > lrb200_graph_halo of the chain)
ALG_BYTES_CHAIN = 8.0 + 4.0 / 25.0          # fused minimum per input sample (SURVEY.md 8d)
ALG_BYTES_TUNER = 8.0 + 8.0 / 5.0           # tuner kernel: read 8 B, write 8/5 B per input sample
ALG_BYTES_TUNER_DISC = 8.0 + 4.0 / 5.0      # tuner with the discriminator fused: the 1/5-rate output is float32
ALG_BYTES_FIR = 16.0                        # plain complex FIR: 8 in + 8 out
ALG_BYTES_CFG2 = 8.0 + 8.0 / 5.0            # translator + FIR + /5 fused: 9.6 B per input sample
FP32_PEAK_TFLOPS = 74.0                     # packed FFMA2, measured on this pool's B200 with tools/ubench.cu (DESIGN.md 3)
WORKLOADS = {"wbfm_mono_256Mi": 268435450, "wbfm_mono_8Gi": 8589934575}
DUMP_BYTES = 64 << 20                       # --dump-outputs: at most this many bytes in all
METRIC = "WBFM-mono chain Msamples/s (input samples) @N B200; FIR-128 HBM GB/s vs roofline"
CHAIN = "Tuner(-250e3,200e3,5)>FreqDiscriminator(1.25)>Lowpass(128,15e3)>FMDeemphasis(75e-6)>Downsampler(5)"
TOLERANCE = ("1e-5*max(1,|ref|_inf) against the pinned oracle (north_star); the reference's own specs use 1e-6 absolute "
             "-- the fused tuner+discriminator stage is also tested at 1e-6 (tests/test_gpu_round2.py)")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the device runs the bench load.

    The timed region of the default run is ~16 ms, shorter than one nvidia-smi period and far shorter than nvidia-smi's own
    start-up, so: start() launches the sampler BEFORE the warm-up and wait_ready() blocks until its first line arrives;
    every line is time-stamped on arrival; mark(t0, t1) names the timed region; and when fewer than MIN_LOAD samples fell
    inside it the caller keeps the identical load running (continue_load) until enough were taken.  The result says how many
    samples came from the timed region itself and how many from warm-up / continuation of the same step loop."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    MIN_LOAD = 4
    PERIOD_MS = 20

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None
        self.t_load0 = self.t_load1 = self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.monotonic(), line.strip()))

    def wait_ready(self, timeout=8.0):
        """Block until the first sample line has arrived (nvidia-smi start-up can take a second on an 8-GPU box)."""
        t_end = time.monotonic() + timeout
        while self.proc and not self.samples and time.monotonic() < t_end and self.proc.poll() is None:
            time.sleep(0.01)
        return bool(self.samples)

    def load_begin(self):
        self.t_load0 = time.monotonic()

    def mark(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def count_in(self, t0, t1):
        return sum(1 for t, _ in list(self.samples) if t0 <= t <= t1)

    def continue_load(self, step, sync, budget_s=1.5):
        """Keep the same step loop running until MIN_LOAD samples were taken under load (or the budget is spent)."""
        if not self.proc or self.t_load0 is None:
            return
        t_end = time.monotonic() + budget_s
        while self.count_in(self.t_load0, time.monotonic()) < self.MIN_LOAD and time.monotonic() < t_end:
            for _ in range(8):
                step()
            sync()
        self.t_load1 = time.monotonic()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        if self.t_load1 is None:
            self.t_load1 = time.monotonic()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons = [], None, set()
            for s in rows:
                f = [t.strip() for t in s.split(",")]
                if len(f) < 6:
                    continue
                try:
                    sm.append(float(f[0]))
                    mx = float(f[1])
                except ValueError:
                    continue
                for nm, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            return sm, mx, reasons

        rows = list(self.samples)
        lo = self.t_load0 if self.t_load0 is not None else float("-inf")
        load = [s for t, s in rows if lo <= t <= self.t_load1]
        timed = [s for t, s in rows if self.t0 is not None and self.t0 <= t <= self.t1]
        sm, mx, reasons = parse(load)
        if not sm:                                   # nothing under load: report what there is and say so
            sm, mx, reasons = parse([s for _, s in rows])
            reasons = set(reasons) | {"no sample under load"}
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_region": len(parse(timed)[0]),
                "period_ms": self.PERIOD_MS,
                "window": "warm-up + timed region + continuation of the same step loop until >= %d samples" % self.MIN_LOAD}


def chain_taps(fu=None):
    """Tap design exactly as the blocks' initialize() does it.  `fu`: a filter_utils-like module (product side by
    default; the reference arm passes the oracle's so that it does not import the GPU package's native library)."""
    if fu is None:
        import luaradio_b200 as radio
        fu = radio.filter_utils
    t1 = np.array(fu.firwin_lowpass(128, (BANDWIDTH / 2) / (RATE / 2)), np.float32)
    r1 = RATE / 5
    t2 = np.array(fu.firwin_lowpass(128, 15e3 / (r1 / 2)), np.float32)
    tau = 75e-6
    cutoff = 1 / (2 * math.pi * tau)
    tt = 1 / (2 * math.pi * cutoff)
    tt = 1 / (2 * r1 * math.tan(1 / (2 * r1 * tt)))
    b = np.array([1 / (1 + 2 * tt * r1)] * 2, np.float32)
    a = np.array([1.0, (1 - 2 * tt * r1) / (1 + 2 * tt * r1)], np.float32)
    return t1, t2, b, a


def build_chain_graph(lib, _lib, iq_format=None):
    """The rtlsdr_wbfm_mono.lua chain as C-ABI blocks appended to a GPU flow graph (what CompositeBlock.run builds).
    `iq_format`: prepend the source-boundary sample-format converter (raw file/dongle bytes in, SURVEY 8f row 1)."""
    t1, t2, b, a = chain_taps()
    D = _lib.LRB200_DEVICE
    g = _lib.check_handle(lib.lrb200_graph_create(), "graph")
    blocks = [lib.lrb200_iqconv_create(iq_format.encode(), D)] if iq_format else []
    blocks += [
        lib.lrb200_rotator_create(TUNE_OFFSET / RATE, D),
        lib.lrb200_fir_create_crcf(t1.ctypes.data, 128, 1, D),
        lib.lrb200_downsample_create(5, 8, D),
        lib.lrb200_discrim_create(2 * math.pi * 1.25, D),
        lib.lrb200_fir_create_rrrf(t2.ctypes.data, 128, 1, D),
        lib.lrb200_iir_create_rrrf(b.ctypes.data, 2, a.ctypes.data, 2, D),
        lib.lrb200_downsample_create(5, 4, D),
    ]
    for h in blocks:
        _lib.check_handle(h, "block")
        _lib.check(lib.lrb200_graph_append(g, h), "graph_append")
    _lib.check(lib.lrb200_graph_commit(g, 1), "graph_commit")
    return g


def oracle_window(O, out_start, out_count):
    """Oracle outputs [out_start, out_start + out_count) of the chain on the global synthetic stream: the numpy chain run
    COLD from ORACLE_LEAD input samples before the window (every stage has finite memory; 4000 samples bury it)."""
    in_start = out_start * 25
    lead = min(ORACLE_LEAD, in_start)
    x = O.synth_fm_iq(in_start - lead, lead + out_count * 25)
    y = O.wbfm_mono_chain().process(x) if lead == 0 else _oracle_from(O, x, in_start - lead)
    return y[lead // 25: lead // 25 + out_count]


def _oracle_from(O, x, n0):
    """The oracle chain started at global input index n0 (multiple of 25): only the translator depends on the index."""
    ch = O.wbfm_mono_chain()
    ch.blocks[0].blocks[0].n0 = n0          # FrequencyTranslator: phase of the GLOBAL sample index
    return ch.process(x)


def dump_outputs(out_dir, name, y, budget):
    """Write the 1-D float array `y` (numpy, or a torch tensor on the device) to out_dir/<name>.npy.  When it exceeds `budget`
    bytes, a sample of it is written instead: sorted output indices drawn with a fixed seed (the same set in every run with
    the same arguments), stored as <name>_index.npy in float64 (exact for any index below 2**53)."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(y.shape[0])
    if n * 4 > budget:
        idx = np.unique(np.random.default_rng(0).integers(0, n, budget // 12))
        np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
        if not isinstance(y, np.ndarray):
            import torch
            idx = torch.from_numpy(idx).to(y.device)
        y = y[idx]
    if not isinstance(y, np.ndarray):
        y = y.cpu().numpy()
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(y, np.float32))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from luaradio_b200 import _lib, sharding
    from oracle import lr_oracle as O

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and rank == 0:
        sys.stderr.write("note: WORLD_SIZE=%d, --gpus=%d; using WORLD_SIZE\n" % (world, args.gpus))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.require_device(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    _lib.check(lib.lrb200_set_stream(ctypes.c_void_p(stream.cuda_stream)), "set_stream")

    strong = args.workload == "wbfm_mono_8Gi"
    total = args.samples if args.samples else WORKLOADS[args.workload]
    if strong:
        n = (total // world // 25) * 25       # one stream, cut into `world` chunks
    else:
        n = (total // 25) * 25                # `total` samples per rank
    start = rank * n                          # global index of this rank's first sample (chunk boundaries on multiples of 25)
    g = build_chain_graph(lib, _lib)
    HALO = int(lib.lrb200_graph_halo(g))
    assert HALO > 0 and HALO % 25 == 0, HALO
    g_head = None
    # this rank's chunk lives at x[HALO:], the halo from the left neighbour is received into x[:HALO]
    xp = lib.lrb200_malloc((n + HALO) * 8)                 # a plain cudaMalloc allocation: exportable to the neighbour process
    assert xp, _lib.last_error()
    x = None
    assert (xp + HALO * 8) % 16 == 0
    _lib.check(lib.lrb200_synth_fm_iq(ctypes.c_void_p(xp + HALO * 8), start, n, 1, RATE, 250e3, 75e3, 0.5, 0.01), "synth")
    n_out_max = lib.lrb200_graph_max_output(g, n)
    y = torch.empty(n_out_max + 16, dtype=torch.float32, device="cuda")
    desc = lib.lrb200_graph_describe(g).decode()
    nstages = lib.lrb200_graph_num_stages(g)
    n_out = ctypes.c_size_t(0)
    comm = torch.cuda.Stream() if world > 1 else None
    halo_ev = torch.cuda.Event() if world > 1 else None
    # halo transport: "ipc" = the copy engine reads the left neighbour's tail through a peer-mapped pointer (no SM, no
    # collective kernel beside the persistent compute kernels); "nccl" = batched NCCL send/recv on the side stream
    transport, peer_tail = args.halo if world > 1 else "none", None
    if world > 1 and transport == "ipc":
        try:
            hbuf = (ctypes.c_ubyte * 64)()
            _lib.check(lib.lrb200_ipc_export(ctypes.c_void_p(xp), hbuf), "ipc_export")
            handles = [None] * world
            dist.all_gather_object(handles, bytes(hbuf))
            if rank > 0:
                base = lib.lrb200_ipc_import(handles[rank - 1])
                if not base:
                    raise RuntimeError(_lib.last_error())
                peer_tail = base + (HALO + n - HALO) * 8          # the neighbour's last HALO samples
            ok = torch.tensor([1], device="cuda")
        except Exception as e:
            sys.stderr.write("rank %d: CUDA IPC unavailable (%s)\n" % (rank, e))
            ok = torch.tensor([0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() == 0:
            transport = "nccl"
    if world > 1 and transport == "nccl":
        xt = torch.empty(2 * HALO, dtype=torch.complex64, device="cuda")    # NCCL staging: [recv halo | send tail]

    def step():
        if world > 1:
            # neighbour exchange on its own stream: it only gates the head piece inside execute_shard
            comm.wait_stream(stream)
            with torch.cuda.stream(comm):
                if transport == "ipc":
                    if rank > 0:
                        _lib.check(lib.lrb200_memcpy_d2d(ctypes.c_void_p(xp), ctypes.c_void_p(peer_tail), HALO * 8,
                                                         ctypes.c_void_p(comm.cuda_stream)), "peer copy")
                else:
                    # stage through torch tensors: tail -> xt[HALO:], exchange, xt[:HALO] -> x[:HALO]
                    _lib.check(lib.lrb200_memcpy_d2d(ctypes.c_void_p(xt.data_ptr() + HALO * 8), ctypes.c_void_p(xp + n * 8), HALO * 8,
                                                     ctypes.c_void_p(comm.cuda_stream)), "stage tail")
                    sharding.exchange_halo(dist, xt[HALO:], xt[:HALO], rank, world, HALO)
                    _lib.check(lib.lrb200_memcpy_d2d(ctypes.c_void_p(xp), ctypes.c_void_p(xt.data_ptr()), HALO * 8,
                                                     ctypes.c_void_p(comm.cuda_stream)), "unstage halo")
                halo_ev.record(comm)
            _lib.check(lib.lrb200_graph_execute_shard(g, None, ctypes.c_void_p(xp), HALO, n, start, ctypes.c_void_p(y.data_ptr()),
                                                      ctypes.byref(n_out), ctypes.c_void_p(halo_ev.cuda_event)), "execute_shard")
        else:
            _lib.check(lib.lrb200_graph_reset(g), "reset")
            _lib.check(lib.lrb200_graph_seek(g, start), "seek")
            _lib.check(lib.lrb200_graph_execute_device(g, ctypes.c_void_p(xp + HALO * 8), n, ctypes.c_void_p(y.data_ptr()),
                                                       ctypes.byref(n_out)), "execute")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_ready()
    barrier()
    sampler.load_begin()
    for _ in range(warm):
        step()
    barrier()
    launches0 = lib.lrb200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_host0 = time.monotonic()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    sampler.mark(t_host0, time.monotonic())
    ms_total = e0.elapsed_time(e1)
    launches = lib.lrb200_launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "audio" if world == 1 else "audio_rank%d" % rank, y[:int(n_out.value)], DUMP_BYTES // world)
    tt = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_step = float(tt.item()) / args.steps
    # the timed region is shorter than a sampling period: every rank keeps the identical load running (untimed) while
    # rank 0 collects its clock samples.  N > 1: the same count on every rank (derived from the all-reduced step time), so
    # that the halo exchange inside step() stays matched across ranks
    if world > 1:
        for _ in range(int(min(512, max(16, 120.0 / max(ms_step, 1e-3))))):
            step()
        barrier()
        sampler.t_load1 = time.monotonic()
    elif rank == 0:
        sampler.continue_load(step, torch.cuda.synchronize)
    clocks = sampler.stop() if rank == 0 else None
    value = world * n / (ms_step * 1e-3) / 1e6          # M input-samples/s, whole job
    n_out_step = int(n_out.value)

    # ---- per-stage device times: a separate pass, so the event pairs are not inside the headline loop
    _lib.check(lib.lrb200_graph_set_timing(g, 1), "timing")
    for _ in range(max(3, min(args.steps, 10))):
        step()
    barrier()
    stage_ms = []
    for k in range(nstages):
        cnt = ctypes.c_int(0)
        t = lib.lrb200_graph_stage_time_ms(g, k, ctypes.byref(cnt))
        stage_ms.append((lib.lrb200_graph_stage_name(g, k).decode(), t / max(cnt.value, 1)))
    _lib.check(lib.lrb200_graph_set_timing(g, 0), "timing")

    # ---- parity check of this run's output (outside the timed region): windows vs the oracle, every rank
    check = None
    if not args.no_check:
        step()
        barrier()
        W = 8000                                           # outputs per window = 200 000 input samples
        first_out = start // 25
        wins = [0, max(0, n_out_step // 2 - W // 2), max(0, n_out_step - W)]
        worst, bad = 0.0, 0
        for w0 in sorted(set(wins)):
            cnt = min(W, n_out_step - w0)
            got = y[w0:w0 + cnt].cpu().numpy()
            ref = oracle_window(O, first_out + w0, cnt)
            scale = max(1.0, float(np.max(np.abs(ref))))
            err = float(np.max(np.abs(got - ref))) / scale
            worst = max(worst, err)
            bad += int(not (err <= 1e-5))
        # gather at the sink (SURVEY.md 8e): rank 0 collects the last W/2 outputs of every rank and the first W/2 of its
        # right neighbour and compares each joined window -- W outputs STRADDLING a shard boundary -- with one continuous
        # oracle run
        gathered = 0
        if world > 1:
            half = W // 2
            edge = torch.cat([y[:half], y[n_out_step - half:n_out_step]]).contiguous()
            parts = [torch.empty_like(edge) for _ in range(world)] if rank == 0 else None
            dist.gather(edge, parts, dst=0)
            if rank == 0:
                per = n // 25
                for r in range(1, world):
                    got = torch.cat([parts[r - 1][half:], parts[r][:half]]).cpu().numpy()
                    ref = oracle_window(O, r * per - half, W)
                    scale = max(1.0, float(np.max(np.abs(ref))))
                    err = float(np.max(np.abs(got - ref))) / scale
                    worst = max(worst, err)
                    bad += int(not (err <= 1e-5))
                    gathered += 1
        res = torch.tensor([worst, float(bad)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(res, op=dist.ReduceOp.MAX)
        check = {"windows_per_rank": len(set(wins)), "window_outputs": W, "boundary_windows_gathered_at_rank0": gathered,
                 "max_rel_err": float(res[0].item()), "ok": res[1].item() == 0.0,
                 "what": "output windows at each rank's chunk start, middle and end vs the numpy oracle run cold %d samples before the "
                         "window; plus, gathered at rank 0, one window straddling every shard boundary (last outputs of rank r-1 + "
                         "first outputs of rank r) vs one continuous oracle run" % ORACLE_LEAD}
        if not check["ok"]:
            if rank == 0:
                emit(json.dumps({"error": "parity check failed", "check": check}))
            sys.exit(1)

    if args.profile:
        if rank == 0:
            emit(json.dumps({"profile_run": True, "ms_per_step": ms_step, "stages_ms": dict(stage_ms)}))
            bench_fir128(lib, _lib, torch, stream, args)
        return

    # ---- e2e: HOST buffers through the C ABI (pinned in, host out), H2D/D2H inside the timed call
    ne = min(n, 268435450)                                # (the 8 Gi workload: the first 256 Mi of the rank's chunk)
    hin = lib.lrb200_host_alloc(ne * 8)
    hout = lib.lrb200_host_alloc((ne // 25 + 64) * 4)
    assert hin and hout, _lib.last_error()
    _lib.check(lib.lrb200_memcpy_d2h(hin, ctypes.c_void_p(xp + HALO * 8), ne * 8), "d2h")
    _lib.check(lib.lrb200_sync(), "sync")
    e2e_steps = max(2, min(args.steps, 8))

    def e2e_step():
        _lib.check(lib.lrb200_graph_reset(g), "reset")
        _lib.check(lib.lrb200_graph_seek(g, start), "seek")
        _lib.check(lib.lrb200_graph_execute(g, hin, ne, hout, ctypes.byref(n_out)), "graph_execute(host)")

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    te = torch.tensor([(t1 - t0) / e2e_steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * ne / float(te.item()) / 1e6
    e2e_out = int(n_out.value)

    e2e_small = bench_e2e_small(lib, _lib, g, hin, ne) if world == 1 else None

    # ---- the same end-to-end call fed the RTL-SDR's native u8 I/Q bytes (2 B/sample over PCIe, converted on the
    # device by the graph's first stage) -- extra information, N == 1 only; the headline e2e stays the f32 boundary
    e2e_u8 = None
    if world == 1 and not strong:
        g8 = build_chain_graph(lib, _lib, "u8")
        h8 = lib.lrb200_host_alloc(n * 2)
        assert h8, _lib.last_error()
        CH = 1 << 24
        xr = torch.empty(2 * CH, dtype=torch.float32, device="cuda")
        for o in range(0, n, CH):      # quantise the synthetic samples to u8 on the device, park them in pinned host memory
            m = min(CH, n - o)
            _lib.check(lib.lrb200_memcpy_d2d(ctypes.c_void_p(xr.data_ptr()), ctypes.c_void_p(xp + (HALO + o) * 8), m * 8, None), "copy")
            _lib.check(lib.lrb200_sync(), "sync")
            q = (xr[:2 * m] * 127.5 + 127.5).round_().clamp_(0, 255).to(torch.uint8).contiguous()
            _lib.check(lib.lrb200_memcpy_d2h(ctypes.c_void_p(h8 + o * 2), ctypes.c_void_p(q.data_ptr()), q.numel()), "d2h")
            _lib.check(lib.lrb200_sync(), "sync")
            torch.cuda.synchronize()
        del q, xr

        def e2e8_step():
            _lib.check(lib.lrb200_graph_reset(g8), "reset")
            _lib.check(lib.lrb200_graph_execute(g8, h8, n, hout, ctypes.byref(n_out)), "graph_execute(host,u8)")

        e2e8_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e8_step()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        e2e_u8 = {"value": round(n / ((t1 - t0) / e2e_steps) / 1e6, 1), "unit": "Msamples/s", "h2d_bytes_per_step": n * 2,
                  "d2h_bytes_per_step": int(n_out.value) * 4, "graph": lib.lrb200_graph_describe(g8).decode(),
                  "note": "input = raw u8 I/Q bytes (IQFileSource/RtlSdrSource format), converted by the graph's first stage"}
        lib.lrb200_host_free(h8)
        lib.lrb200_graph_destroy(g8)

    result = None
    if rank == 0:
        peak, peak_src = peaks()
        dom = max(stage_ms, key=lambda kv: kv[1])
        dom_bytes = (ALG_BYTES_TUNER_DISC if dom[0].startswith("tuner+discrim") else
                     ALG_BYTES_TUNER if dom[0].startswith("tuner") else ALG_BYTES_FIR)
        achieved = dom_bytes * n / (dom[1] * 1e-3) / 1e9 if dom[1] > 0 else 0.0
        # useful FP32 work of the tuner kernel: 128/5 complex-by-real MACs per input sample = 4 flop each
        fp32_tflops = (4.0 * 128 / 5) * n / (dom[1] * 1e-3) / 1e12 if dom[1] > 0 and dom[0].startswith("tuner") else None
        traffic = None
        try:
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel at this workload size,
            # from the committed `ncu --set full` capture (profiles/); GB
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom[0])
            if traffic is not None and n != 268435450:
                traffic = None
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": dom[0], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "hbm_frac": round(achieved / peak, 4), "peak_source": peak_src, "traffic": traffic,
                "algorithmic_bytes_per_input_sample": dom_bytes,
                "chain_fused_min_GBs": round(ALG_BYTES_CHAIN * world * n / (ms_step * 1e-3) / 1e9, 1)}
        if fp32_tflops is not None:
            roof.update({"fp32_frac": round(fp32_tflops / FP32_PEAK_TFLOPS, 4), "fp32_achieved_tflops": round(fp32_tflops, 2),
                         "fp32_peak_tflops": FP32_PEAK_TFLOPS,
                         "fp32_note": "useful MAC flops only (4*128/5 per input sample) against the measured packed-FFMA2 peak; this kernel is "
                                      "FP32/issue-bound before it is HBM-bound (DESIGN.md 3)"})
        result = {
            "metric": METRIC,
            "value": round(value, 1), "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload if total == WORKLOADS[args.workload] else "wbfm_mono_%d" % total,
                       "samples_per_gpu": n, "total_samples": world * n, "sample_rate_hz": RATE, "chain": CHAIN,
                       "graph": desc, "halo_samples": HALO if world > 1 else 0,
                       "sharding": ("time-chunk; halo = %s on a side stream; only the tiles that read it wait (lrb200_graph_execute_shard)" %
                                    {"ipc": "copy-engine read of the left neighbour's tail through a CUDA-IPC peer pointer over NVLink",
                                     "nccl": "NCCL P2P send/recv"}[transport]) if world > 1 else "single GPU",
                       "halo_transport": transport,
                       "l2": "inputs (%.1f GiB/step) larger than L2, no flush" % (n * 8 / 2**30), "tolerance": TOLERANCE},
            "gpu_launches": int(launches),
            "stages_ms": {k: round(v, 4) for k, v in stage_ms},
            "roofline": roof,
            "e2e": {"value": round(e2e_value, 1), "unit": "Msamples/s", "h2d_bytes_per_step": ne * 8,
                    "d2h_bytes_per_step": e2e_out * 4, "api": "lrb200_graph_execute (host pointers)", "steps": e2e_steps,
                    "samples_per_call": ne},
            "clocks": clocks,
        }
        if check:
            result["check"] = check
        if e2e_small:
            result["e2e_small"] = e2e_small
        if e2e_u8:
            result["e2e_u8"] = e2e_u8
    lib.lrb200_host_free(hin)
    lib.lrb200_host_free(hout)
    lib.lrb200_graph_destroy(g)
    if g_head:
        lib.lrb200_graph_destroy(g_head)
    if world > 1:
        dist.barrier()                 # nobody frees a buffer a neighbour may still read
    if peer_tail:
        lib.lrb200_ipc_close(ctypes.c_void_p(peer_tail - n * 8))
    lib.lrb200_free(ctypes.c_void_p(xp))
    del y

    # ---- FIR-128 alone (second half of the BASELINE metric), configs[1] and the CPU baseline: rank 0, N == 1 only
    if rank == 0 and world == 1:
        result["fir128"] = bench_fir128(lib, _lib, torch, stream, args)
        result["cfg2"] = bench_cfg2(lib, _lib, torch, stream, args)
        result["cpu_baseline"] = cpu_baseline(args)
    if rank == 0:
        emit(json.dumps(result))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_e2e_small(lib, _lib, g, hin_pinned, n_avail):
    """The drop-in regime: lrb200_graph_execute on PAGEABLE host vectors of the sizes the reference's pipes deliver."""
    out = {"unit": "Msamples/s", "memory": "pageable (numpy) in and out; sync_pinned: vectors in lrb200_host_alloc memory "
                                          "(what a platform.alloc hook gives the reference's pipe buffers, INTEGRATION.md)",
           "api": "lrb200_graph_execute", "sync": {}, "superchunk_1Mi": {}, "sync_pinned": {}}
    src = np.ctypeslib.as_array(ctypes.cast(hin_pinned, ctypes.POINTER(ctypes.c_float)), shape=(2 * n_avail,))
    for vec, total in ((8192, 1 << 25), (32768, 1 << 26), (131072, 1 << 27)):
        total = min(total, (n_avail // vec) * vec)
        x = np.array(src[:2 * total], copy=True)             # pageable copy of the stream
        for mode, sc in (("sync", 0), ("superchunk_1Mi", 1 << 20), ("sync_pinned", 0)):
            _lib.check(lib.lrb200_graph_reset(g), "reset")
            _lib.check(lib.lrb200_graph_set_superchunk(g, sc), "set_superchunk")
            cap = lib.lrb200_graph_max_output(g, vec) + 64
            y = np.empty(cap, np.float32)
            no = ctypes.c_size_t(0)
            xp, yp = x.ctypes.data, y.ctypes.data
            ypin = None
            if mode == "sync_pinned":
                ypin = lib.lrb200_host_alloc(cap * 4)
                xp, yp = hin_pinned, ypin
            produced = 0
            for o in range(0, 64 * vec, vec):                 # warm-up
                _lib.check(lib.lrb200_graph_execute(g, xp + o * 8, vec, yp, ctypes.byref(no)), "execute")
            _lib.check(lib.lrb200_graph_flush(g, yp, ctypes.byref(no)), "flush")
            _lib.check(lib.lrb200_graph_reset(g), "reset")
            execute, byref = lib.lrb200_graph_execute, ctypes.byref
            t0 = time.perf_counter()
            for o in range(0, total, vec):
                if execute(g, xp + o * 8, vec, yp, byref(no)) != 0:
                    raise RuntimeError(_lib.last_error())
                produced += no.value
            _lib.check(lib.lrb200_graph_flush(g, yp, ctypes.byref(no)), "flush")
            produced += no.value
            el = time.perf_counter() - t0
            assert produced == (total + 24) // 25, (produced, total)
            out[mode][str(vec)] = round(total / el / 1e6, 1)
            if ypin:
                lib.lrb200_host_free(ypin)
        del x
    _lib.check(lib.lrb200_graph_set_superchunk(g, 0), "set_superchunk")
    _lib.check(lib.lrb200_graph_reset(g), "reset")
    return out


def _time_block(lib, _lib, torch, stream, h, xptr, n, yptr, steps):
    no = ctypes.c_size_t(0)
    for _ in range(3):
        _lib.check(lib.lrb200_block_execute(h, ctypes.c_void_p(xptr), n, ctypes.c_void_p(yptr), ctypes.byref(no)), "execute")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        _lib.check(lib.lrb200_block_execute(h, ctypes.c_void_p(xptr), n, ctypes.c_void_p(yptr), ctypes.byref(no)), "execute")
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_fir128(lib, _lib, torch, stream, args):
    """LowpassFilterBlock(128, 15e3) @ 220.5 kHz taps on white IQ resident in HBM: GB/s = 16 B * n / t."""
    import luaradio_b200 as radio
    n = args.fir_samples
    taps = np.array(radio.filter_utils.firwin_lowpass(128, 15e3 / 110250.0), np.float32)
    x = torch.empty(n, dtype=torch.complex64, device="cuda")
    y = torch.empty(n, dtype=torch.complex64, device="cuda")
    _lib.check(lib.lrb200_synth_white_iq(ctypes.c_void_p(x.data_ptr()), 0, n, 1), "synth")
    peak, _ = peaks()
    h = _lib.check_handle(lib.lrb200_fir_create_crcf(taps.ctypes.data, 128, 1, _lib.LRB200_DEVICE), "fir")
    ms = _time_block(lib, _lib, torch, stream, h, x.data_ptr(), n, y.data_ptr(), max(3, min(args.steps, 20)))
    gbs = ALG_BYTES_FIR * n / (ms * 1e-3) / 1e9
    out = {"workload": "LowpassFilterBlock(128,15e3) crcf, %d complex samples" % n, "ms": round(ms, 4),
           "msamples_per_s": round(n / (ms * 1e-3) / 1e6, 1), "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s",
           "frac": round(gbs / peak, 4), "algorithm": "fft-overlap-save" if lib.lrb200_fir_get_algorithm(h) == _lib.FIR_FFT else "direct"}
    lib.lrb200_fir_destroy(h)
    return out


def bench_cfg2(lib, _lib, torch, stream, args):
    """BASELINE.json configs[1]: FrequencyTranslator + 128-tap FIR + decimate-by-5 on 64 Mi white IQ samples, as a fused
    flow graph; complex taps (firwin_complex_bandpass) and the Tuner's real taps.  9.6 algorithmic bytes per input sample."""
    import luaradio_b200 as radio
    fu = radio.filter_utils
    n = 1 << 26
    D = _lib.LRB200_DEVICE
    x = torch.empty(n, dtype=torch.complex64, device="cuda")
    y = torch.empty(n // 5 + 16, dtype=torch.complex64, device="cuda")
    _lib.check(lib.lrb200_synth_white_iq(ctypes.c_void_p(x.data_ptr()), 0, n, 1), "synth")
    peak, _ = peaks()
    nyq = RATE / 2
    ctaps = np.array(fu.firwin_complex_bandpass(128, [-100e3 / nyq, 100e3 / nyq]), np.complex64)
    rtaps = np.array(fu.firwin_lowpass(128, 100e3 / nyq), np.float32)
    out = {"workload": "FrequencyTranslator(-250e3) > FIR(128) > Downsampler(5), %d white IQ samples" % n,
           "algorithmic_bytes_per_input_sample": ALG_BYTES_CFG2, "peak": peak, "unit": "GB/s"}
    for name, mk in (("complex_taps", lambda: lib.lrb200_fir_create_cccf(ctaps.ctypes.data, 128, 1, D)),
                     ("real_taps", lambda: lib.lrb200_fir_create_crcf(rtaps.ctypes.data, 128, 1, D))):
        g = _lib.check_handle(lib.lrb200_graph_create(), "graph")
        for h in (lib.lrb200_rotator_create(TUNE_OFFSET / RATE, D), mk(), lib.lrb200_downsample_create(5, 8, D)):
            _lib.check_handle(h, "block")
            _lib.check(lib.lrb200_graph_append(g, h), "append")
        _lib.check(lib.lrb200_graph_commit(g, 1), "commit")
        no = ctypes.c_size_t(0)

        def run():
            _lib.check(lib.lrb200_graph_execute_device(g, ctypes.c_void_p(x.data_ptr()), n, ctypes.c_void_p(y.data_ptr()), ctypes.byref(no)), "execute")
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        steps = max(3, min(args.steps, 20))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            run()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        gbs = ALG_BYTES_CFG2 * n / (ms * 1e-3) / 1e9
        out[name] = {"graph": lib.lrb200_graph_describe(g).decode(), "ms": round(ms, 4), "msamples_per_s": round(n / (ms * 1e-3) / 1e6, 1),
                     "achieved": round(gbs, 1), "frac": round(gbs / peak, 4)}
        lib.lrb200_graph_destroy(g)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle/lr_oracle.c): no GPU library involved
# ---------------------------------------------------------------------------------------------------------------------
def cpu_setup(n):
    from oracle import cbuild
    from oracle import lr_oracle as O
    olib = cbuild.load(native=True)
    cores = olib.lro_usable_cpus()
    x = np.empty(n, np.complex64)
    olib.lro_synth_fm_iq(x.ctypes.data, 0, n, 1, RATE, 250e3, 75e3, 0.5, 0.01, cores)
    return olib, O, cores, x


def cpu_chain_call(olib, x, n, taps, threads, use_fft, out):
    t1, t2, b, a = taps
    omega = 2 * math.pi * (TUNE_OFFSET / RATE)
    return olib.lro_wbfm_chain2(x.ctypes.data, n, 0, t1.ctypes.data, 128, 5, omega, 2 * math.pi * 1.25, t2.ctypes.data, 128,
                                b.ctypes.data, a.ctypes.data, 5, out.ctypes.data, threads, ORACLE_LEAD, use_fft)


def cpu_rate(olib, x, n, taps, threads, use_fft, out, min_seconds, max_reps=50):
    cpu_chain_call(olib, x, n, taps, threads, use_fft, out)
    reps, t0 = 0, time.perf_counter()
    while True:
        cpu_chain_call(olib, x, n, taps, threads, use_fft, out)
        reps += 1
        el = time.perf_counter() - t0
        if el >= min_seconds or reps >= max_reps:
            return n * reps / el / 1e6, el, reps


def cpu_baseline(args):
    """Both FIR algorithms of the reference's CPU path on this box's usable host cores, plus the single-thread rates."""
    n = args.cpu_samples
    olib, O, cores, x = cpu_setup(n)
    taps = chain_taps(O)
    out = np.zeros(n // 25 + 8, np.float32)
    algos = {}
    for name, fft in (("dot_product_volk", 0), ("overlap_save_fft", 1)):
        v, el, reps = cpu_rate(olib, x, n, taps, cores, fft, out, 4.0)
        v1, _, _ = cpu_rate(olib, x, min(n, 1 << 22), taps, 1, fft, out, 1.0)
        algos[name] = {"all_cores": round(v, 1), "one_thread": round(v1, 1), "seconds": round(el, 1), "reps": reps}
    best = max(algos, key=lambda k: algos[k]["all_cores"])
    return {"value": algos[best]["all_cores"], "unit": "Msamples/s", "cores": cores, "kind": "port", "algorithm": best,
            "algorithms": algos,
            "sample": "%d-sample synthetic FM IQ (same generator), whole chain, %d threads time-chunked with a %d-sample lead-in, "
                      ">= 4 s per algorithm" % (n, cores, ORACLE_LEAD),
            "note": "C port of the reference's CPU path: VOLK dot-product FIRs (firfilter.lua:111-163) and the overlap-save FIRs it "
                    "defaults to with FFTW (firfilter.lua:55-62,320-398; in-house FFT).  LuaJIT/VOLK/liquid/FFTW are not installable "
                    "here; the published reference number for the FIR is 133.85 MS/s per core (2013 i5, FFTW)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = ((args.samples if args.samples else WORKLOADS["wbfm_mono_256Mi"]) // 25) * 25
    olib, O, cores, x = cpu_setup(n)
    taps = chain_taps(O)
    out = np.zeros(n // 25 + 8, np.float32)
    # pick the faster of the reference's two FIR algorithms on a 16 Mi-sample trial
    trial = min(n, 1 << 24)
    rates = {}
    for name, fft in (("dot_product_volk", 0), ("overlap_save_fft", 1)):
        rates[name] = cpu_rate(olib, x, trial, taps, cores, fft, out, 0.5, 4)[0]
    best = max(rates, key=rates.get)
    fft = 1 if best == "overlap_save_fft" else 0
    steps = args.steps
    warm = max(3, args.warmup)
    for _ in range(warm):
        cpu_chain_call(olib, x, n, taps, cores, fft, out)
    t0 = time.perf_counter()
    for _ in range(steps):
        n_out = cpu_chain_call(olib, x, n, taps, cores, fft, out)
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "audio", out[:n_out], DUMP_BYTES)
    v = n * steps / el / 1e6
    emit(json.dumps({
        "impl": "reference", "metric": METRIC,
        "value": round(v, 1), "unit": "Msamples/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": round(el / steps * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "wbfm_mono_256Mi" if n == 268435450 else "wbfm_mono_%d" % n, "samples_per_gpu": n, "total_samples": n,
                   "sample_rate_hz": RATE, "chain": CHAIN, "algorithm": best, "trial_msamples_per_s": {k: round(r, 1) for k, r in rates.items()}},
        "cpu_baseline": {"value": round(v, 1), "unit": "Msamples/s", "cores": cores, "kind": "port", "algorithm": best,
                         "sample": "%d-sample synthetic FM IQ per step (the full workload), whole chain, %d threads time-chunked" % (n, cores)},
        "e2e": {"value": round(v, 1), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


_RESULT_OUT = None


def emit(line):
    """The one JSON line goes to the process's ORIGINAL stdout; see main()."""
    out = _RESULT_OUT or sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    # Libraries write to fd 1 behind Python's back (NCCL prints "NCCL version ..." there at init): keep a private copy of
    # the real stdout for the result line and point fd 1 at stderr for everything else.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="wbfm_mono_256Mi", choices=sorted(WORKLOADS))
    ap.add_argument("--samples", type=int, default=0, help="override the workload's sample count (per GPU for the weak workload)")
    ap.add_argument("--fir-samples", type=int, default=1 << 28)
    ap.add_argument("--cpu-samples", type=int, default=1 << 26)
    ap.add_argument("--halo", default="ipc", choices=["ipc", "nccl"], help="N > 1: transport of the halo exchange")
    ap.add_argument("--no-check", action="store_true", help="skip the oracle window check of the run's output")
    ap.add_argument("--check", action="store_true", help="(default) compare output windows with the oracle and fail on mismatch")
    ap.add_argument("--profile", action="store_true", help="profiling run (ncu): skip the e2e, FIR-128 sweep and CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
