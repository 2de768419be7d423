#!/usr/bin/env python
"""bench.py — render-quanta/sec of the OfflineAudioContext hot path on N B200s (one process per GPU).

Workload (BASELINE.json configs[1], "C2"): 1000 independent OfflineAudioContexts per GPU, each
AudioBufferSource(stereo, seeded uniform noise) -> BiquadFilter(lowpass, seeded f0/Q) -> Gain -> destination,
48 kHz stereo, 10 s (3750 render quanta of 128 frames).  A "step" = one render of the whole batch.
  value    : graph-quanta/s, kernel-only (batch prepared once, source PCM resident in HBM), CUDA events on the engine's stream
  e2e      : the ONE-SHOT plugin call, every step on freshly built graphs: wae_render_batch(engine, graphs, n, out, HOST) —
             sizing + planning + H2D of the source PCM + render + D2H into the caller's pageable buffer, all inside the timed call
             (what `start_rendering_sync` is for a batch of contexts; a context can be rendered only once, offline.rs:163)
  e2e_pinned_out / e2e_warm : the same call with a page-locked `out`; re-renders of an already prepared batch (H2D + render + D2H)
  roofline / cpu_baseline   : see DESIGN.md "Measurement"
Multi-GPU (torchrun): graphs are sharded by rank, no data-path collective in C2.  The other BASELINE configs run too: C3 / C4 /
north_star / C5 at N=1 (fixed per-GPU sizes), C4 as "512 graphs, 2/4 GPU shard" at N=2,4 and C5 as "2048 graphs, 8 GPU, NCCL
gather" at N=8, both also WITH the gather of the rendered PCM inside the step (all-gather of group k overlapped with the render of
group k+1).
--impl reference times the reference's CPU algorithm (the oracle port, all host threads) on the same config and batch size.
Every timed leg runs --steps steps.  --dump-outputs DIR writes a seeded sample of the C2 PCM the last timed step rendered
(DIR/c2_pcm.npy): the inputs are the same on every run, so two builds can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 48000.0
METRIC = "offline render-quanta/sec (48kHz stereo, 128-frame)"
FP64_PEAK_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12  # B200 non-tensor FP64 (nominal)
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # B200 non-tensor FP32: 148 SMs x 128 lanes x FMA at the 1965 MHz boost clock
PARKING_GARAGE_IR_FRAMES = 178899  # samples/parking-garage-response.wav (164 363 frames @ 44.1 kHz) resampled to 48 kHz (SURVEY §8a a9)
DUMP_BYTES = 64 * 10**6  # --dump-outputs: at most this much PCM on disk


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm_sorted = sorted(sm)
        # median of the samples under load (upper half: idle samples before/after the region pull it down)
        med = sm_sorted[len(sm_sorted) * 3 // 4] if sm_sorted else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


class Dist:
    """rank / world plumbing shared by the legs (NCCL process group when world > 1)."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))

    def init(self):
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, v):
        import torch
        import torch.distributed as dist
        if self.world == 1:
            return float(v)
        t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        import torch.distributed as dist
        if self.world > 1:
            dist.destroy_process_group()


def conv_model(n_graphs, length, ir_frames, in_ch=2, paths=2):
    """Bytes / flops of the TIME-BATCHED convolution the engine runs (SURVEY §8d "time-batched alternative"): overlap-save with
    8192-frame partitions, one real FFT of 16384 per input block, S8 = ceil(ir / 8192) spectrum MACs per output block and path.
    Compulsory HBM bytes of that algorithm = input PCM + output PCM (spectra could stay on chip); flops: 5 N log2 N per complex FFT
    of N = 8192 plus ~10 flops per bin of real-FFT post-processing, 8 flops per complex MAC."""
    blocks = (length + 8191) // 8192
    s8 = (ir_frames + 8191) // 8192
    fft = 5 * 8192 * 13 + 10 * 8192
    flops = n_graphs * blocks * (in_ch * fft + paths * (s8 * 8192 * 8 + fft))
    bytes_io = n_graphs * (in_ch + paths) * length * 4
    return {"blocks_per_graph": blocks, "ir_partitions_8192": s8, "ir_partitions_1024_reference": (ir_frames + 1023) // 1024,
            "flops": flops, "compulsory_bytes": bytes_io}


def add_models(a, b2):
    """Two convolution stages of one graph (C5: the ConvolverNode and the static HRTF panner lowered to the same kernels)."""
    out = dict(a)
    out["flops"] = a["flops"] + b2["flops"]
    out["compulsory_bytes"] = a["compulsory_bytes"] + b2["compulsory_bytes"]
    out["second_convolution"] = {k: b2[k] for k in ("blocks_per_graph", "ir_partitions_8192", "flops", "compulsory_bytes")}
    return out


def measure_workload(pkg, eng, D, oracle, name, build, n_gpu, n_cpu, length, steps, cores, note, model=None, gather=False, groups=0):
    """One additional BASELINE workload: kernel-only (max over ranks), one-shot e2e, optional NCCL gather inside the step, CPU port."""
    import torch
    import torch.distributed as dist
    ctxs = [build(eng.backend, g) for g in range(n_gpu)]
    eng.set_option(pkg.OPT_PIPELINE_GROUPS, groups if gather else 1)
    batch = pkg.Batch(ctxs)
    st = batch.stats()
    batch.set_timing(True)
    for _ in range(3):
        batch.run()
    batch.sync()
    ms = []
    for _ in range(steps):
        D.barrier()
        batch.run()
        batch.sync()
        ms.append(D.max(batch.stats().last_run_ms))
    stages = {}
    for n, t, _k in batch.stage_times():
        stages[n] = stages.get(n, 0.0) + t
    batch.set_timing(False)
    quanta = n_gpu * ((length + 127) // 128) * D.world
    med = float(np.median(ms))
    out = {"workload": name, "note": note, "graphs_per_gpu": n_gpu, "graphs_total": n_gpu * D.world, "frames_per_graph": length,
           "steps": steps, "ms_per_step": med, "value": quanta / (med * 1e-3), "unit": "graph-quanta/s",
           "kernel_launches_per_step": int(st.kernel_launches_per_run), "chunks": int(st.chunks),
           "stages_ms_per_step": {k: round(v, 4) for k, v in stages.items()}}
    # ---- the NCCL gather of the rendered PCM INSIDE the step (north_star): all-gather of group k's PCM on a side stream while
    # group k+1 renders; every rank ends the step holding the PCM of all ranks (layout [group][rank][graphs of the group][ch][len])
    if gather and D.world > 1:
        p, _nfl = batch.device_ptr()

        class _W:  # the engine's output buffer as a torch tensor (CUDA array interface, no copy)
            __cuda_array_interface__ = {"shape": (n_gpu, 2, length), "typestr": "<f4", "data": (p, False), "version": 2}
        shard = torch.as_tensor(_W(), device="cuda")
        groups_r = batch.groups()
        full = [torch.empty((D.world, g1 - g0, 2, length), dtype=torch.float32, device="cuda") for g0, g1 in groups_r]
        comm = torch.cuda.Stream()
        eng_stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", D.local_rank))

        def step_with_gather():
            evs = []
            for k, (g0, g1) in enumerate(groups_r):
                batch.run_group(k)
                ev = torch.cuda.Event()
                ev.record(eng_stream)
                comm.wait_event(ev)
                with torch.cuda.stream(comm):
                    pkg.parallel.all_gather_group(full[k], shard[g0:g1])
            comm.synchronize()
            batch.sync()

        for _ in range(2):
            step_with_gather()
        tg = []
        for _ in range(steps):
            D.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(eng_stream)
            step_with_gather()
            e1.record(comm)
            torch.cuda.synchronize()
            tg.append(D.max(e0.elapsed_time(e1)))
        # the gather alone (no render to hide behind), same buffers
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(comm):
            e0.record(comm)
            for k, (g0, g1) in enumerate(groups_r):
                pkg.parallel.all_gather_group(full[k], shard[g0:g1])
            e1.record(comm)
        torch.cuda.synchronize()
        alone = D.max(e0.elapsed_time(e1))
        ok = bool(torch.equal(full[0][D.rank], shard[groups_r[0][0]:groups_r[0][1]]))
        gm = float(np.median(tg))
        out["with_nccl_gather"] = {"ms_per_step": gm, "value": quanta / (gm * 1e-3), "gather_alone_ms": alone, "groups": len(groups_r),
                                   "gathered_bytes_per_gpu": int(n_gpu * D.world * 2 * length * 4), "own_shard_round_trips": ok,
                                   "how": "all_gather_into_tensor per graph group on a side stream, overlapped with the render of the next group"}
        del full
    # ---- one-shot e2e: fresh graphs, one wae_render_batch(HOST) call, pageable out
    host = np.zeros((n_gpu, 2, length), np.float32)
    eng.set_option(pkg.OPT_PIPELINE_GROUPS, 0)
    e2e = []
    for i in range(1 + steps):
        fresh = [build(eng.backend, g) for g in range(n_gpu)]
        D.barrier()
        t0 = time.perf_counter()
        pkg.render_batch_oneshot(fresh, host)
        e2e.append(D.max(time.perf_counter() - t0))
        del fresh
    e2e_s = float(np.median(e2e[1:]))
    out["e2e_value"] = quanta / e2e_s
    out["e2e_ms_per_step"] = e2e_s * 1e3
    out["e2e_how"] = f"one wae_render_batch(HOST) call on fresh graphs, pageable out, median of {steps} after 1 warm-up"
    if model is not None:
        out["time_batched_model"] = model
    if oracle is not None and n_cpu > 0 and D.rank == 0:
        octx = [build(oracle, g) for g in range(n_cpu)]
        arr = (ctypes.c_void_p * n_cpu)(*[c._g for c in octx])
        ref = np.empty((n_cpu, 2, length), np.float32)
        secs = ctypes.c_double()
        oracle.api.check(oracle.api.render_many(arr, n_cpu, ref.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), min(cores, n_cpu), ctypes.byref(secs)))
        got = host[:n_cpu]
        out["cpu_port"] = {"value": n_cpu * ((length + 127) // 128) / secs.value, "cores_used": min(cores, n_cpu),
                           "sample": f"{n_cpu} graphs, {secs.value:.2f} s wall", "max_abs_diff_vs_gpu": float(np.abs(got - ref).max()),
                           "ref_abs_max": float(np.abs(ref).max())}
        # the batch the kernel-only figure was timed on may be lowered differently from the one-shot call's one-graph groups (k_voice_sum
        # needs a whole group's work items): check its PCM as well
        timed = batch.fetch()[:n_cpu]
        out["cpu_port"]["max_abs_diff_vs_timed_batch"] = float(np.abs(timed - ref).max())
        del timed
    batch.destroy()
    return out


def kernel_rooflines(w, peak_gbs):
    """Per dominant kernel of a workload: achieved rate against the bound that applies to it."""
    m = w.get("time_batched_model")
    st = w["stages_ms_per_step"]
    res = []
    if m:
        conv_ms = sum(v for k, v in st.items() if k.startswith("k_conv"))
        if conv_ms > 0:
            tf = m["flops"] / (conv_ms * 1e-3) / 1e12
            gbs = m["compulsory_bytes"] / (conv_ms * 1e-3) / 1e9
            res.append({"kernels": "k_conv_fft_in + k_conv_mac_ifft", "ms": round(conv_ms, 4), "bound": "fp32 (FFT butterflies + spectrum MACs)",
                        "achieved_tflops": tf, "peak_tflops": FP32_PEAK_TFLOPS, "frac": tf / FP32_PEAK_TFLOPS,
                        "hbm_gbs_vs_compulsory_io": gbs, "hbm_frac": gbs / peak_gbs})
    vf = w.get("voice_frames")
    if vf:
        # oscillator -> biquad voices: SURVEY §8(d) counts 0 HBM bytes for them (state in registers), so the bound is arithmetic.  Model: the
        # biquad of one voice frame = 3 feed-forward + 2 x 2 recurrence DFMA (the time-parallel scan runs the recurrence twice) = 14 f64
        # flops; oscillator, conversions and the warp scan come on top and are not counted.  Peak: 148 SMs x 64 f64 lanes x FMA at 1965 MHz
        # (nominal, not in MEASURED_PEAKS.json).
        names = [k for k in st if k in ("k_voice_sum", "k_chain", "k_mix")]
        ms = sum(st[k] for k in names)
        if ms > 0:
            tf = vf * 14 / (ms * 1e-3) / 1e12
            res.append({"kernels": " + ".join(names), "ms": round(ms, 4), "bound": "issue slots / f64 pipe (no compulsory HBM bytes)",
                        "voice_frames_per_s": vf / (ms * 1e-3), "achieved_tflops": tf, "peak_tflops": FP64_PEAK_TFLOPS, "frac": tf / FP64_PEAK_TFLOPS,
                        "peak_source": "nominal"})
    return res


def run_extra_workloads(pkg, eng, D, oracle, cores, steps, peak_gbs):
    import graphs as G
    res = []
    ir = G.synthetic_ir(PARKING_GARAGE_IR_FRAMES, 2, decay=0.6)  # synthetic response of the parking-garage IR's length: 175 partitions of 1024
    # the reference's IRC_1003_C sphere (44.1 kHz, 512 taps, 187 vertices) cannot travel: synthetic data of the same rate and size,
    # resampled to the 48 kHz context rate by the library exactly as the embedded one would be (~417 taps)
    sphere = G.synthetic_hrir_sphere(44100, 512)
    eng.backend.set_hrir_sphere(sphere)
    if oracle is not None:
        oracle.set_hrir_sphere(sphere)
    c5_len = 240000

    def c4(be, g):
        return G.c4_convolver(pkg, be, g + D.rank * 100000, 480000, ir)

    def c5(be, g):
        return G.c5_full_chain(pkg, be, g + D.rank * 100000, c5_len, ir, curve_points=1024)

    if D.world == 1:
        res.append(measure_workload(pkg, eng, D, oracle, "C3", lambda be, g: G.c3_many_voices(pkg, be, 4096, 48000), 1, 1, 48000, steps, cores,
                                    "configs[2]: ONE graph, 4096 x (Oscillator -> Biquad) summed in reference order at the destination, 1 s"))
        res.append(measure_workload(pkg, eng, D, oracle, "C4", c4, 128, min(cores, 128), 480000, steps, cores,
                                    "configs[3] at 128 graphs/GPU (the 4-GPU share of 512): stereo source -> Convolver(3.73 s stereo IR = 175 "
                                    "partitions of 1024, normalize) -> destination, 10 s", model=conv_model(128, 480000, PARKING_GARAGE_IR_FRAMES)))
        res.append(measure_workload(pkg, eng, D, oracle, "north_star", lambda be, g: G.north_star_voices_convolver(pkg, be, 1000, 480000, ir, seed=g),
                                    8, 8, 480000, steps, cores,
                                    "north_star: 8 graphs/GPU, each 1000 voices (Oscillator -> Biquad -> Gain) summed into one Convolver -> destination, 10 s",
                                    model=conv_model(8, 480000, PARKING_GARAGE_IR_FRAMES, in_ch=1, paths=2)))
        res.append(measure_workload(pkg, eng, D, oracle, "C5", c5, 256, min(cores, 64), c5_len, steps, cores,
                                    "configs[4] per-GPU share (2048 graphs / 8 GPUs): Oscillator -> WaveShaper(1024-pt tanh) -> Biquad -> Convolver -> "
                                    "Panner(HRTF, 44.1 kHz / 512-tap sphere resampled to 48 kHz) -> Analyser -> destination, 5 s; HRTF parity is UNPINNED "
                                    "(hrtf crate absent from the reference tree, SURVEY §8c)", model=add_models(conv_model(256, c5_len, PARKING_GARAGE_IR_FRAMES, in_ch=1, paths=2), conv_model(256, c5_len, 558, in_ch=2, paths=4))))
    elif D.world > 1 and os.environ.get("WAE_BENCH_EXTRA") == "c5_small":  # validation of the N = 8 leg on fewer GPUs (not a BASELINE size)
        res.append(measure_workload(pkg, eng, D, None, "C5", c5, 32, 0, c5_len, steps, cores,
                                    "configs[4] path check: 32 graphs per GPU, with the NCCL gather inside the step", gather=True, groups=4))
    elif D.world in (2, 4):
        n = 512 // D.world
        res.append(measure_workload(pkg, eng, D, None, "C4", c4, n, 0, 480000, steps, cores,
                                    f"configs[3]: 512 graphs sharded over {D.world} GPUs ({n} per GPU): stereo source -> Convolver(175-partition stereo IR, "
                                    "normalize) -> destination, 10 s; also with the NCCL gather of the PCM inside the step",
                                    model=conv_model(n, 480000, PARKING_GARAGE_IR_FRAMES), gather=True, groups=8))
    elif D.world == 8:
        res.append(measure_workload(pkg, eng, D, None, "C5", c5, 256, 0, c5_len, steps, cores,
                                    "configs[4]: 2048 graphs over 8 GPUs (256 per GPU), full chain with HRTF panner (parity unpinned, SURVEY §8c), 5 s; also "
                                    "with the NCCL gather of the PCM inside the step", model=add_models(conv_model(256, c5_len, PARKING_GARAGE_IR_FRAMES, in_ch=1, paths=2), conv_model(256, c5_len, 558, in_ch=2, paths=4)),
                                    gather=True, groups=8))
    for w in res:
        if w["workload"] == "north_star":
            w["voice_frames"] = w["graphs_per_gpu"] * 1000 * w["frames_per_graph"]
        elif w["workload"] == "C3":
            w["voice_frames"] = 4096 * w["frames_per_graph"]
        w["kernel_rooflines"] = kernel_rooflines(w, peak_gbs)
    return res


def c2_config(n_graphs, length, seconds):
    """The `config` object of BOTH arms (ours and --impl reference): same workload, same batch per GPU / per step."""
    return {"workload": "C2 (BASELINE configs[1]): %d OfflineAudioContexts per GPU (per step for the CPU arm), AudioBufferSource->Biquad->Gain->"
                        "destination, 48 kHz stereo, %.0f s each" % (n_graphs, seconds),
            "graphs_per_gpu": n_graphs, "graphs_per_step": n_graphs, "frames_per_graph": length,
            "l2": "inputs (%.2f GB of source PCM per GPU) larger than L2, no flush" % (n_graphs * 2 * length * 4 / 1e9),
            "sharding": "independent graphs per rank, no data-path collective"}


def load_oracle_only():
    """The checker / CPU arm without mapping the product library: package python + oracle/_build/liboracle.so."""
    import __graft_entry__ as ge
    if not os.path.exists(ge.ORACLE_SO):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-j8"], stdout=subprocess.DEVNULL)
    pkg = ge.load_package()
    return pkg, pkg.context.Backend(pkg.Api(ctypes.CDLL(ge.ORACLE_SO), "wao_"))


def build_c2_batch(pkg, backend, n_graphs, length, seed_base=0, pcm=None):
    import graphs as G
    return [G.c2_buffer_biquad_gain(pkg, backend, seed_base + g, length, pcm=None if pcm is None else pcm[g]) for g in range(n_graphs)]


def dump_pcm(out_dir, pcm):
    """--dump-outputs: the PCM of the last timed step, [graphs][2][length] float32 as the caller receives it.  At C2 size that is
    3.84 GB, so whole graphs are sampled, the same seeded choice on every run, up to DUMP_BYTES."""
    per_graph = pcm[0].nbytes
    k = min(len(pcm), max(1, (DUMP_BYTES - 4096) // per_graph))  # 4096: room for the .npy header
    pick = np.sort(np.random.default_rng(0).choice(len(pcm), k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "c2_pcm.npy"), pcm[pick])


def run_reference(args, D):
    """--impl reference: the reference's CPU path (oracle port: the Rust crate cannot be built here, no cargo), same config and the
    same number of graphs per step as the GPU arm, all host threads, one context per worker thread."""
    if D.rank != 0:
        return
    pkg, oracle = load_oracle_only()
    import graphs as G
    cores = os.cpu_count() or 1
    length = int(args.seconds * SR)
    n = args.graphs
    quanta_per_graph = (length + 127) // 128
    pcm = [G.c2_source(g, length) for g in range(n)]
    out = np.empty((n, 2, length), np.float32)
    times = []
    for step in range(args.warmup + args.steps):
        ctxs = build_c2_batch(pkg, oracle, n, length, pcm=pcm)  # fresh contexts every step (a context renders once)
        arr = (ctypes.c_void_p * n)(*[c._g for c in ctxs])
        secs = ctypes.c_double()
        oracle.api.check(oracle.api.render_many(arr, n, out.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), cores, ctypes.byref(secs)))
        if step >= args.warmup:
            times.append(secs.value)
        del ctxs
    if args.dump_outputs:
        dump_pcm(args.dump_outputs, out)
    t = float(np.mean(times))
    value = n * quanta_per_graph / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "graph-quanta/s", "n_gpus": D.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 filter state / f32 PCM", "data": "synthetic",
        "config": c2_config(n, length, args.seconds),
        "cpu_baseline": {"value": value, "unit": "graph-quanta/s", "cores": cores, "kind": "port",
                         "sample": f"{n} graphs x {args.seconds:.0f} s per step (the GPU arm's per-GPU batch), one context per worker thread"},
        "e2e": {"value": value, "unit": "graph-quanta/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--graphs", type=int, default=1000, help="graphs per GPU (C2: 1000)")
    ap.add_argument("--seconds", type=float, default=10.0, help="rendered seconds per graph (C2: 10)")
    ap.add_argument("--cpu-sample-graphs", type=int, default=512)
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--groups", type=int, default=32, help="graph groups of the warm e2e pipeline (H2D | render | D2H overlap)")
    ap.add_argument("--serial-filters", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bind-numa", type=int, default=1, help="bind every rank's host threads to its GPU's NUMA node (pinned memory local to the GPU)")
    ap.add_argument("--kernel-only", action="store_true", help="tuning runs: only the kernel-only leg of C2 (no e2e legs, no other workloads)")
    ap.add_argument("--extra", type=int, default=1, help="also measure the other BASELINE configs (C3 / C4 / north_star / C5 at N=1; C4 at N=2,4; C5 at N=8)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the PCM the last timed step rendered (rank 0; the "
                                                          "kernel-only leg of C2) to DIR/c2_pcm.npy, so that two builds can be compared output for output")
    args = ap.parse_args()

    D = Dist()
    if args.impl == "reference":
        run_reference(args, D)
        return

    import torch
    import __graft_entry__ as ge
    import graphs as G

    pkg = ge.build()
    D.init()
    rank, local_rank, world = D.rank, D.local_rank, D.world
    all_cpus = os.sched_getaffinity(0)
    eng = pkg.Engine(local_rank)
    numa = None
    if args.bind_numa:
        try:
            eng.set_option(pkg.OPT_BIND_NUMA, 1)
            numa = sorted(os.sched_getaffinity(0))
        except pkg.WaeError:
            numa = None
    eng.set_option(pkg.OPT_CHUNK_FRAMES, args.chunk)
    eng.set_option(pkg.OPT_SERIAL_FILTERS, args.serial_filters)
    length = int(args.seconds * SR)
    quanta_per_graph = (length + 127) // 128
    n_graphs = args.graphs
    total_quanta = n_graphs * quanta_per_graph * world

    # ---- the graphs: different seeds per rank (independent shards, weak scaling).  The source PCM is generated once; graphs are
    # rebuilt from it for every one-shot step (wae_create_buffer_source copies it into the library's page-locked pool).
    seed_base = rank * n_graphs
    pcm = [G.c2_source(seed_base + g, length) for g in range(n_graphs)]
    eng.set_option(pkg.OPT_PIPELINE_GROUPS, 1)
    ctxs = build_c2_batch(pkg, eng.backend, n_graphs, length, seed_base=seed_base, pcm=pcm)
    batch = pkg.Batch(ctxs)  # un-grouped: every stage is ONE launch over all graphs (the clean kernel-only / roofline measurement)
    stats0 = batch.stats()
    out_floats = n_graphs * 2 * length
    pinned_out = torch.empty(out_floats, dtype=torch.float32, pin_memory=True)
    pinned_view = pinned_out.numpy().reshape(n_graphs, 2, length)
    pageable_out = np.zeros((n_graphs, 2, length), np.float32)  # the caller's buffer of the one-shot call (touched once here)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))

    def timed(fn, steps):
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        batch.sync()
        D.barrier()
        wall = time.perf_counter() - t0
        return D.max(e0.elapsed_time(e1)), wall

    # ---- kernel-only: inputs resident in HBM (3.84 GB of source PCM per 1000 graphs >> 126 MB L2: every step
    # streams its inputs from HBM again, no explicit L2 flush needed)
    batch.set_timing(True)
    for _ in range(args.warmup):
        batch.run()
    batch.sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total, _ = timed(batch.run, args.steps)
    clocks = sampler.stop()
    stage_times = batch.stage_times()  # last run of the timed region
    stats = batch.stats()
    ms_per_step = ms_total / args.steps
    value = total_quanta / (ms_per_step * 1e-3)
    batch.set_timing(False)
    batch.sync()
    if args.dump_outputs and rank == 0:
        dump_pcm(args.dump_outputs, batch.fetch())
    if args.kernel_only:
        agg = {}
        for name, ms, _n in stage_times:
            agg[name] = agg.get(name, 0.0) + ms
        if rank == 0:
            peak = load_peaks()[0]
            k_ms = max(agg.values()) if agg else 0.0
            print(json.dumps({"kernel_only": True, "ms_per_step": ms_per_step, "kernel_ms": k_ms,
                              "frac": 2048 * n_graphs * quanta_per_graph / (k_ms * 1e-3) / 1e9 / peak if k_ms else None, "clocks": clocks}))
        batch.destroy()
        eng.close()
        D.close()
        return

    # ---- e2e, the one-shot plugin call: fresh graphs every step, ONE wae_render_batch(engine, graphs, n, out, HOST)
    eng.set_option(pkg.OPT_PIPELINE_GROUPS, 0)  # the library's own choice of graph groups

    def oneshot(out_array, n_steps, n_warm):
        walls = []
        for i in range(n_warm + n_steps):
            fresh = build_c2_batch(pkg, eng.backend, n_graphs, length, seed_base=seed_base, pcm=pcm)
            D.barrier()
            t0 = time.perf_counter()
            pkg.render_batch_oneshot(fresh, out_array)
            torch.cuda.synchronize()
            dt = D.max(time.perf_counter() - t0)
            if i >= n_warm:
                walls.append(dt)
            del fresh
        return walls

    e2e_walls = oneshot(pageable_out, args.steps, max(1, min(args.warmup, 2)))
    e2e_s = float(np.mean(e2e_walls))
    e2e_pinned_walls = oneshot(pinned_view, args.steps, 1)
    e2e_pinned_s = float(np.mean(e2e_pinned_walls))
    h2d = stats.asset_bytes * world  # whole job, like `value`: every rank copies its own shard over its own PCIe link
    d2h = out_floats * 4 * world

    # ---- e2e_warm: re-renders of a prepared batch (H2D of the pinned source PCM + render + D2H into pinned memory, per group)
    eng.set_option(pkg.OPT_PIPELINE_GROUPS, args.groups)
    t_prep = time.perf_counter()
    batch_e2e = pkg.Batch(ctxs)
    prepare_ms = (time.perf_counter() - t_prep) * 1e3
    pinned_ptr = ctypes.c_void_p(pinned_out.data_ptr())
    batch_e2e.run_pipelined(pinned_ptr)
    _, warm_wall = timed(lambda: batch_e2e.run_pipelined(pinned_ptr), args.steps)
    warm_s = D.max(warm_wall / args.steps)
    batch_e2e.destroy()

    # ---- roofline of the dominant kernel (CUDA events around every stage launch, on the launching stream)
    peak, peak_src = load_peaks()
    agg, launches_of = {}, {}
    for name, ms, _n in stage_times:  # one entry per (graph group, stage): aggregate by kernel
        agg[name] = agg.get(name, 0.0) + ms
        launches_of[name] = launches_of.get(name, 0) + int(stats.chunks)
    dom_name = max(agg, key=agg.get) if agg else ""
    dom = (dom_name, agg.get(dom_name, 0.0), 0)
    n_chunks = launches_of.get(dom_name, 1)
    # SURVEY §8(d): C2 = 2048 B per graph-quantum (1024 B source read + 1024 B destination write); one launch of the
    # dominant kernel covers all graphs of the batch for one chunk
    alg_bytes_step = 2048 * n_graphs * quanta_per_graph
    alg_bytes_launch = alg_bytes_step / n_chunks
    dom_ms_launch = dom[1] / n_chunks if n_chunks else 0.0
    achieved = alg_bytes_launch / (dom_ms_launch * 1e-3) / 1e9 if dom_ms_launch > 0 else 0.0
    # DRAM traffic of the same launch from an `ncu` capture of this very command (measured/dram_traffic.json, written by
    # tools/record_traffic.py on the GPU box); null when no capture matches the workload size
    traffic = None
    try:
        rec = json.load(open(os.path.join(ROOT, "web-audio-api-rs_b200", "measured", "dram_traffic.json")))
        if rec.get("kernel") == dom[0] and rec.get("graphs") == n_graphs and rec.get("frames_per_graph") == length:
            traffic = rec["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes_launch,
                "kernel_ms_per_launch": dom_ms_launch, "kernel_share_of_step": dom[1] / ms_per_step if ms_per_step else None,
                "step_achieved_gbs": alg_bytes_step / (ms_per_step * 1e-3) / 1e9,
                "launches_per_step": n_chunks, "stages_ms_per_step": {n: round(ms, 4) for n, ms in agg.items()}}

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample of the same workload (rank 0, N=1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)  # the CPU arm gets every host thread, not just the GPU's NUMA node
        oracle = pkg.context.Backend(pkg.Api(ctypes.CDLL(ge.ORACLE_SO), "wao_"))
        cores = len(all_cpus)
        ns = min(args.cpu_sample_graphs, n_graphs)  # bounded sample of the same workload
        out = np.empty((ns, 2, length), np.float32)
        secs = ctypes.c_double()
        walls = []
        for _ in range(3):  # the sample takes well under a second on a many-core host: median of three fresh renders
            octx = build_c2_batch(pkg, oracle, ns, length, pcm=pcm)
            arr = (ctypes.c_void_p * ns)(*[c._g for c in octx])
            oracle.api.check(oracle.api.render_many(arr, ns, out.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), cores, ctypes.byref(secs)))
            walls.append(secs.value)
        wall = float(np.median(walls))
        cpu_baseline = {"value": ns * quanta_per_graph / wall, "unit": "graph-quanta/s", "cores": cores, "kind": "port",
                        "sample": f"{ns} graphs x {args.seconds:.0f} s of the same workload, one context per worker thread, "
                                  f"median of 3 renders: {wall:.3f} s wall ({ns * wall:.1f} core-seconds upper bound)"}
        # parity spot check of the bench output itself (the one-shot call's pageable buffer) against the oracle
        cpu_baseline["max_abs_diff_vs_gpu"] = float(np.abs(pageable_out[:ns] - out).max())
        cpu_baseline["oneshot_pinned_equals_pageable"] = bool(np.array_equal(pageable_out, pinned_view))
        if numa:
            os.sched_setaffinity(0, set(numa))

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "graph-quanta/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 filter state / f32 PCM", "data": "synthetic",
            "config": c2_config(n_graphs, length, args.seconds),
            "engine": {"chunk_frames": int(stats0.chunks and (length + 127) // 128 * 128 // stats0.chunks),
                       "source_pcm_gb_per_gpu": stats.asset_bytes / 1e9,
                       "numa_bound_cpus": (f"{numa[0]}..{numa[-1]} ({len(numa)} CPUs)" if numa else None)},
            "samples_per_sec": value * 128, "gpu_launches": int(stats.kernel_launches_per_run) * args.steps,
            "clocks": clocks,
            "e2e": {"value": total_quanta / e2e_s, "unit": "graph-quanta/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_s * 1e3, "steps": len(e2e_walls), "ms_each": [round(w * 1e3, 2) for w in e2e_walls],
                    "how": "one wae_render_batch(engine, graphs, n, out, HOST) call per step on freshly built graphs: sizing + planning + H2D of "
                           "the source PCM (page-locked AudioBuffer memory owned by the graphs) + render + D2H into the caller's PAGEABLE "
                           "buffer (page-locked staging slots + copy-out threads); wall clock around the call, max over ranks"},
            "e2e_pinned_out": {"value": total_quanta / e2e_pinned_s, "unit": "graph-quanta/s", "ms_per_step": e2e_pinned_s * 1e3,
                               "how": "the same call with a page-locked `out` (D2H lands in it directly)"},
            "e2e_warm": {"value": total_quanta / warm_s, "unit": "graph-quanta/s", "ms_per_step": warm_s * 1e3, "groups": args.groups,
                         "prepare_ms_once": prepare_ms,
                         "how": "wae_batch_run_pipelined on an already prepared batch (H2D + render + D2H per group, page-locked both ends)"},
            "roofline": roofline, "cpu_baseline": cpu_baseline,
        }
    batch.destroy()
    del ctxs, pinned_view, pinned_out, pageable_out
    if args.extra:
        oracle2 = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)
            oracle2 = pkg.context.Backend(pkg.Api(ctypes.CDLL(ge.ORACLE_SO), "wao_"))
        extra = run_extra_workloads(pkg, eng, D, oracle2, len(all_cpus), args.steps, load_peaks()[0])
        if line is not None:
            line["other_workloads"] = extra
    if line is not None:
        print(json.dumps(line))
    eng.close()
    D.close()


if __name__ == "__main__":
    main()
