#!/usr/bin/env python
"""bench.py — headline throughput of the fundsp_b200 voice-bank hot path (contract in the task brief).

A "step" renders `--seconds` of audio (48 kHz, block 64) for the workload's voice bank on every GPU and mixes
it down to the voice's channel count — the `Wave::render` loop over "a Vec of V units + a sum" (SURVEY.md §3.6).
  value   Msamples/s = voices x samples / time, whole job, device-resident result (CUDA events, max over ranks)
  e2e     same metric through the public C-ABI call `fdsp_bank_render` with HOST buffers (D2H of the mix inside
          the timed region; generators have no audio input, so h2d is 0 bytes unless the workload has a gate)
  roofline / cpu_baseline / clocks / gpu_launches as the contract asks.
`--impl reference` times the reference's CPU algorithm (the C++ oracle, all host threads) on the same config.
Multi-GPU: one process per GPU (torchrun), voices sharded contiguously (weak scaling: V per GPU), the per-GPU
stereo/mono partial mixes are summed with one NCCL reduce per step (SURVEY.md §8e).
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True   # the tree may be read-only: no __pycache__ from the modules imported below
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SR = 48000.0
def _baseline_metric():
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "Msamples/sec (f32) rendered across N voices at 1/2/4/8 B200 vs host-CPU ref"


METRIC = _baseline_metric()   # the metric string of BASELINE.json, verbatim
HEADLINE = {"conv": 16384, "saw_svf_events": 16384, "saw_svf": 16384, "noise_svf": 16384, "fm": 4096, "biquad_bank": 2048, "subtractive_dry": 1024, "subtractive": 1024, "net": 65536}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="saw_svf", choices=sorted(HEADLINE))
    ap.add_argument("--voices", type=int, default=None, help="voices per GPU (default: the BASELINE config size)")
    ap.add_argument("--seconds", type=float, default=1.0, help="audio seconds rendered per step")
    ap.add_argument("--per-voice", action="store_true", help="also materialise per-voice outputs in HBM (value only)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --voices per GPU (default); strong: the config's voices split over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last timed step as DIR/<name>.npy (float32, at most 64 MB in all); "
                         "the warm-up is then exactly max(3, --warmup) steps, so the same arguments give the same outputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_BYTES = 64 << 20


def dump_sample(shape, budget, itemsize=4):
    """Row and column indices of a [rows, cols] output that fit in `budget` bytes: all of it when it fits, else a fixed, seeded sample
    of rows (and, if one row alone is too large, of columns), the same for the same shape so that two builds dump the same elements."""
    import numpy as np
    rows, cols = shape
    rng = np.random.default_rng(0)
    r, c = np.arange(rows), np.arange(cols)
    if rows * cols * itemsize > budget:
        r = np.sort(rng.choice(rows, min(rows, max(1, budget // (cols * itemsize))), replace=False))
    if len(r) * cols * itemsize > budget:
        c = np.sort(rng.choice(cols, max(1, budget // (len(r) * itemsize)), replace=False))
    return r, c


def dump_outputs(d, arrays):
    """`arrays`: {name: callable(rows, cols) -> float32 ndarray of those rows and columns, shape}; each gets an equal share of DUMP_BYTES."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, (take, shape) in arrays.items():
        r, c = dump_sample(shape, DUMP_BYTES // len(arrays))
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(take(r, c), dtype=np.float32))


_SCRATCH = []


def scratch_dir():
    """What the run compiles or caches goes here, never into the tree (which may be read-only); removed at exit."""
    if not _SCRATCH:
        _SCRATCH.append(tempfile.mkdtemp(prefix="fundsp_bench_"))
        atexit.register(shutil.rmtree, _SCRATCH[0], True)
    return _SCRATCH[0]


def jit_cache_overlay():
    """Points the JIT disk cache at a scratch directory holding links to the units build() compiled into fundsp_b200/jit_cache: those
    are still hits, and a unit compiled during the run is stored beside them instead of in the tree. An explicit FDSP_JIT_CACHE wins."""
    if os.environ.get("FDSP_JIT_CACHE"):
        return
    d = os.path.join(scratch_dir(), "jit_cache")
    os.makedirs(d)
    src = os.path.join(ROOT, "fundsp_b200", "jit_cache")
    for f in (os.listdir(src) if os.path.isdir(src) else ()):
        if f.endswith(".fdspjit"):
            os.symlink(os.path.join(src, f), os.path.join(d, f))
    os.environ["FDSP_JIT_CACHE"] = d


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, name in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_cores():
    """Threads the CPU arms may really use: the affinity mask capped by the cgroup CPU quota (os.cpu_count() reports the machine,
    not the lease — round 1's two boxes both said 128 and differed 5x)."""
    import math
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = max(1, min(aff, int(math.ceil(quota)))) if quota else max(1, aff)
    return eff, {"affinity": aff, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def native_oracle():
    """The timed CPU arm runs the oracle built for THIS host (-march=native, as BASELINE.md §3 states); the parity tests keep the
    portable x86-64-v3 build. Built per run in the scratch directory; falls back to the portable build if the compiler is missing."""
    so = os.path.join(scratch_dir(), "libfundsp_oracle_native.so")
    try:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "native", "NATIVE=" + so], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
        if os.path.exists(so):
            os.environ["FDSP_ORACLE_SO"] = so
            return "g++ -O3 -march=native -ffp-contract=off"
    except Exception:
        pass
    return "g++ -O3 -march=x86-64-v3 -ffp-contract=off (native build unavailable)"


def gate_for(workload, n):
    from fundsp_b200 import workloads
    return workloads.gate_signal(n) if workload.startswith("subtractive") else None


def cpu_reference(workload, voices, n, threads, first=0):
    """The reference's CPU algorithm for this path: V units, block-64 `process`, index-order mix (oracle, C++)."""
    from fundsp_b200 import workloads
    from oracle import oracle_bank_render
    exprs = workloads.build(workload, voices, first)
    _, mix = oracle_bank_render(exprs, SR, n, gate_for(workload, n), per_voice=False, mix=True, threads=threads)
    return oracle_bank_render.last_seconds, mix  # steady state: graph construction excluded, like the GPU arm


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = int(round(a.seconds * SR))
    Vg = a.voices or HEADLINE[a.workload]
    V = Vg * max(1, a.gpus) if a.scaling == "weak" else Vg   # the same whole-job configuration our arm runs at --gpus N
    if a.workload == "conv":
        Vg = V = min(V, 256)         # (a 1000-tap direct form on the CPU: a bounded number of voices stands for the bank)
    build = native_oracle()
    cores, core_info = host_cores()
    from fundsp_b200 import capi, workloads
    channels = capi.NodeHandle(workloads.build(a.workload, 1)[0]).outputs()   # host-side graph: no GPU involved
    # the whole step at N = 1 (and whenever it is at most ~1.5e9 voice-samples); beyond that a bounded sample of the step so that K
    # steps end within minutes on the host cores — the sample is stated, `ms_per_step` is what was measured, not an extrapolation
    ns = n if V * n <= 1.5e9 else max(64, int(1.5e9 / V) // 64 * 64)
    for _ in range(a.warmup):
        cpu_reference(a.workload, V, min(ns, 4800), cores)
    ts = []
    for _ in range(a.steps):
        dt, mix = cpu_reference(a.workload, V, ns, cores)
        ts.append(dt)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"mix": (lambda r, c: mix[r][:, c], mix.shape)})
    t = sum(ts) / len(ts)
    val = V * ns / t / 1e6
    v1 = min(V, 64)
    cpu_reference(a.workload, v1, 480, 1)
    dt1, _ = cpu_reference(a.workload, v1, min(ns, 24000), 1)
    per_core = v1 * min(ns, 24000) / dt1 / 1e6
    sample = (f"{V} voices x {ns} of {n} samples per step ({'the whole step' if ns == n else 'bounded sample'}), {cores} threads "
              f"(affinity {core_info['affinity']}, cgroup quota {core_info['cgroup_quota']}, os.cpu_count {core_info['os_cpu_count']}), voices sharded contiguously over the threads; {build}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Msamples/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": job_config(a, max(1, a.gpus), channels),
        "note": "the reference's CPU algorithm for this path: C++ oracle restating the block path (no Rust toolchain on the box), index-order mix of all voices, host cores only"
                + ("; the 1000-tap direct form is timed on %d voices standing for the bank" % V if a.workload == "conv" else ""),
        "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": "port", "sample": sample, "single_core": per_core,
                         "samples_per_step_timed": ns, "samples_per_step_config": n},
        "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def job_config(a, world, channels):
    """The configuration both arms print — identical keys and values for `bench.py` and `bench.py --impl reference` at the same flags."""
    V0 = a.voices or HEADLINE[a.workload]
    per, total = (V0 // world, V0) if a.scaling == "strong" else (V0, V0 * world)
    return {"workload": workload_name(a.workload, V0), "voices_per_gpu": per, "voices_total": total, "sample_rate": SR, "block": 64, "seconds_per_step": a.seconds,
            "output": "mix-down to %d channel(s)%s" % (channels, " + per-voice rows in HBM" if a.per_voice else ""),
            "parallelism": "voices sharded x%d, one mix-down per step below the C ABI (NCCL send/recv gather over NVLink + rank-order fold)" % world if world > 1 else "1 GPU",
            "l2": "flushed between timed steps (512 MB write)"}


def workload_name(w, V):
    names = {"saw_svf": f"{V}-voice saw_hz(f) >> lowpass_hz(fc,q) bank (north-star headline)", "noise_svf": f"{V}-voice white().seed(i) >> lowpass_hz(fc,q) bank (config 3a)",
             "fm": f"{V}-voice FM bank sine_hz(f)*f*m+f >> sine() (config 2)", "biquad_bank": f"{V} x biquad_bank() = {8 * V} voices on white() (config 3b)",
             "subtractive_dry": f"{V}-voice saw >> moog * adsr_live >> pan (config 4 without reverb)", "subtractive": f"{V}-voice subtractive + per-voice reverb_stereo (config 4)",
             "net": f"{V}-voice dynamic Net, 4 classes (config 5)",
             "conv": f"{V}-voice white().seed(i) >> convolve(h), one shared 1000-tap response (the dense tap contraction; not a BASELINE config)",
             "saw_svf_events": f"{V} held sequencer events of saw_hz(f) >> lowpass_hz(fc,q) (the headline voices behind Sequencer::push; not a BASELINE config)"}
    return names[w]


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)

    import numpy as np
    import torch

    from fundsp_b200 import workloads
    from fundsp_b200.bank import GpuBank

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; fundsp_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    jit_cache_overlay()
    torch.cuda.set_device(local)
    dist = None
    group = None
    if world > 1:
        import torch.distributed as dist
        from datetime import timedelta
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=timedelta(seconds=180))
        # the mix-down collective itself runs below the C ABI (fdsp_group_*: NCCL gather over NVLink + rank-order fold on the bank's
        # stream); torch.distributed only carries the 128-byte id, the barriers and the max-over-ranks of the timings
        from fundsp_b200.parallel import BankGroup
        group = BankGroup.from_torch_distributed(local)
    V = a.voices or HEADLINE[a.workload]
    if a.scaling == "strong":
        if V % world:
            raise SystemExit(f"--scaling strong: {V} voices do not split evenly over {world} GPUs")
        V //= world                       # the configuration's voices split over the GPUs: total work fixed
    n = int(round(a.seconds * SR))
    gate = gate_for(a.workload, n)

    # ---- build this rank's shard: voices [rank*V, (rank+1)*V)
    t_build = time.perf_counter()
    bank = GpuBank(workloads.build(a.workload, V, first=rank * V), device=local, per_voice=a.per_voice, mix=True, sample_rate=SR)
    bank.allocate(n)
    t_build = time.perf_counter() - t_build
    c = bank.voice_outputs()
    mix = torch.zeros((c, n), device="cuda", dtype=torch.float32)
    out = torch.empty((V * c, n), device="cuda", dtype=torch.float32) if a.per_voice else None
    gin = torch.from_numpy(gate).cuda() if gate is not None else None
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    host_mix = torch.empty((c, n), dtype=torch.float32).pin_memory()
    host_in = torch.from_numpy(gate).pin_memory() if gate is not None else None

    def device_step():
        bank.render_device(n, gin.data_ptr() if gin is not None else 0, n, out.data_ptr() if out is not None else 0, n, mix.data_ptr(), n, sync=False)
        if group is not None:
            group.reduce_device(bank, n, mix.data_ptr(), n, 0)      # fdsp_bank_reduce_device, on the bank's stream
        bank.sync()

    def e2e_step():
        from fundsp_b200.capi import check
        import ctypes as C
        fp = C.POINTER(C.c_float)
        hin = C.cast(host_in.data_ptr(), fp) if host_in is not None else None
        if group is None:
            check(bank.L.fdsp_bank_render(bank.h, n, hin, None, C.cast(host_mix.data_ptr(), fp)))
        else:   # one call per rank: render the shard, reduce the device mix over NVLink, ONE D2H on the root
            check(bank.L.fdsp_bank_render_reduced(bank.h, group.h, n, hin, C.cast(host_mix.data_ptr(), fp) if rank == 0 else None, 0))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(step_fn, steps):
        """K steps, each bracketed by CUDA events on the current stream; L2 flushed between steps (untimed)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kern, dom = [], []
        barrier()
        wall0 = time.perf_counter()
        for e0, e1 in evs:
            flush.fill_(1)
            torch.cuda.synchronize()
            e0.record()
            step_fn()
            e1.record()
            kern.append(bank.last_kernel_ms())
            dom.append(bank.last_dominant_ms())
        barrier()
        wall = time.perf_counter() - wall0
        ms = [e0.elapsed_time(e1) for e0, e1 in evs]
        timed.dominant_ms = sum(dom) / len(dom)
        return sum(ms) / len(ms), sum(kern) / len(kern), wall

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # >= W warm-up steps and about 1 s under load for the clock samples. The number of extra steps is decided by rank 0 and
    # broadcast: every rank must issue the same number of collectives.
    t_w = time.perf_counter()
    for _ in range(max(3, a.warmup)):
        device_step()
        e2e_step()
    per = (time.perf_counter() - t_w) / max(3, a.warmup)
    # (with --dump-outputs no extra steps: their number depends on timing, and every step advances the bank's state)
    extra = torch.tensor([0 if a.dump_outputs else min(500, max(0, int(1.0 / max(per, 1e-4))))], device="cuda", dtype=torch.int64)
    if dist is not None:
        dist.broadcast(extra, src=0)
    for _ in range(int(extra.item())):
        device_step()
        e2e_step()
    launches0 = bank.launch_count()
    ms_step, ms_kernel, wall = timed(device_step, a.steps)
    ms_dom = timed.dominant_ms      # the dominant kernel alone (CUDA events on the stream it is launched on, inside the bank)
    if not ms_dom > 0.0:            # FDSP_NO_DOM=1 (the A/B switch of those event records): fall back on the whole device region
        ms_dom = ms_kernel
    launches = bank.launch_count() - launches0
    if a.dump_outputs and rank == 0:   # the mix (reduced over the ranks) and, with --per-voice, this rank's voice rows
        def take(t):
            return lambda r, c: t[torch.from_numpy(r).cuda()][:, torch.from_numpy(c).cuda()].cpu().numpy()
        dump_outputs(a.dump_outputs, {"mix": (take(mix), tuple(mix.shape)), **({"voices": (take(out), tuple(out.shape))} if out is not None else {})})
    ms_e2e, _, _ = timed(e2e_step, a.steps)
    # AudioUnit::process granularity: one C-ABI call per 64-sample block with host buffers (the Wave::render call pattern)
    pb = 200
    barrier()
    t_p = time.perf_counter()
    for _ in range(pb):
        bank.process(64, gate[:, :64] if gate is not None else None)
    t_p = time.perf_counter() - t_p
    proc_val = world * V * 64 * pb / t_p / 1e6
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([ms_step, ms_e2e, ms_kernel, ms_dom], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, ms_e2e, ms_kernel, ms_dom = (float(x) for x in t.tolist())
        ln = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(ln)
        launches = int(ln.item())
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    total = world * V * n
    value = total / (ms_step * 1e-3) / 1e6
    e2e = total / (ms_e2e * 1e-3) / 1e6
    # ---- roofline of the dominant kernel (the fused voice program): algorithmic bytes per step / kernel time
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    cls = bank.classes()
    state_b = sum(k["voices"] * (2 * k["state_words"] + k["param_words"]) * 4 for k in cls)
    nlaunch_chunks = (n + 16383) // 16384
    grid = sum((k["voices"] + 127) // 128 for k in cls)
    bytes_step = state_b * nlaunch_chunks + grid * c * n * 4 * 2 + c * n * 4 + (V * c * n * 4 if a.per_voice else 0) + (n * 4 if gate is not None else 0)
    kernel_name, bound, unit, roof_extra = "fdsp::bank_kernel<...>", "hbm", "GB/s", {}
    if a.workload == "subtractive":
        # the HBM-bound kernel of the path: per voice-sample 32 lines x (4 B read + 4 B write) + 2 x 4 B dry in + 2 x 4 B mix-row out
        kernel_name = "fdsp::fdn_kernel<2>"
        bytes_step = V * n * (32 * 8 + 8 + 8)
        roof_extra = {"dry_stage": "the stage-pipelined voice program (Moog ladder in its own warp) runs beside it on the other stream and is the longer of the two: "
                                   "kernel_ms_all_per_step - kernel_ms_per_step is what it adds"}
    if a.workload == "conv":
        # the tensor-core tiles: issued = 3 (3xTF32) x 2 x V(padded to 128) x n(padded to 128 per 16384-chunk) x (128 + P, padded to 32) flops
        kernel_name, bound, unit = "fdsp::conv_tc_kernel<4>", "tensor", "TFLOP/s"
        K = 1000
        J = (128 + ((K - 1 + 3) // 4 * 4) + 31) // 32 * 32
        npad = sum(((min(16384, n - t0) + 127) // 128) * 128 for t0 in range(0, n, 16384))
        flops = 3 * 2.0 * ((V + 127) // 128 * 128) * npad * J
        peak = float(peaks.get("bf16_tflops", 1720.0)) / 2.0
        achieved = flops / (ms_dom * 1e-3) / 1e12
        roof_extra = {"useful_tflops": 2.0 * V * n * K / (ms_dom * 1e-3) / 1e12, "issued_flops_per_step": flops,
                      "peak_note": "TF32 dense = half of the measured BF16 dense rate of MEASURED_PEAKS.json (bf16_tflops / 2)"}
    else:
        achieved = bytes_step / (ms_dom * 1e-3) / 1e9
    traffic = None
    issue = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        t = prof.get(a.workload + ("+voices" if a.per_voice else ""))
        # ncu dram bytes of one 16384-sample launch of the dominant kernel, scaled to the step
        traffic = t["dram_bytes_per_launch"] * n / t["samples_per_launch"] if t else None
        if t and t.get("warp_inst_per_launch") and V == HEADLINE[a.workload] and bound == "hbm":
            # what actually bounds a voice program: warp-instructions issued (ncu count of one 16384-sample launch, scaled to the
            # step) against 148 SMs x 4 schedulers x 1 instruction per clock at the SM clock sampled during the timed region
            winst = t["warp_inst_per_launch"] * n / t["samples_per_launch"]
            mhz = float(clocks.get("sm_mhz") or 1965.0)
            issue = {"warp_inst_per_step": winst, "achieved_ginst_s": winst / (ms_dom * 1e-3) / 1e9, "peak_ginst_s": 592 * mhz * 1e6 / 1e9,
                     "frac": winst / (ms_dom * 1e-3) / (592 * mhz * 1e6), "source": "profiles/r02_traffic.json (smsp__inst_executed.sum of one launch)"}
    except Exception:
        pass
    # ---- CPU baseline on this box's host cores (bounded sample of the same workload)
    # (timed at N=1 only; multi-GPU runs carry the object with value null — the reference arm `--impl reference` covers every N)
    cores, core_info = host_cores()
    ns = min(n, 24000)
    cpu_val = per_core = None
    build = ""
    Vc = V
    if world == 1:
        build = native_oracle()
        if a.workload == "conv":
            Vc, ns = min(V, 2 * cores), 4800       # (1000 taps in the direct form on the CPU: a small sample stands for the bank)
        cpu_reference(a.workload, min(Vc, 256), 480, cores)
        dt, _ = cpu_reference(a.workload, Vc, ns, cores)
        cpu_val = Vc * ns / dt / 1e6
        dt1, _ = cpu_reference(a.workload, min(Vc, 64), ns, 1)
        per_core = min(Vc, 64) * ns / dt1 / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": job_config(a, world, c), "build_s": round(t_build, 3),
        "e2e": {"value": e2e, "unit": "Msamples/s", "h2d_bytes_per_step": int(n * 4 if gate is not None else 0), "d2h_bytes_per_step": int(c * n * 4),
                "call": "fdsp_bank_render(host buffers)" if world == 1 else "fdsp_bank_render_reduced(host buffers; D2H of the reduced mix on the root)", "ms_per_step": ms_e2e,
                "process_granularity": {"value": proc_val, "unit": "Msamples/s", "us_per_call": t_p / pb * 1e6, "call": "fdsp_bank_process(64) per block, host buffers"}},
        "gpu_launches": launches,
        "roofline": {"bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak, "traffic": traffic,
                     "kernel": kernel_name, "kernel_ms_per_step": ms_dom, "kernel_ms_all_per_step": ms_kernel, "algorithmic_bytes_per_step": int(bytes_step), **roof_extra,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)", "issue": issue,
                     "note": "IIR voice programs are issue/latency bound, not HBM bound (DESIGN.md §Roofline); see profiles/ for issue-slot utilisation"},
        "cpu_baseline": {"value": cpu_val, "unit": "Msamples/s", "cores": cores, "kind": "port", "single_core": per_core, "core_info": core_info,
                         "sample": (f"{Vc} voices x {ns} samples, oracle (C++ restatement of the reference block path; {build}), {cores} threads" if world == 1
                                    else "not timed at N > 1 (see the N=1 line and the --impl reference arm)")},
        "clocks": clocks,
        "wall_s_timed_region": wall,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
