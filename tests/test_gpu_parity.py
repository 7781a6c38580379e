"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded voices.

Bars (DESIGN.md §Parity): bit-exact wherever the path is integer / pure IEEE f32 arithmetic (noise, SVF,
biquad bank, routing, and the `wide`-polynomial sine of the block path); where a libm transcendental or the
independently built wavetable enters the sample loop (tanh in Moog, sinf in tail samples, table entries that
differ by an f32 rounding), the bound is the north-star's 1e-5 relative f32:  |g - o| <= 1e-5 * max(|o|, floor)
with floor = 1e-2 * peak(|o|) of that voice (relative error is undefined at zero crossings).
"""
import ctypes as C

import numpy as np
import pytest

from fundsp_b200 import workloads
from fundsp_b200.prelude import *  # noqa: F401,F403
from oracle import lib as olib, oracle_bank_render

pytestmark = pytest.mark.gpu
SR = 48000.0


def gpu_render(voices, n, inp=None, mix=False, per_voice=True, sr=SR):
    from fundsp_b200.bank import GpuBank
    b = GpuBank(voices, per_voice=per_voice, mix=mix, sample_rate=sr)
    out, mx = b.render_samples(n, inp)
    return b, out, mx


def rel_err(g, o):
    """max over samples of |g-o| / max(|o|, 1e-2 * per-voice peak)."""
    peak = np.abs(o).max(axis=-1, keepdims=True)
    den = np.maximum(np.abs(o), 1e-2 * np.maximum(peak, 1e-30))
    return float((np.abs(g.astype(np.float64) - o) / den).max())


def check(name, V, n, exact, inp=None, tol=1e-5):
    olib().fo_set_denormal_emulation(0)
    voices = workloads.build(name, V)
    _, g, _ = gpu_render(voices, n, inp)
    o, _ = oracle_bank_render(workloads.build(name, V), SR, n, inp, threads=4)
    assert g.shape == o.shape and np.isfinite(g).all()
    assert np.abs(o).max() > 1e-3, "degenerate test signal"
    if exact:
        bad = np.argwhere(g != o)
        assert bad.size == 0, (name, bad[:4].tolist(), float(np.abs(g - o).max()))
    else:
        e = rel_err(g, o)
        assert e <= tol, (name, e)
    return g, o


def test_noise_svf_bit_exact():
    check("noise_svf", 300, 4800, exact=True)


def test_biquad_bank_bit_exact():
    check("biquad_bank", 40, 4800, exact=True)


def test_fm_bank_bit_exact_on_full_blocks():
    check("fm", 257, 4800, exact=True)  # 75 full 64-blocks: only the wide-sin block path runs


def test_fm_bank_tail_samples_within_tolerance():
    check("fm", 64, 4800 + 61, exact=False)  # last block of 61: 5 tail samples go through libm sinf


def test_saw_svf_headline():
    check("saw_svf", 300, 4800, exact=False)


def test_net_voice_classes():
    g, o = check("net", 256, 4800, exact=False)
    assert g.shape == (256, 2, 4800)


def test_subtractive_dry_chain():
    n = 24000
    check("subtractive_dry", 96, n, exact=True, inp=workloads.gate_signal(n))   # Moog tanh / sin through the restated musl libm: bit-exact


def test_subtractive_with_fdn_reverb():
    n = 9600
    check("subtractive", 33, n, exact=True, inp=workloads.gate_signal(n, SR) * 0 + np.concatenate(
        [np.zeros((1, 480), np.float32), np.ones((1, 4800), np.float32), np.zeros((1, n - 5280), np.float32)], axis=1))


def test_plumbing_config_1_voice():
    voices = [workloads.plumbing()]
    _, g, _ = gpu_render(voices, 48000)
    o, _ = oracle_bank_render([workloads.plumbing()], SR, 48000)
    assert np.array_equal(g, o)


# ---------------------------------------------------------------- block structure / AudioUnit::process semantics
def test_process_granularity_equals_render_and_oracle_blocks():
    """process(size) calls with ragged sizes must reproduce the reference's block quirks (phase wrap per block,
    table choice per 8 samples, tail through tick): compare against the oracle driven with the same sizes."""
    from fundsp_b200.bank import GpuBank
    from oracle import OracleUnit
    sizes = [64, 61, 8, 7, 1, 0, 64, 33, 64, 17]
    for name, exact in (("noise_svf", True), ("saw_svf", False), ("fm", False)):
        voices = workloads.build(name, 40)
        b = GpuBank(voices, per_voice=True, sample_rate=SR)
        units = [OracleUnit(v) for v in workloads.build(name, 40)]
        for u in units:
            u.set_sample_rate(SR)
        for s in sizes:
            g = b.process(s)
            o = np.concatenate([u.process(s) for u in units], axis=0) if s else np.zeros((40, 0), np.float32)
            assert g.shape == o.shape
            if s == 0:
                continue
            if exact:
                assert np.array_equal(g, o), (name, s)
            else:
                assert np.abs(g - o).max() <= 2e-6, (name, s, float(np.abs(g - o).max()))


@pytest.mark.parametrize("name,V", [("saw_svf", 300), ("noise_svf", 5000), ("fm", 130)])
def test_resident_process_kernel_equals_launch_per_block(name, V, monkeypatch):
    """A mix-mode bank that is driven block by block keeps ONE kernel resident and rings a doorbell per block (csrc/dsp/bank_kernel_rt.cuh).
    Same blocks, same CTA mix, same fold: the mixes must equal the one-launch-per-block path bit for bit, through ragged sizes, across a
    render() in the middle (which stops the resident kernel: its state words must be saved and picked up), reset and clone."""
    from fundsp_b200.bank import GpuBank
    sizes = [64, 64, 64, 61, 8, 7, 1, 64, 0, 33, 64, 17, 64, 64]
    def run(rt):
        monkeypatch.setenv("FDSP_RT", rt)
        b = GpuBank(workloads.build(name, V), per_voice=False, mix=True, sample_rate=SR)
        out = [b.process(s) for s in sizes if s]
        _, mid = b.render_samples(200)                  # any other call stops the resident kernel first
        out += [mid] + [b.process(s) for s in (64, 64, 64, 64, 5)]
        c = b.clone()
        out += [b.process(64), c.process(64)]
        b.reset()
        out += [b.process(s) for s in (64, 64, 64, 64)]
        return out
    a, r = run("1"), run("0")
    assert len(a) == len(r) and all(np.array_equal(x, y) for x, y in zip(a, r)), [i for i, (x, y) in enumerate(zip(a, r)) if not np.array_equal(x, y)]
    assert np.abs(np.concatenate(a, axis=-1)).max() > 0.1
    assert np.array_equal(a[-6], a[-5])                 # the clone continues exactly like the original


def test_two_banks_share_the_resident_slot(monkeypatch):
    """A resident process() kernel occupies every SM; a second bank of the device (or any other launch) must not sit behind it until its
    idle time-out. Two banks driven alternately, three blocks each, hand the slot over (every entry point of a bank first asks the owner of
    the device's resident kernel to leave): same mixes as the launch-per-block path, and no second-long stalls."""
    import time
    from fundsp_b200.bank import GpuBank
    def run(rt):
        monkeypatch.setenv("FDSP_RT", rt)
        a = GpuBank(workloads.build("saw_svf", 600), per_voice=False, mix=True, sample_rate=SR)
        b = GpuBank(workloads.build("saw_svf", 500, first=600), per_voice=False, mix=True, sample_rate=SR)
        a.process(64); b.process(64)                        # (first launches: module load, table upload)
        t = time.perf_counter()
        out = []
        for _ in range(6):
            out += [a.process(64) for _ in range(4)] + [b.process(64) for _ in range(4)]
        _, tail = b.render_samples(300)                       # a render of one bank while the OTHER may hold the slot
        out += [a.process(33), tail]
        return out, time.perf_counter() - t
    (x, tx), (y, ty) = run("1"), run("0")
    assert all(np.array_equal(p, q) for p, q in zip(x, y))
    assert tx < 0.5, (tx, ty)                                 # 12 hand-overs and a render: one idle time-out alone is about a second


def test_ragged_length_and_time_chunking():
    n = 16384 * 2 + 64 * 3 + 5  # crosses the kernel's time chunk and ends in a ragged block
    check("noise_svf", 130, n, exact=True)


def test_empty_and_single_sample_inputs():
    from fundsp_b200.bank import GpuBank
    b = GpuBank(workloads.build("noise_svf", 5), per_voice=True, sample_rate=SR)
    out, _ = b.render_samples(0)
    assert out.shape == (5, 1, 0)
    out, _ = b.render_samples(1)
    o, _ = oracle_bank_render(workloads.build("noise_svf", 5), SR, 1)
    assert np.array_equal(out, o)


# ---------------------------------------------------------------- mix-down, reset, clone, sample rate
def test_mix_down_matches_f64_sum():
    V, n = 1000, 4800
    b, g, mx = gpu_render(workloads.build("saw_svf", V), n, mix=True)
    ref = g.astype(np.float64).sum(axis=0)
    assert mx.shape == (1, n)
    scale = np.abs(g).sum(axis=0).max()
    assert np.abs(mx - ref).max() <= 1e-6 * scale  # deterministic tree vs f64 sum: ~sqrt(V) * eps
    # mix-only bank (no per-voice materialisation) gives the same mix bit for bit
    _, _, mx2 = gpu_render(workloads.build("saw_svf", V), n, mix=True, per_voice=False)
    assert np.array_equal(mx, mx2)


def test_mix_is_deterministic_and_stereo():
    V, n = 512, 2400
    _, _, a = gpu_render(workloads.build("net", V), n, mix=True, per_voice=False)
    _, _, b = gpu_render(workloads.build("net", V), n, mix=True, per_voice=False)
    assert a.shape == (2, n) and np.array_equal(a, b) and np.abs(a).max() > 0.1


def test_reset_and_clone_and_continuation():
    from fundsp_b200.bank import GpuBank
    voices = workloads.build("saw_svf", 64)
    b = GpuBank(voices, per_voice=True, sample_rate=SR)
    a1, _ = b.render_samples(1000)
    c = b.clone()
    a2, _ = b.render_samples(1000)
    c2, _ = c.render_samples(1000)
    assert np.array_equal(a2, c2)  # clone carries the device state (dyn_clone)
    full, _ = GpuBank(workloads.build("saw_svf", 64), per_voice=True, sample_rate=SR).render_samples(2000)
    # state carried across calls: ragged split points change block boundaries, compare with tolerance-free only at 64-multiples
    b.reset()
    r1, _ = b.render_samples(1024)
    r2, _ = b.render_samples(976)
    assert np.array_equal(np.concatenate([r1, r2], axis=-1), full)
    assert np.array_equal(a1, full[..., :1000])


def test_mixed_bank_two_stage_and_plain_classes():
    """A bank holding a pipelined two-stage class (dry program + FDN kernel on a second stream) next to plain classes: per-voice
    rows stay bit-exact and the mix (cleared, then accumulated by every class) equals the f64 sum of the rows."""
    from fundsp_b200.bank import GpuBank
    n = 6000 + 13
    gate = workloads.gate_signal(n)
    mk = lambda i: workloads.subtractive_voice(i) if i % 3 == 0 else ((pass_() * noise().seed(i) >> lowpass_hz(400.0 + 30.0 * i, 1.0) >> pan(0.1 * (i % 7) - 0.3)) if i % 3 == 1
                                                                       else (pass_() * saw_hz(110.0 + 5.0 * i) >> pan(-0.5)))
    V = 30
    b = GpuBank([mk(i) for i in range(V)], per_voice=True, mix=True, sample_rate=SR)
    assert len(b.classes()) == 3
    rows, mix = b.render_samples(n, gate)
    o, _ = oracle_bank_render([mk(i) for i in range(V)], SR, n, gate, threads=4)
    assert np.array_equal(rows, o)
    ref = rows.astype(np.float64).sum(axis=0)
    assert np.abs(mix - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    again, mix2 = GpuBank([mk(i) for i in range(V)], per_voice=True, mix=True, sample_rate=SR).render_samples(n, gate)
    assert np.array_equal(mix, mix2)     # deterministic across runs (fixed accumulation order)


def test_set_on_live_bank_matches_oracle_units():
    """AudioUnit::set (src/audiounit.rs:62) on single voices of a running bank: new coefficients, state continues."""
    from fundsp_b200.bank import GpuBank
    from oracle import OracleUnit
    V, n1, n2 = 48, 1024, 1500
    mk = lambda i: noise().seed(i) >> lowpass_hz(500.0 + 40.0 * i, 1.0 + 0.05 * i) >> highpass_hz(100.0, 0.7)
    b = GpuBank([mk(i) for i in range(V)], per_voice=True, sample_rate=SR)
    units = [OracleUnit(mk(i)) for i in range(V)]
    olib().fo_set_denormal_emulation(0)
    for u in units:
        u.set_sample_rate(SR)
    g1, _ = b.render_samples(n1)
    o1 = np.stack([u.process_many(n1) for u in units])
    CENTER_Q, LEFT, RIGHT = 2, (1, 0), (1, 1)          # Parameter::CenterQ; Address::Index(0|1) through Pipe<Pipe<Noise,Svf>,Svf>
    for v in (0, 7, V - 1):
        b.set(v, CENTER_Q, (2500.0 + v, 4.0), address=(LEFT, RIGHT))
        units[v].L.fo_set(units[v].h, CENTER_Q, (C.c_float * 2)(2500.0 + v, 4.0), 2, 0, (C.c_int64 * 4)(1, 0, 1, 1), 2)
    g2, _ = b.render_samples(n2)
    o2 = np.stack([u.process_many(n2) for u in units])
    assert np.array_equal(g1, o1)
    assert np.array_equal(g2, o2)
    b2 = GpuBank([mk(i) for i in range(V)], per_voice=True, sample_rate=SR)
    b2.render_samples(n1)
    h2, _ = b2.render_samples(n2)
    changed = [v for v in range(V) if not np.array_equal(h2[v], g2[v])]
    assert changed == [0, 7, V - 1]                    # only the addressed voices changed
    b.reset()
    g3, _ = b.render_samples(n1)
    assert np.array_equal(g3[1:7], g1[1:7]) and not np.array_equal(g3[0], g1[0])   # reset keeps the new setting (reference: set is sticky)


def test_set_sample_rate_recomputes_coefficients():
    for sr in (44100.0, 96000.0):
        _, g, _ = gpu_render(workloads.build("noise_svf", 32), 2205, sr=sr)
        o, _ = oracle_bank_render(workloads.build("noise_svf", 32), sr, 2205)
        assert np.array_equal(g, o)


# ---------------------------------------------------------------- structural coverage beyond the configs
def test_generic_graphs_via_registry_or_jit():
    from fundsp_b200.bank import GpuBank
    from fundsp_b200.capi import FdspError
    g = lambda i: (noise().seed(i) | dc((500.0 + 50.0 * i, 0.7))) >> lowpass() >> pan(0.1 * (i % 7) - 0.3)  # noqa: E731
    try:
        b = GpuBank([g(i) for i in range(37)], per_voice=True, sample_rate=SR)
    except FdspError as e:
        pytest.skip(f"graph class needs the JIT path: {e}")
    out, _ = b.render_samples(960)
    o, _ = oracle_bank_render([g(i) for i in range(37)], SR, 960)
    assert rel_err(out, o) <= 1e-5


# ---------------------------------------------------------------- full-size, size-independent properties
def test_full_size_headline_properties():
    """BASELINE size (16384 voices): per-voice parity on a strided sample of voices + linearity of the mix."""
    V, n = 16384, 4800
    voices = workloads.build("saw_svf", V)
    b, g, mx = gpu_render(voices, n, mix=True)
    idx = list(range(0, V, 997))
    o, _ = oracle_bank_render([workloads.saw_svf_voice(i) for i in idx], SR, n)
    assert rel_err(g[idx], o) <= 1e-5
    assert np.abs(mx - g.astype(np.float64).sum(axis=0)).max() <= 2e-6 * np.abs(g).sum(axis=0).max()
    assert np.isfinite(g).all() and np.abs(g).max() < 8.0


# Every BASELINE configuration at ITS OWN size (class layout, CTA spreading of bank_grid, the concurrent class streams of the 4-class Net
# bank, the stage-pipelined Moog classes, 1024 FDN voices in one wave): per-voice rows of a strided sample of voices against the oracle.
FULL = {
    # name: (voices, samples, voice stride, exact)
    "fm": (4096, 64 * 20, 173, True),                  # full blocks only: the wide-sin block path
    "noise_svf": (16384, 64 * 12 + 5, 701, True),
    "biquad_bank": (2048, 64 * 12 + 5, 97, True),
    "subtractive": (1024, 4800 + 7, 53, True),         # 1024 voices: stage-pipelined dry program -> FDN kernel, two-stream pipeline
    "net": (65536, 64 * 10, 2731, False),              # 4 classes x 16384 on concurrent streams; odd stride: every class is sampled
}


@pytest.mark.parametrize("name", sorted(FULL))
def test_full_size_config_sampled_voices(name):
    import os
    from fundsp_b200.bank import GpuBank
    if "mock" in os.environ.get("FDSP_B200_LIB", ""):
        pytest.skip("BASELINE-size banks are for the GPU (the CPU mock device walks every voice serially)")
    olib().fo_set_denormal_emulation(0)
    V, n, stride, exact = FULL[name]
    inp = workloads.gate_signal(n) if name == "subtractive" else None
    b = GpuBank(workloads.build(name, V), per_voice=True, mix=True, sample_rate=SR)
    g, mx = b.render_samples(n, inp)
    idx = list(range(0, V, stride)) + [V - 1]
    fn = workloads.WORKLOADS[name][0]
    o, _ = oracle_bank_render([fn(i) for i in idx], SR, n, inp, threads=4)
    assert np.abs(o).max() > 1e-3 and np.isfinite(g).all()
    if exact:
        assert np.array_equal(g[idx], o), (name, int((g[idx] != o).sum()), float(np.abs(g[idx] - o).max()))
    else:
        assert rel_err(g[idx], o) <= 1e-5, (name, rel_err(g[idx], o))
    # the mix of ALL voices against the f64 sum of the rows: sqrt(V) * eps * sum|x| (SURVEY.md §8d)
    ref = g.astype(np.float64).sum(axis=0)
    assert np.abs(mx - ref).max() <= 4.0 * np.sqrt(V) * 2.0 ** -24 * np.abs(g).astype(np.float64).sum(axis=0).max() + 1e-7


# ---------------------------------------------------------------- stage-pipelined kernels (csrc/dsp/bank_kernel_st.cuh)
@pytest.mark.parametrize("width", [32, 128])
@pytest.mark.parametrize("name,V", [("subtractive_dry", 70), ("net", 4 * 45)])
def test_stage_pipelined_kernels_equal_plain_kernels_and_oracle(name, V, width, monkeypatch):
    """Programs with a Moog run their stages in different warps (saw | Moog | ADSR, pan). Rows must equal the plain kernel's and the
    oracle's bit for bit (same per-node code on the same 8-sample groups), at both CTA shapes, with a ragged last block, a partly
    filled last CTA, per-voice rows and the CTA mix; state saved by one form continues in the other."""
    from fundsp_b200.bank import GpuBank
    olib().fo_set_denormal_emulation(0)
    n = 64 * 21 + 61
    inp = workloads.gate_signal(2 * n)[:, :n] if name.startswith("subtractive") else None
    monkeypatch.setenv("FDSP_STAGED_W", str(width))
    monkeypatch.setenv("FDSP_STAGED", "1")
    b = GpuBank(workloads.build(name, V), per_voice=True, mix=True, sample_rate=SR)
    rows, mix = b.render_samples(n, inp)
    import os
    assert "mock" in os.environ.get("FDSP_B200_LIB", "") or any(c["stages"] >= 2 for c in b.classes()), b.classes()   # (the CPU mock device has no staged form)
    o, _ = oracle_bank_render(workloads.build(name, V), SR, n, inp, threads=4)
    assert np.abs(o).max() > 1e-3
    assert np.array_equal(rows, o), (int((rows != o).sum()), float(np.abs(rows - o).max()))
    monkeypatch.setenv("FDSP_STAGED", "0")
    p = GpuBank(workloads.build(name, V), per_voice=True, mix=True, sample_rate=SR)
    rows0, mix0 = p.render_samples(n, inp)
    assert np.array_equal(rows0, rows)
    assert np.abs(mix - rows.astype(np.float64).sum(axis=0)).max() <= 1e-5 * max(1.0, np.abs(rows).sum(axis=0).max())
    # continuation: the staged bank goes on with the plain kernel, the plain bank with the staged one
    inp2 = np.zeros((1, n), np.float32) if inp is not None else None
    a2, _ = b.render_samples(n, inp2)
    monkeypatch.setenv("FDSP_STAGED", "1")
    b2, _ = p.render_samples(n, inp2)
    assert np.array_equal(a2, b2) and np.abs(a2).max() > 1e-4


# ---------------------------------------------------------------- warp-per-voice FDN kernel (reverb_stereo)
def test_reverb_only_bank_on_stereo_bus_input():
    """`reverb_stereo` applied to the bank's shared stereo input (one voice per room setting)."""
    n = 6000 + 37
    rng = np.random.default_rng(3)
    x = (rng.uniform(-1, 1, (2, n)) * (np.arange(n) < 3000)).astype(np.float32)
    mk = lambda i: reverb_stereo(10.0 + i, 1.0 + 0.5 * i, 0.3 + 0.1 * i)  # noqa: E731  (different delay lengths -> one class per voice)
    b, g, _ = gpu_render([mk(i) for i in range(3)], n, x)
    assert len(b.classes()) == 3
    o, _ = oracle_bank_render([mk(i) for i in range(3)], SR, n, x)
    assert np.array_equal(g, o) and np.abs(o).max() > 0.05


def test_shared_bus_reverb_send_uses_the_fdn_kernel():
    """`multipass() & g * reverb_stereo(..)` on a stereo bus (the shared-bus form of config 4, examples/keys.rs:164-181)."""
    from fundsp_b200.bank import GpuBank
    n = 4000 + 29
    rng = np.random.default_rng(7)
    x = rng.uniform(-0.5, 0.5, (2, n)).astype(np.float32)
    mk = lambda i: multipass(2) & (0.2 + 0.05 * i) * reverb_stereo(10.0, 2.0, 0.5)
    b = GpuBank([mk(i) for i in range(3)], per_voice=True, sample_rate=SR)
    assert b.classes()[0]["delay_floats"] > 90000
    g, _ = b.render_samples(n, x)
    o, _ = oracle_bank_render([mk(i) for i in range(3)], SR, n, x, threads=3)
    assert np.array_equal(g, o)


def test_fdn_kernel_process_granularity_and_wet_only_pipe():
    from fundsp_b200.bank import GpuBank
    from oracle import OracleUnit
    mk = lambda i: (noise().seed(i) >> pan(0.1 * i - 0.3)) >> reverb_stereo(12.0, 1.5, 0.4)  # noqa: E731  Pipe<X, Reverb>
    V = 9
    b = GpuBank([mk(i) for i in range(V)], per_voice=True, mix=True, sample_rate=SR)
    units = [OracleUnit(mk(i)) for i in range(V)]
    for u in units:
        u.set_sample_rate(SR)
    for s in (64, 64, 17, 64, 1, 0, 33, 64, 64, 64, 5):
        g = b.process(s)
        if s == 0:
            continue
        per_voice = np.stack([u.process(s) for u in units])  # [V, 2, s]
        ref = per_voice.astype(np.float64).sum(axis=0)
        assert g.shape == (2, s)
        assert np.abs(g - ref).max() <= 1e-5 * max(1.0, np.abs(per_voice).sum(axis=0).max())


def test_fdn_kernel_equals_generic_thread_per_voice_form(tmp_path):
    """The specialised kernel and the generic lowering of the same graph must agree bit for bit."""
    import os
    import subprocess
    import sys
    code = ("import sys; sys.path[:0]=['.','tests']; import numpy as np; from fundsp_b200 import workloads; from fundsp_b200.bank import GpuBank;"
            "b=GpuBank(workloads.build('subtractive',24),per_voice=True,sample_rate=48000.0); g,_=b.render_samples(4000+9, workloads.gate_signal(4009));"
            "np.save(sys.argv[1], g); print(b.classes()[0]['signature'][:20])")
    outs = []
    for k, env in enumerate(({}, {"FDSP_DISABLE_FDN": "1"})):
        path = str(tmp_path / f"fdn_ab_{k}.npy")
        subprocess.check_call([sys.executable, "-c", code, path], env={**os.environ, **env}, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        outs.append(np.load(path))
    assert np.array_equal(outs[0], outs[1]) and np.abs(outs[0]).max() > 0.01


# ---------------------------------------------------------------- dynamic Net (config 5): voices + Net::bus adder trees
@pytest.mark.parametrize("V,n", [(64, 1500), (37, 700 + 13), (1, 200), (1300, 300)])   # 1300: above 1024 voices the balanced tree reduces its 256-voice subtrees first
def test_net_of_voices_mix_is_bit_exact(V, n):
    """The reference form of config 5: each voice `Net::wrap`ped and bussed as a balanced tree (one Pass+Pass adder per output
    per `&`). The bank built from that Net must reproduce Net::ping's hashes and the tree's association order exactly."""
    from fundsp_b200.bank import GpuBank
    from fundsp_b200.net import voice_net
    from oracle import OracleBackend, OracleUnit
    olib().fo_set_denormal_emulation(0)
    net = voice_net([workloads.net_voice(i) for i in range(V)])
    ref = OracleUnit(net.lower(OracleBackend())).render(SR, n / SR)
    b = GpuBank.from_net(voice_net([workloads.net_voice(i) for i in range(V)]), per_voice=True, mix=True, sample_rate=SR)
    rows, mix = b.render_samples(n)
    assert mix.shape == ref.shape == (2, n) and np.abs(ref).max() > 0.05
    assert np.array_equal(mix, ref), (int((mix != ref).sum()), float(np.abs(mix - ref).max()))
    assert len(b.classes()) == min(V, 4) and rows.shape == (V, 2, n)
    # mix-only bank (internal row buffer) gives the same bits
    b2 = GpuBank.from_net(voice_net([workloads.net_voice(i) for i in range(V)]), per_voice=False, mix=True, sample_rate=SR)
    _, mix2 = b2.render_samples(n)
    assert np.array_equal(mix2, ref)


def test_net_bank_setting_by_node_id():
    """`net.set(Setting::center_q(..).node(id))` (src/net.rs:1159-1169) on a bank made from the Net: vertex id -> voice index."""
    from fundsp_b200.bank import GpuBank
    from fundsp_b200.net import Net
    from oracle import OracleUnit
    V, n = 6, 1500
    mk = lambda i: noise().seed(i) >> lowpass_hz(300.0 + 100.0 * i, 1.0) >> pan(0.0)
    net = Net.wrap(mk(0))
    for i in range(1, V):
        net = net & Net.wrap(mk(i))          # each `&` appends the new voice vertex and one adder vertex per output channel
    ids = [0] + [1 + 3 * (i - 1) for i in range(1, V)]
    b = GpuBank.from_net(net, per_voice=True, sample_rate=SR)
    assert [b.voice_of_vertex(v) for v in ids] == list(range(V))
    assert b.voice_of_vertex(2) == -1 and b.voice_of_vertex(3) == -1      # adder vertices are not voices
    rows0, _ = b.render_samples(n)
    b.set(b.voice_of_vertex(ids[3]), 2, (2500.0, 3.0), address=((1, 0), (1, 1)))   # CenterQ -> Pipe<Pipe<Noise,Svf>,Pan>: left, right
    rows1, _ = b.render_samples(n)
    olib().fo_set_denormal_emulation(0)
    u = OracleUnit(mk(3)); u.set_sample_rate(SR)
    o0 = u.process_many(n)
    u.L.fo_set(u.h, 2, (C.c_float * 2)(2500.0, 3.0), 2, 0, (C.c_int64 * 4)(1, 0, 1, 1), 2)
    o1 = u.process_many(n)
    assert np.array_equal(rows0[3], o0) and np.array_equal(rows1[3], o1)
    assert np.array_equal(rows1[2], np.concatenate([rows0[2], rows1[2]], axis=-1)[:, n:])  # other voices just continue


def test_net_left_fold_chain_mix_is_bit_exact():
    from fundsp_b200.bank import GpuBank
    from fundsp_b200.net import Net
    from oracle import OracleBackend, OracleUnit
    def build():
        net = Net.wrap(workloads.net_voice(0))
        for i in range(1, 9):
            net = net & Net.wrap(workloads.net_voice(i))
        return net
    ref = OracleUnit(build().lower(OracleBackend())).render(SR, 0.02)
    _, mix = GpuBank.from_net(build(), sample_rate=SR).render_samples(960)
    assert np.array_equal(mix, ref)


def test_tanh_fast_form_equals_plain_form():
    """The Moog ladder's tanhf runs on the device in a FAST form (csrc/dsp/libm.cuh: guard-free correctly rounded divisions, select tree, the sign carried in the operands);
    the host and the oracle comparison (tests/cpp/libm_equiv.cpp) know the PLAIN form. The probe compares the two on the device over all
    2^32 arguments and along a 16 384-sample ladder recurrence of 32 voices (silent, tiny, hot and ordinary lanes): not one bit may differ."""
    import os, re, subprocess
    if "mock" in os.environ.get("FDSP_B200_LIB", ""):
        pytest.skip("the fast form exists on the device only (MUFU.RCP); the CPU mock device runs the plain form")
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "probe", "_build", "moog_chain_probe")
    assert os.path.exists(exe), "tools/probe/_build/moog_chain_probe is missing: __graft_entry__.build() compiles it"
    out = subprocess.run([exe, "--sweep"], capture_output=True, text=True, timeout=300).stdout
    lines = [l for l in out.splitlines() if l.startswith("V8") or l.startswith("V9")]   # fast form, fast form with the sign off the chain (the default)
    assert len(lines) == 2, out
    for line in lines:
        m = re.search(r"chain-mismatches (\d+)\s+sweep-mismatches (\d+).*err no error", line)
        assert m and int(m.group(1)) == 0 and int(m.group(2)) == 0, line
