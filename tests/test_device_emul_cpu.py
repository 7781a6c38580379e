"""CPU-only check of the DEVICE node templates: tests/cpp/device_emul.cpp compiles csrc/dsp/nodes.cuh for the host and runs one
voice of a graph's fused program through the kernels' own block walk (csrc/dsp/voice_block.cuh walk_block); the output must equal the
oracle's bit for bit.
This is how device-side logic (here: the Dag form of nested Nets, and a sample of ordinary graphs) is exercised without a GPU.
The GPU tests remain the parity tests proper; nothing here is part of the product."""
import os
import struct
import subprocess

import numpy as np
import pytest

from fundsp_b200 import capi
from fundsp_b200.net import Net
from fundsp_b200.prelude import *  # noqa: F401,F403
from oracle import OracleUnit, lib as olib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SR = 44100.0   # the construction-time default rate (src/lib.rs:42): node handles are lowered as constructed


def emulate(g, n, x=None, tmp=None, sr=SR, staged=False):
    h = capi.NodeHandle(g)
    if sr != SR:
        h.set_sample_rate(sr)
    sig = h.signature()
    P, S, U = h.lowering()
    nin = h.inputs()
    exe = os.path.join(tmp, "emul")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-w", f"-DGRAPH={sig}"] + (["-DSTAGED=1"] if staged else []) +
                          [os.path.join(ROOT, "tests", "cpp", "device_emul.cpp"), "-o", exe])
    blob = os.path.join(tmp, "in.bin"); outp = os.path.join(tmp, "out.bin")
    with open(blob, "wb") as f:
        f.write(struct.pack("<5I", len(P), len(S), len(U), nin, n))
        f.write(struct.pack("<d", sr))
        f.write(P.tobytes()); f.write(S.tobytes()); f.write(U.tobytes())
        if nin:
            f.write(np.ascontiguousarray(x, np.float32).tobytes())
        kinds = [k for k in range(6) if f"WaveSynth<{k}," in sig or f"PhaseSynth<{k}>" in sig]   # as csrc/host/bank.cpp
        f.write(struct.pack("<I", len(kinds)))
        for k in kinds:
            f.write(_table_blob(k))
    r = subprocess.run([exe, blob, outp], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stderr)
    if staged:
        emulate.stages = [int(x[7:]) for x in r.stderr.split() if x.startswith("stages=")][0]
    claimed = [int(x[3:]) for x in r.stderr.split() if x.startswith("dl=")]
    assert claimed == [h.delay_floats()], ("delay-line storage: device program claims", claimed, "host allocates", h.delay_floats(), sig)
    return np.fromfile(outp, np.float32).reshape(h.outputs(), n), sig


def _table_blob(kind):
    """The wavetable set of one waveform in the layout the kernels read (csrc/host/wavetable.cpp device_wavetable): every table
    stored as [t[len-1]] t[0..len) [t[0] t[1]], padded to a multiple of 4 floats; `off` points at t[0]."""
    import ctypes as C
    L = capi.lib()
    n = L.fdsp_wavetable_count(kind)
    pitch, off, length, data = [], [], [], []
    for i in range(n):
        p, ln = C.c_float(0), C.c_int(0)
        L.fdsp_wavetable_info(kind, i, C.byref(p), C.byref(ln))
        t = np.ctypeslib.as_array(L.fdsp_wavetable_data(kind, i), shape=(ln.value,)).astype(np.float32)
        pitch.append(p.value); length.append(ln.value)
        data.append(t[-1:]); off.append(__import__("builtins").sum(len(d) for d in data)); data += [t, t[:1], t[1 % ln.value: 1 % ln.value + 1]]
    flat = np.concatenate(data).astype(np.float32)
    flat = np.concatenate([flat, np.zeros((-len(flat)) % 4, np.float32)])
    return (struct.pack("<3I", kind, n, len(flat)) + np.float32(pitch).tobytes() + np.int32(off).tobytes() + np.int32(length).tobytes() + flat.tobytes())


def oracle(g, n, x=None, sr=SR):
    olib().fo_set_denormal_emulation(0)
    u = OracleUnit(g)
    u.set_sample_rate(sr)
    return u.process_many(n, x)


def diamond_net():
    net = Net(1, 2)
    a = net.push(lowpass_hz(800.0, 1.0)); b = net.push(highpass_hz(300.0, 2.0)); c = net.push(pass_() + pass_())
    net.connect_input(0, a, 0); net.connect_input(0, b, 0); net.connect(a, 0, c, 0); net.connect(b, 0, c, 1)
    net.connect_output(c, 0, 0); net.connect_output(b, 0, 1)
    return net


def _chain_net():
    net = Net(0, 2)
    net.chain(noise().seed(11) | noise().seed(12)); net.chain(moog_hz(1500.0, 0.5) | moog_hz(1000.0, 0.6)); net.chain(lowpole_hz(1000.0) | lowpole_hz(500.0))
    return net


def _routing_net():
    net = Net(2, 3)
    v = net.push(mul(2.0))
    net.connect_input(1, v, 0)
    net.pass_through(0, 2); net.connect_output(v, 0, 0)      # output 1 stays unconnected (zero)
    return net


CASES = {
    "plain_pipe": lambda: noise().seed(1) >> lowpass_hz(900.0, 1.5) >> shape(Tanh(1.2)) >> pan(0.2),
    "dag_diamond": lambda: noise().seed(3) >> diamond_net().node(),
    "dag_operators": lambda: ((Net.wrap(sine_hz(110.0)) | Net.wrap(noise().seed(5))) >> Net.wrap(lowpass_hz(500.0, 1.0) | pass_())).node() >> join(2),
    "dag_chain_with_moog": lambda: _chain_net().node(),
    "dag_in_feedback": lambda: noise().seed(9) >> feedback((Net.wrap(delay(0.001) * 0.5) >> Net.wrap(lowpole_hz(2000.0))).node()),
    "dag_pass_through_and_zero": lambda: (noise().seed(2) | noise().seed(4)) >> _routing_net().node(),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_templates_on_host_match_oracle(name, tmp_path):
    n = 64 * 3 + 61                         # three full blocks + a block with a 5-sample tick-path tail
    g = CASES[name]()
    want = oracle(CASES[name](), n)
    got, sig = emulate(g, n, None, str(tmp_path))
    assert ("Dag<" in sig) == name.startswith("dag"), sig
    assert got.shape == want.shape and np.abs(want).max() > 1e-3
    assert np.array_equal(got, want), (name, int((got != want).sum()), float(np.abs(got - want).max()))


# ---- the whole JIT case list of the GPU suite, one voice each, on the host emulation (the GPU run checks 40 voices per case)
import test_gpu_jit as _jit  # noqa: E402


_ALL = {**_jit.CASES, **_jit.WIDER}


@pytest.mark.parametrize("name", sorted(_ALL))
def test_jit_case_on_host_emulation(name, tmp_path):
    n = 64 * 2 + 61 if not name.startswith("events") else 64 * 31 + 61   # events: long enough to start, fade and end
    mk = _ALL[name]
    vi = 4 if name.startswith("events") else 3
    want = oracle(mk(vi), n)
    got, _ = emulate(mk(vi), n, None, str(tmp_path))
    assert got.shape == want.shape
    assert np.array_equal(got, want), (name, int((got != want).sum()), float(np.abs(got - want).max()))
    assert not name.startswith("events") or np.abs(want).max() > 1e-3


# ---- the BASELINE configuration voices (AOT graph classes), incl. the gate-driven subtractive chain and the full voice with the
# 32-line reverb in its generic thread-per-voice form
from fundsp_b200 import workloads as _wl  # noqa: E402

WORKLOAD_VOICES = {
    "fm": lambda: _wl.fm_voice(5), "noise_svf": lambda: _wl.noise_svf_voice(5), "saw_svf": lambda: _wl.saw_svf_voice(5),
    "biquad_bank": lambda: _wl.biquad_bank_unit(1), "net_a": lambda: _wl.net_voice(0), "net_b": lambda: _wl.net_voice(1),
    "net_c": lambda: _wl.net_voice(2), "net_d": lambda: _wl.net_voice(3),
    "subtractive_dry": lambda: _wl.subtractive_dry_voice(5), "subtractive": lambda: _wl.subtractive_voice(5),
}


@pytest.mark.parametrize("name", sorted(WORKLOAD_VOICES))
def test_workload_voice_on_host_emulation(name, tmp_path):
    n = 64 * 40 + 61 if name.startswith("subtractive") else 64 * 4 + 61
    mk = WORKLOAD_VOICES[name]
    nin = capi.NodeHandle(mk()).inputs()
    x = None
    if nin:
        x = np.zeros((nin, n), np.float32)
        x[0, 100:1500] = 1.0                     # gate: arms on the low -> high edge, releases inside the render
    want = oracle(mk(), n, x)
    got, _ = emulate(mk(), n, x, str(tmp_path))
    assert np.abs(want).max() > 1e-3
    assert np.array_equal(got, want), (name, int((got != want).sum()), float(np.abs(got - want).max()))


@pytest.mark.parametrize("name", sorted(_ALL))
def test_every_voice_of_the_gpu_cases_builds(name):
    """The GPU suite renders 40 voices per case: all of them must be constructible (arity and argument checks of the C ABI) and fall
    into few classes; the GPU is not needed to find a case whose parameters run out of range at some voice index."""
    sigs = set()
    for i in range(40):
        h = capi.NodeHandle(_ALL[name](i))
        assert h.inputs() == 0 and h.outputs() >= 1
        sigs.add(h.signature())
    assert all("Unsupported" not in s for s in sigs) and len(sigs) <= 8, (name, len(sigs))


@pytest.mark.parametrize("name", sorted(k for k in _ALL if k.startswith("events")))
@pytest.mark.parametrize("vi", [0, 1, 7, 22, 39])
def test_event_voices_at_the_gpu_suite_rate(name, vi, tmp_path):
    """Event voices at 48 kHz (the rate of the GPU suite; the units and the sequencer clock are re-rated after construction) over the
    GPU suite's length, several voice indices: start / end times on and off block boundaries, events that never start."""
    n = 2000 + 61
    want = oracle(_ALL[name](vi), n, sr=48000.0)
    got, _ = emulate(_ALL[name](vi), n, None, str(tmp_path), sr=48000.0)
    assert np.array_equal(got, want), (name, vi, int((got != want).sum()), float(np.abs(got - want).max()))


def test_sequencer_event_voices_sum_to_the_oracle_sequencer(tmp_path):
    """The GPU sequencer is a bank of event voices whose mix is Sequencer::process. Here every voice of the five-event sequence of
    tests/test_gpu_wider.py runs on the host emulation and the rows are summed on the CPU: the sum must be the oracle Sequencer's
    output (exactly where one event sounds, to rounding where several overlap)."""
    from fundsp_b200.sequencer import Sequencer, Fade, ReplayMode
    q = Sequencer(0, 2, ReplayMode.All)
    q.push(0.1, 0.2, Fade.Smooth, 0.01, 0.0, noise() | sine_hz(220.0))
    q.push(0.3, 0.4, Fade.Smooth, 0.09, 0.08, sine_hz(110.0) | noise())
    q.push(0.25, 0.5, Fade.Power, 0.0, 0.01, mls() | noise())
    q.push(0.6, 0.7, Fade.Power, 0.02, 0.03, noise() | mls())
    q.push(0.31234, 0.45678, Fade.Smooth, 0.02, 0.05, (saw_hz(220.0) >> lowpass_hz(1000.0, 1.0)) | sine_hz(330.0))
    n = int(0.75 * SR)
    want = oracle(q.node(), n)
    rows = []
    for k, v in enumerate(q.voices()):
        d = tmp_path / f"v{k}"; d.mkdir()
        rows.append(emulate(v, n, None, str(d))[0])
    total = np.sum(np.stack(rows).astype(np.float64), axis=0)
    assert np.abs(want).max() > 0.5 and np.abs(total - want).max() <= 1e-6
    solo = slice(int(0.1 * SR) + 2, int(0.2 * SR) - 2)
    assert np.array_equal(rows[0][:, solo], want[:, solo])
    # an edited event (recorded before the start) ends early with the new fade-out
    q2 = Sequencer(0, 1, ReplayMode.None_)
    e = q2.push(100.0 / SR, 2000.0 / SR, Fade.Smooth, 0.0, 0.0, dc(1.0))
    q2.edit(e, 600.0 / SR, 100.0 / SR)
    got = emulate(q2.voices()[0], 800, None, str(tmp_path))[0]
    assert np.array_equal(got, oracle(q2.node(), 800)) and got[0, 300] == 1.0 and not got[0, 600:].any()


# ---- stage plans (csrc/dsp/stage_plan.cuh): the cut of a program into the warp stages of bank_kernel_st must keep every bit and the
# word layout. The emulation runs the stages of StagePlan<G> back to back per block, each from its own span of the word arrays.
STAGED = {
    # name: (graph, expected stages)
    "subtractive_dry": (lambda: _wl.subtractive_dry_voice(5), 3),                    # [saw | dc(fc,q) | gate] -> [Moog<3> | gate] -> [x ADSR >> pan]
    "net_b_saw_moog_pan": (lambda: _wl.net_voice(1), 2),                             # [saw] -> [Moog<1> >> pan]  (the pan is absorbed by the heavy stage)
    "moog_in_stack": (lambda: ((noise().seed(3) >> moog_hz(900.0, 0.4)) | sine_hz(220.0)) >> join(2), 2),   # noise (tiny) is absorbed into the Moog stage; [sine | join] behind it
    "two_moogs_in_series": (lambda: noise().seed(5) >> moog_hz(2000.0, 0.3) >> lowpass_hz(700.0, 1.0) >> moog_hz(500.0, 0.6) >> pan(-0.3), 3),
    "delay_in_front_of_moog": (lambda: noise().seed(8) >> delay(0.002) >> moog_hz(1500.0, 0.5) >> (pass_() & delay(0.001)), 3),   # delay-line cursors across stages
    "audio_rate_moog_sum": (lambda: ((noise().seed(2) | (sine_hz(3.0) * 400.0 + 900.0) | dc(0.5)) >> moog()) + sine_hz(50.0), 3),
}


@pytest.mark.parametrize("name", sorted(STAGED))
def test_stage_plan_keeps_every_bit(name, tmp_path):
    mk, k = STAGED[name]
    n = 64 * 30 + 61
    nin = capi.NodeHandle(mk()).inputs()
    x = None
    if nin:
        x = np.zeros((nin, n), np.float32)
        x[0, 100:1200] = 1.0
    want = oracle(mk(), n, x)
    got, sig = emulate(mk(), n, x, str(tmp_path), staged=True)
    assert emulate.stages == k, (sig, emulate.stages)
    assert np.abs(want).max() > 1e-3
    assert np.array_equal(got, want), (name, int((got != want).sum()), float(np.abs(got - want).max()))
