"""The HOST runtime (csrc/host/bank.cpp, graph.cpp, capi.cpp: class building, word layout, launch sequencing, mix reduction, process()
path, settings on a live bank, sequencer clock / edit / push / growth in place, clone, reset ...) exercised WITHOUT a GPU.

tests/cpp/mock/ builds the host sources against a stand-in <cuda_runtime.h> ("device" memory is host memory, calls are synchronous) and
replaces the kernels by the device node library compiled for the CPU (FDSP_HOST_EMUL), one small shared object per graph class walking
every voice through the kernels' own block walk (csrc/dsp/voice_block.cuh) and summing the mix in the kernels' association
(csrc/dsp/mix_order.h), so the per-CTA partials equal the GPU's bit for bit. The whole GPU test-suite then runs against that library in a
subprocess (FDSP_B200_LIB selects it there and only there). What this does NOT cover is the CUDA side proper — the mix tile's shared
memory and barriers, TMA table staging, the warp-per-voice FDN kernel itself (the mock runs the equivalent generic reverb program on its argument block, so the host side of
the two-stage classes IS covered), stream concurrency — which the same tests check on a B200.
The mock is test infrastructure: it is never built into, or loaded by, the product."""
import hashlib
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fundsp_b200", "csrc")
MOCK = os.path.join(ROOT, "tests", "cpp", "mock")


def _tree_hash():
    h = hashlib.sha256()
    files = [os.path.join(MOCK, f) for f in sorted(os.listdir(MOCK)) if f.endswith((".h", ".cpp"))]
    for d in ("dsp", "host"):
        files += [os.path.join(CSRC, d, f) for f in sorted(os.listdir(os.path.join(CSRC, d)))]
    files += [os.path.join(CSRC, "capi.cpp"), os.path.join(ROOT, "include", "fundsp_b200.h")]
    for f in files:
        h.update(f.encode()); h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


SAN = os.environ.get("FDSP_MOCK_SANITIZE", "")   # "address" or "undefined": build the mock device and every class module with that sanitizer


@pytest.fixture(scope="module")
def mock_env():
    build = os.path.join(MOCK, "_build", _tree_hash() + ("_" + SAN if SAN else ""))        # keyed by every source that goes into it: never stale
    os.makedirs(build, exist_ok=True)
    for d in os.listdir(os.path.dirname(build)):            # builds of older sources are never used again
        if not d.startswith(_tree_hash()):
            import shutil
            shutil.rmtree(os.path.join(os.path.dirname(build), d), ignore_errors=True)
    lib = os.path.join(build, "libfundsp_b200_mock.so")
    if not os.path.exists(lib):
        srcs = [os.path.join(CSRC, "host", f) for f in ("graph.cpp", "wavetable.cpp", "bank.cpp", "group.cpp", "wavfile.cpp")] + [os.path.join(CSRC, "capi.cpp"), os.path.join(MOCK, "registry_mock.cpp")]
        san = ["-fsanitize=" + SAN, "-g", "-fno-omit-frame-pointer"] if SAN else []
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-w", "-shared", "-fPIC", "-DFDSP_HOST_EMUL=1", *san, "-I", MOCK, "-I", CSRC,
                               "-x", "c++", *srcs, "-o", lib + ".tmp", "-ldl"])
        os.replace(lib + ".tmp", lib)
    env = dict(os.environ, FDSP_B200_LIB=lib, FDSP_MOCK_ROOT=ROOT, FDSP_MOCK_CACHE=os.path.join(build, "classes"))
    if SAN:   # every "device" buffer is a host allocation here, so the sanitizer sees each out-of-bounds word the GPU would silently read or write
        rt = subprocess.check_output(["gcc", "-print-file-name=lib" + ("asan" if SAN == "address" else "ubsan") + ".so"], text=True).strip()
        env.update(LD_PRELOAD=rt, ASAN_OPTIONS="detect_leaks=0", UBSAN_OPTIONS="halt_on_error=1",
                   FDSP_MOCK_CXXFLAGS="-fsanitize=" + SAN + " -g -fno-omit-frame-pointer" + (" -fno-sanitize-recover=undefined" if SAN == "undefined" else ""))
    return env


def test_gpu_suite_runs_on_the_mock_device(mock_env):
    files = [os.path.join(ROOT, "tests", f) for f in ("test_gpu_jit.py", "test_gpu_parity.py", "test_gpu_wider.py")]
    r = subprocess.run([sys.executable, "-m", "pytest", *files, "-m", "gpu", "-q", "-n", "8", "-p", "no:cacheprovider", "--tb=short"],
                       capture_output=True, text=True, env=mock_env, cwd=ROOT, timeout=3000)
    tail = r.stdout[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail and "failed" not in tail and "error" not in tail.lower(), tail


def test_sharded_bank_on_the_mock_device(mock_env):
    """bench.py --gpus N in small: two gloo ranks, each a real GpuBank over its shard of the voices (mock device), one reduce of the mix."""
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tests", "_mock_sharded_worker.py")], capture_output=True, text=True, env=mock_env, cwd=ROOT, timeout=900)
    assert r.returncode == 0 and r.stdout.count(": ok") == 3 and "MISMATCH" not in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])


def test_gpu_box_scripts_run_on_the_mock_device(mock_env):
    """The scripts of the first GPU call of a round (tools/gpu_first_call.sh) are dry-run here at toy sizes, so GPU minutes are not
    spent finding a typo: smoke() and the sequencer timing script."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "prof_sequencer.py"), "--voices", "24", "--samples", "2048"],
                       capture_output=True, text=True, env=mock_env, cwd=ROOT, timeout=900)
    assert r.returncode == 0 and "sequencer bank" in r.stdout and "per push_event" in r.stdout, (r.stdout[-800:], r.stderr[-1500:])
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], capture_output=True, text=True, env=mock_env, cwd=ROOT, timeout=900)
    assert r.returncode == 0 and "smoke ok" in r.stdout, (r.stdout[-800:], r.stderr[-1500:])


def test_product_library_is_not_the_mock():
    """The mock is selected by FDSP_B200_LIB in the subprocess above only: the library the package loads by default is the CUDA build."""
    from fundsp_b200 import capi
    assert "FDSP_B200_LIB" not in os.environ or "mock" not in os.environ["FDSP_B200_LIB"]
    path = capi.lib()._name
    assert path.endswith("libfundsp_b200.so") and "mock" not in path
    out = subprocess.run(["nm", "-D", "--undefined-only", path], capture_output=True, text=True).stdout
    assert "fdsp_emul_launch" not in out and "g++" not in out
