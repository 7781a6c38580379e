"""Compile the JIT translation unit of a graph signature with NVRTC, exactly as csrc/host/jit.cpp does (same headers, same
options), WITHOUT a GPU: catches header / template errors on the CPU box. Usage: nvrtc_check.py 'Pipe<Constant<1>,Dsf<1>>' ..."""
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDRS = ["math.cuh", "libm.cuh", "bank_args.h", "nodes.cuh", "mix_order.h", "voice_block.cuh", "bank_kernel.cuh"]   # = JITHDRS in csrc/Makefile


def compile_sig(sig):
    """Returns (ok, log)."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            from cuda.bindings import nvrtc
        except Exception:
            from cuda import nvrtc
    names, srcs = [], []
    for h in HDRS:
        text = open(os.path.join(ROOT, "fundsp_b200", "csrc", "dsp", h), "rb").read()
        for nm in (h, "dsp/" + h):
            names.append(nm.encode()); srcs.append(text)
    src = ('#include "dsp/bank_kernel.cuh"\nnamespace fdsp { typedef ' + sig + ' JitG; }\n'
           'extern "C" __device__ int fdsp_jit_layout[6] = {fdsp::JitG::IN, fdsp::JitG::OUT, fdsp::JitG::NP, fdsp::JitG::NS, fdsp::JitG::NU, fdsp::WaveKind<fdsp::JitG>::value};\n').encode()
    err, prog = nvrtc.nvrtcCreateProgram(src, b"fdsp_jit.cu", len(names), srcs, names)
    if int(err) != 0:
        return False, f"nvrtcCreateProgram: {err}"
    for mode in (1, 2, 3):
        for tb in ("false", "true"):
            nvrtc.nvrtcAddNameExpression(prog, f"fdsp::bank_kernel<fdsp::JitG, 128, {mode}, {tb}>".encode())
    opts = [b"--gpu-architecture=sm_100a", b"-std=c++17", b"--fmad=false", b"-lineinfo", b"-default-device"]
    (err,) = nvrtc.nvrtcCompileProgram(prog, len(opts), opts)
    _, n = nvrtc.nvrtcGetProgramLogSize(prog)
    log = b" " * n
    nvrtc.nvrtcGetProgramLog(prog, log)
    nvrtc.nvrtcDestroyProgram(prog)
    return int(err) == 0, log.decode(errors="replace")


if __name__ == "__main__":
    bad = 0
    for sig in sys.argv[1:]:
        ok, log = compile_sig(sig)
        print(("ok   " if ok else "FAIL ") + sig)
        if not ok:
            bad += 1
            print(log[:3000])
    sys.exit(1 if bad else 0)
