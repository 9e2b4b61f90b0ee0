"""Build mocopci_b200/libb200pci.so in-tree with nvcc for sm_100a (no torch headers, seconds).

    python -m mocopci_b200.build [--force]

The library is a plain C-ABI shared object (include/b200pci.h); Python binds it with ctypes.
An object is rebuilt when the hash of (its source, every header, the flags, the nvcc version)
differs from the stamp written next to it, so stale binaries cannot survive a change of flags,
compiler or -D variants; ``build/BUILD_INFO.json`` records what the current library was made from
(``mode``: "full" when every object was compiled in that call, else "incremental").
"""
import concurrent.futures
import hashlib
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libb200pci.so")
SOURCES = ["common.cu", "knn.cu", "fps.cu", "gather.cu", "emd.cu", "probe.cu", "cosine.cu", "scatter.cu",
           "ball_p3d.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC"] + os.environ.get("B200PCI_EXTRA_NVCC_FLAGS", "").split()


def _nvcc_version():
    try:
        return subprocess.run([NVCC, "--version"], capture_output=True, text=True).stdout.strip().splitlines()[-1]
    except Exception:  # noqa: BLE001
        return "unknown"


def _headers_digest():
    h = hashlib.sha256()
    hdrs = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "b200pci.h"))
    for p in hdrs:
        h.update(p.encode())
        h.update(open(p, "rb").read())
    return h.hexdigest()


def _stamp(src, common):
    h = hashlib.sha256(common.encode())
    h.update(open(os.path.join(CSRC, src), "rb").read())
    return h.hexdigest()


def _compile(src, force, common):
    s = os.path.join(CSRC, src)
    o = os.path.join(OBJ, src[:-3] + ".o")
    stamp_file = o + ".stamp"
    want = _stamp(src, common)
    if not force and os.path.exists(o) and os.path.exists(stamp_file) and open(stamp_file).read() == want:
        return o, False
    subprocess.check_call([NVCC, *FLAGS, "-c", s, "-o", o])
    with open(stamp_file, "w") as f:
        f.write(want)
    return o, True


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    sources = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    common = "|".join([_nvcc_version(), " ".join(FLAGS), _headers_digest()])
    t0 = time.time()
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(sources)) as ex:
        res = list(ex.map(lambda s: _compile(s, force, common), sources))
    objs = [o for o, _ in res]
    compiled = [s for s, (_, c) in zip(sources, res) if c]
    if compiled or not os.path.exists(LIB):
        subprocess.check_call([NVCC, "-shared", "-Xlinker", "--no-undefined", "-o", LIB, *objs, "-lcudart"])
        info = {"mode": "full" if len(compiled) == len(sources) else "incremental",
                "compiled": compiled, "sources": sources, "flags": FLAGS, "nvcc": _nvcc_version(),
                "seconds": round(time.time() - t0, 1), "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
                "digest": hashlib.sha256("".join(_stamp(s, common) for s in sources).encode()).hexdigest()[:16]}
        with open(os.path.join(OBJ, "BUILD_INFO.json"), "w") as f:
            json.dump(info, f, indent=1)
        if verbose:
            print("built", LIB, f"({info['mode']}: {', '.join(compiled) or 'link only'}; {info['seconds']} s)")
    elif verbose:
        print("up to date", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
