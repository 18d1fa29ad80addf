"""Builds libmsg_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m multi_style_transfer_gan_b200.build [--force]

No torch involvement: the library links cudart only and is opened with ctypes.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libmsg_b200.so")
SOURCES = ["api.cu", "conv_simt.cu", "conv_tc.cu", "conv_tma.cu", "conv_slab.cu", "conv_shift.cu", "msb_ring.cu", "convt_ring.cu", "out7_ring.cu", "down_ring.cu", "conv_wgrad_tc.cu", "instnorm.cu", "local_attn.cu", "local_attn_tc.cu", "local_attn_bwd_tc.cu", "la_stage.cu",
           "elementwise.cu", "blend_maps.cu", "gram.cu", "style_affine.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
if os.environ.get("MSG_LA_TRACE") == "1":      # development build: role timelines of the fused LocalAttention kernel (tools/la_trace.py)
    FLAGS.append("-DMSG_LA_TRACE")
# development A/B builds: MSG_NVCC_DEFS="-DX=1 -DY" MSG_LIB_SUFFIX=_x python -m multi_style_transfer_gan_b200.build writes
# libmsg_b200_x.so beside the product library; MSG_B200_LIB=<path> makes _lib.py open it instead
FLAGS += os.environ.get("MSG_NVCC_DEFS", "").split()
_SUFFIX = os.environ.get("MSG_LIB_SUFFIX", "")
if _SUFFIX:
    OBJ = os.path.join(HERE, "build" + _SUFFIX)
    LIB = os.path.join(HERE, f"libmsg_b200{_SUFFIX}.so")


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "msg_b200.h")]
    stamp = os.path.join(OBJ, "stamp")
    dig = _digest(deps)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    srcs = sources()

    def compile_one(s):
        o = os.path.join(OBJ, s.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(o + ".log", "w") as f:
            f.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(f"[build] {s} ok")
        return o

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
