"""Build + load the device-math harness (tests/device_math/harness.cu) for one of two backends.

device: nvcc for sm_100a with the library's code-generation flags (lambdaworks_kzg_b200/csrc/Makefile), so the
        headers are compiled the way the product's kernels are; the cases run on the GPU.
emul:   g++ with -DLWKZG_HOST_EMUL: the same per-case functions in a host loop (no GPU needed).
"""
import ctypes
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "device_math")
SRC = os.path.join(DIR, "harness.cu")
CSRC = os.path.join(os.path.dirname(HERE), "lambdaworks_kzg_b200", "csrc")
LIBS = {"device": os.path.join(DIR, "libdm_device.so"), "emul": os.path.join(DIR, "libdm_emul.so")}

# dm_run's own return codes (anything else non-zero is a cudaError_t)
UNSUPPORTED = -1


def _stale(lib):
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    return any(os.path.getmtime(d) > t for d in deps)


def _command(backend, out):
    if backend == "device":
        nvcc = os.environ.get("NVCC") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc")
        return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared", "-o", out, SRC]
    return ["g++", "-O2", "-std=c++17", "-x", "c++", "-DLWKZG_HOST_EMUL", "-DLWKZG_EMUL_PAIRING",
            "-shared", "-fPIC", "-o", out, SRC]


def load(backend):
    lib = LIBS[backend]
    if _stale(lib):
        tmp = "%s.%d.tmp" % (lib, os.getpid())
        try:
            subprocess.check_call(_command(backend, tmp))
            os.replace(tmp, lib)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    dll = ctypes.CDLL(lib)
    dll.dm_run.restype = ctypes.c_int
    dll.dm_run.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                           ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
    return dll


class Harness:
    """dm_run over Python records: each record is a list of u32 words (in) and comes back as one (out)."""

    def __init__(self, backend):
        self.backend = backend
        self.lib = load(backend)

    def run(self, op, records, out_words, threads_per_block=32, odd_lanes_only=False):
        n = len(records)
        in_words = max(len(r) for r in records)
        inb = (ctypes.c_uint32 * (in_words * n))()
        for i, r in enumerate(records):
            inb[i * in_words: i * in_words + len(r)] = r
        outb = (ctypes.c_uint32 * (out_words * n))()
        rc = self.lib.dm_run(op, n, threads_per_block, 1 if odd_lanes_only else 0,
                             ctypes.addressof(inb), 4 * in_words, ctypes.addressof(outb), 4 * out_words)
        if rc == UNSUPPORTED:
            return None
        assert rc == 0, "dm_run(op=%d) failed with code %d" % (op, rc)
        return [list(outb[i * out_words:(i + 1) * out_words]) for i in range(n)]


def words(v, n):
    """Integer -> n little-endian u32 words."""
    assert 0 <= v < 1 << (32 * n)
    return [(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)]


def from_words(w):
    return sum(int(x) << (32 * i) for i, x in enumerate(w))


def bytes_words(b):
    """Byte string (length a multiple of 4) -> u32 words holding those bytes in memory order."""
    assert len(b) % 4 == 0
    return [int.from_bytes(b[i:i + 4], "little") for i in range(0, len(b), 4)]


def words_bytes(w):
    return b"".join(int(x).to_bytes(4, "little") for x in w)
