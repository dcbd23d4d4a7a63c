"""In-tree nvcc build of libellc_gn.so (sm_100a only).  nvcc cross-compiles without a GPU."""
import os
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libellc_gn.so")
SOURCES = ["ellc_api.cu", "ellc_preprocess.cu", "ellc_track.cu", "ellc_ingest.cu", "ellc_sequence.cu"]
HEADERS = ["ellc_common.cuh", "ellc_internal.h", "ellc_lie.cuh", os.path.join("..", "..", "include", "ellc_gn.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def _code_only(text):
    """C / CUDA source without comments and with runs of whitespace collapsed (string literals are left alone)."""
    import re
    pat = re.compile(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\])*"|\'(?:\\.|[^\'\\])*\'', re.S)
    text = pat.sub(lambda m: m.group(0) if m.group(0)[0] in "\"'" else " ", text)
    return re.sub(r"\s+", " ", text).strip()


def source_hash():
    """SHA-1 over the CODE of the kernel / ABI sources (comments and layout do not count): ellc_version() carries it, so that a
    profile (profiles/r02_traffic.json, r02_sass_histogram.json) can be matched to the build it was taken from."""
    import hashlib
    h = hashlib.sha1()
    for f in sorted(SOURCES + HEADERS):
        with open(os.path.join(CSRC, f), "r", encoding="utf-8", errors="replace") as fh:
            h.update(f.encode() + b"\0" + _code_only(fh.read()).encode())
    return h.hexdigest()[:12]


def build(force=False, verbose=False):
    """Compile every CUDA source of the package for sm_100a into one shared library; returns its path."""
    if not (force or _stale()):
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-DELLC_SRC_HASH=\"%s\"" % source_hash()] + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return LIB


def build_variant(name, defines):
    """EXPERIMENTS: the library with extra -D flags as build/variants/libellc_gn_<name>.so (select it with ELLC_LIB=...)."""
    out_dir = os.path.join(os.path.dirname(PKG), "build", "variants")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "libellc_gn_%s.so" % name)
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-DELLC_SRC_HASH=\"%s+%s\"" % (source_hash(), name)] + ["-D" + d for d in defines] + ["-o", out] + SOURCES
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
