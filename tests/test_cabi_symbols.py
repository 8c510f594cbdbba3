"""The C-ABI library loads on a machine without a GPU and exports every symbol include/*.h declares."""
import ctypes
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for h in ("scema_hist.h", "scema_synth.h", "scema_ingest.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b(scema_[a-z0-9_]+)\s*\(", src))
    return sorted(names)


def test_exports_every_declared_symbol():
    import scema_b200
    lib = ctypes.CDLL(scema_b200.lib_path())
    syms = declared_symbols()
    assert len(syms) >= 24
    for s in syms:
        assert hasattr(lib, s), s
    from scema_b200 import binding
    assert set(binding.EXPORTED) <= set(syms)


def test_no_cpu_fallback():
    """Without a CUDA device the product refuses to run; it never routes to the oracle. (Any device is hidden from the
    process that tries.)"""
    code = "import scema_b200\ntry:\n    scema_b200.HistCluster(0)\nexcept scema_b200.ScemaError:\n    raise SystemExit(3)\n"
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 3, r.stderr[-2000:]


def test_product_never_touches_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "scema_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in src and "liboracle" not in src and "oracle/" not in src.replace("oracle/_ref binaries", ""), f


def test_k1_tune_hook_needs_no_device():
    """scema_k1_tune is process-wide host state (which spline kernel, warps per SM, memory hints): callable without a
    GPU, negative arguments leave a setting as it is, -2 returns the flags to the per-launch default."""
    import scema_b200
    lib = ctypes.CDLL(scema_b200.lib_path())
    lib.scema_k1_tune.argtypes = [ctypes.c_int] * 4
    lib.scema_k1_tune.restype = ctypes.c_int
    assert lib.scema_k1_tune(1, 12, 20, 2) == 0
    assert lib.scema_k1_tune(-1, -1, -1, -1) == 0
    assert lib.scema_k1_tune(1, 0, 0, -2) == 0   # back to the shipped defaults
