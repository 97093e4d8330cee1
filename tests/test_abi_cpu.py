"""CPU: the C-ABI library loads, exports every symbol include/seekstorm_b200.h declares, and refuses to run
without a GPU (no CPU fallback).  No compute calls."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np

from seekstorm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "seekstorm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ssb_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_exported():
    names = _declared_symbols()
    assert len(names) >= 20
    L = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"
    assert sorted(_lib.EXPORTS) == names


def test_abi_version_and_struct_sizes():
    L = _lib.lib()
    assert L.ssb_abi_version() == 3
    assert ctypes.sizeof(_lib.SsbHitExt) == 48
    assert ctypes.sizeof(_lib.SsbVecQuery) == 40
    assert ctypes.sizeof(_lib.SsbHit) == 16
    assert ctypes.sizeof(_lib.SsbConfig) == 32
    assert ctypes.sizeof(_lib.SsbLevelDesc) == 16 + 6 * 8
    assert ctypes.sizeof(_lib.SsbLexBatch) == 8 + 7 * 8
    assert ctypes.sizeof(_lib.SsbFacetFilter) == 32 and ctypes.sizeof(_lib.SsbFacetField) == 8
    assert ctypes.sizeof(_lib.SsbStats) == 96


def test_no_cpu_fallback():
    """Without a GPU the product path fails loudly.  Checked in a child process that sees no device, so that a machine with a GPU
    runs the check too."""
    code = ("from seekstorm_b200 import Index, SsbError\n"
            "try:\n    Index(0)\nexcept SsbError as e:\n    print(e)\nelse:\n    print('Index(0) succeeded')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "no CUDA device" in r.stdout, r.stdout + r.stderr


def test_rrf_fuse_host_entry(golden):
    """ssb_rrf_fuse is pure host code in the library (search.rs:1962-2035): check it against the golden list."""
    L = _lib.lib()
    r = golden["rrf"]
    dt = np.dtype([("doc_id", "<u8"), ("score", "<f4"), ("pad", "<u4")])
    a = np.array([(d, s, 0) for d, s in r["lex"]], dtype=dt)
    b = np.array([(d, s, 0) for d, s in r["vec"]], dtype=dt)
    o = np.zeros(len(a) + len(b), dtype=dt)
    n = ctypes.c_uint32(0)
    assert L.ssb_rrf_fuse(a.ctypes.data, len(a), b.ctypes.data, len(b), o.ctypes.data, ctypes.byref(n)) == 0
    got = [(int(o[i]["doc_id"]), float(o[i]["score"])) for i in range(n.value)]
    assert [d for d, _ in got] == [d for d, _ in r["fused"]]
    for (_, s), (_, w) in zip(got, r["fused"]):
        assert np.float32(s) == np.float32(w)


def test_product_does_not_import_oracle():
    """The product package must never reference oracle/ (③): grep the sources."""
    pkg = os.path.join(ROOT, "seekstorm_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f)).read()
                assert "ssb_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f
