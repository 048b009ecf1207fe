"""CPU: the C-ABI library loads and exports every symbol include/pcgnn_b200.h declares; the ctypes
signature table covers exactly those symbols. No compute calls (no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HEADER = os.path.join(ROOT, "include", "pcgnn_b200.h")


def declared():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"PCG_API\s+[\w\s\*]+?\b(pcg_\w+)\s*\(", src)))


def test_header_declares_the_path():
    names = declared()
    for need in ("pcg_choose", "pcg_aggregate", "pcg_score_table", "pcg_pick_step", "pcg_last_error"):
        assert need in names


def test_library_exports_every_declared_symbol():
    from pcgnn_b200 import _lib

    if not os.path.exists(_lib.SO_PATH):
        import __graft_entry__ as g
        g.build()
    L = ctypes.CDLL(_lib.SO_PATH)
    for name in declared():
        assert hasattr(L, name), f"{name} declared in the header but not exported"


def test_binding_table_matches_header():
    from pcgnn_b200 import _lib

    assert sorted(_lib.SIGNATURES) == declared()
    src = open(HEADER).read()
    for name, (_, args) in _lib.SIGNATURES.items():
        m = re.search(r"PCG_API\s+[\w\s\*]+?\b" + name + r"\s*\(([^;]*?)\)\s*;", src, re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("void", "") else len(params.split(","))
        assert n == len(args), f"{name}: header has {n} parameters, binding has {len(args)}"


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from pcgnn_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "SO_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.PcgError, match="no CPU fallback"):
        _lib.lib()


def test_no_gpu_means_error_not_fallback():
    """Run in a child process that sees no CUDA device, so that the check also runs on a machine with a GPU."""
    code = ("from pcgnn_b200 import _lib\n"
            "from pcgnn_b200.engine import Engine\n"
            "try:\n"
            "    Engine(None)\n"
            "except _lib.PcgError as e:\n"
            "    print('PcgError:', e)\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.startswith("PcgError: pcgnn_b200 needs a CUDA device"), r.stdout


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pc-gnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "pcg_oracle" not in src, f
