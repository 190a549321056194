"""CPU-only: the C-ABI library builds/loads, exports every symbol include/als_b200.h declares, and the
ctypes table covers exactly that set.  No compute calls (there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "als_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(als_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from implicit_b200 import _build

    path = _build.build()
    lib = ctypes.CDLL(path)
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/als_b200.h but not exported"
    assert lib.als_abi_version() == 1


def test_ctypes_table_matches_header():
    from implicit_b200 import _lib

    assert sorted(_lib.SIGNATURES) == _declared()


def test_no_gpu_means_loud_failure():
    """There is no CPU fallback: without a device, creating a context raises.  Checked in a child process that sees
    no device, so that it holds on a GPU machine too."""
    code = ("import pytest\nfrom implicit_b200 import _lib\nassert _lib.device_count() == 0\n"
            "with pytest.raises(_lib.AlsError):\n    _lib.Context(0)\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_does_not_import_the_oracle():
    """oracle/ is test infrastructure: nothing under implicit_b200/ may reference it."""
    pkg = os.path.join(ROOT, "implicit_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "oracle/" not in src, f


def test_graft_entry_build_runs():
    """The driver's build check: compiles (or finds up to date) the library, the oracle port and, where the
    reference is present, oracle/_ref -- and every header symbol resolves."""
    import __graft_entry__ as entry

    assert entry.build() is None
    import importlib

    import oracle

    if importlib.import_module("oracle.build_ref").ref_available():
        assert oracle.have_ref() and oracle.have_ref_evaluation()


def test_library_holds_the_blackwell_paths():
    """The sm_100a-specific data paths are in the built library, kernel by kernel (cuobjdump, no GPU needed): tcgen05
    MMAs with TMEM loads and TMA in the dense pre-pass, the Gramian and the top-k kernel; tcgen05 + setmaxnreg in the
    opt-in long-row kernel.  A refactor that silently falls back to mma.sync everywhere fails here."""
    import shutil
    import subprocess

    from implicit_b200 import _build

    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([exe, "-sass", _build.build()], capture_output=True, text=True).stdout
    per_kernel = {}
    fn = None
    for line in sass.splitlines():
        if "Function :" in line:
            fn = line.split("Function :")[1].strip()
            per_kernel[fn] = set()
        elif fn is not None:
            for m in ("UTCHMMA", "UTMALDG", "UTMASTG", "LDTM", "USETMAXREG"):
                if m in line:
                    per_kernel[fn].add(m)

    def has(kernel, *mnemonics):
        hits = [ms for name, ms in per_kernel.items() if kernel in name]
        return bool(hits) and all(any(m in ms for ms in hits) for m in mnemonics)

    assert has("dense_apply_kernel", "UTCHMMA", "UTMALDG", "UTMASTG", "LDTM")
    assert has("gramian_tc_kernel", "UTCHMMA", "UTMALDG", "LDTM")
    assert has("topk_tc_kernel", "UTCHMMA", "UTMALDG", "LDTM")
    assert has("cholesky_tc_kernel", "UTCHMMA", "LDTM", "USETMAXREG")
