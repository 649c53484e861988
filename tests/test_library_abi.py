"""CPU-side checks of the C-ABI boundary: the shared library loads and exports every symbol the header
declares (no compute calls -- there is no GPU in the build container), and the loader fails loudly."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tblup_b200.h")


def header_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tb_[a-z_0-9]+)\s*\(", text)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge
    ge.build()
    from tblup_b200 import _lib
    return _lib


def test_header_and_loader_agree(built):
    assert header_symbols() == sorted(built.SYMBOLS)


def test_library_exports_every_symbol(built):
    lib = ctypes.CDLL(built.LIB_PATH)
    for name in header_symbols():
        assert hasattr(lib, name), name
    assert built.load().tb_abi_version() == 1


def test_header_cites_reference_for_each_entry_point():
    text = open(HEADER).read()
    assert text.count("evaluator.py") >= 6 and "tblup/utils.py" in text


def test_no_cpu_fallback_without_device(built):
    """Creating a context with no GPU must raise with a clear message, never silently compute on the CPU.  Runs in a
    child process that sees no device, so it holds on machines with and without GPUs."""
    import subprocess
    import sys
    code = ("import numpy as np\n"
            "from tblup_b200 import GblupEngine\n"
            "try:\n"
            "    GblupEngine(np.zeros((8, 8), dtype=np.int8), np.zeros(8))\n"
            "except RuntimeError as e:\n"
            "    print(e)\n"
            "else:\n"
            "    raise SystemExit('GblupEngine was created without a device')\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stdout + out.stderr
    assert re.search("no CUDA device|no CPU fallback|CUDA", out.stdout), out.stdout


def test_product_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "tblup_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_genome_packing_semantics():
    import numpy as np
    from tblup_b200.engine import pack_genomes, as_dosage_int8
    flat, off = pack_genomes([np.array([3, -1, 3]), [0], np.array([], dtype=int)], 10)
    assert flat.tolist() == [3, 9, 3, 0] and off.tolist() == [0, 3, 4, 4]
    with pytest.raises(IndexError):
        pack_genomes([[10]], 10)
    with pytest.raises(IndexError):
        pack_genomes([[-11]], 10)
    # the threaded path of tb_pack_index_lists (>= 2^20 indices) against numpy's own fancy-index arithmetic, mixed
    # element widths, strided / unsigned / float-valued inputs, and the error names the first offending value
    rng = np.random.default_rng(0)
    m = 5000
    big = [rng.integers(-m, m, size=rng.integers(900, 1300)).astype(np.int32 if i % 3 else np.int64) for i in range(1100)]
    big[7] = big[7][::2]
    big[8] = big[8].astype(np.float64)
    big[9] = (big[9] % 200).astype(np.uint8)
    flat, off = pack_genomes(big, m)
    want = np.concatenate([np.arange(m)[np.asarray(b, dtype=np.int64)] for b in big])
    assert flat.dtype == np.int32 and np.array_equal(flat, want) and off[-1] == len(want) >= 1 << 20
    assert np.array_equal(np.diff(off), [len(b) for b in big])
    big[600] = big[600].copy()
    big[600][5] = m + 3
    big[900] = big[900].copy()
    big[900][0] = -m - 1
    with pytest.raises(IndexError, match="index %d is out of bounds" % (m + 3)):
        pack_genomes(big, m)
    with pytest.raises(IndexError, match="integer type"):
        pack_genomes([np.array([1.5])], m)
    with pytest.raises(ValueError):
        as_dosage_int8(np.array([[0.5, 1.0]]))
    with pytest.raises(ValueError):
        as_dosage_int8(np.array([[0, 3]]))
    assert as_dosage_int8(np.array([[0.0, 2.0]])).dtype == np.int8
