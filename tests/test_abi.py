"""The C-ABI library builds, loads and exports every symbol include/csmpn_b200.h declares (no GPU needed)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def built_lib():
    import __graft_entry__ as g

    g.build()
    from csmpn_b200 import _lib

    return _lib


def header_symbols():
    text = open(os.path.join(ROOT, "include", "csmpn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(csmpn_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(built_lib):
    lib = ctypes.CDLL(built_lib.LIB_PATH)
    names = header_symbols()
    assert len(names) >= 25
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in the header but not exported: {missing}"


def test_bindings_cover_header(built_lib):
    built_lib.lib()
    from csmpn_b200.models import fused

    assert fused.available()
    bound = set(built_lib.EXPORTED)
    assert set(header_symbols()) <= bound, sorted(set(header_symbols()) - bound)


def test_host_only_entry_points(built_lib):
    lib = built_lib.lib()
    assert lib.csmpn_version() >= 100
    assert lib.csmpn_status_string(0) == b"ok"
    assert b"workspace" in lib.csmpn_status_string(-5)
    # algebra tables on the host: Cl(3,0) multiplication table known answers (SURVEY.md section 4)
    B = 8
    out = (ctypes.c_int32 * (B * B))()
    coef = (ctypes.c_float * (B * B))()
    grades = (ctypes.c_int32 * B)()
    paths = (ctypes.c_uint8 * 64)()
    metric = (ctypes.c_float * 3)(1, 1, 1)
    assert lib.csmpn_algebra_tables(3, metric, out, coef, grades, paths) == 0
    assert list(grades) == [0, 1, 1, 1, 2, 2, 2, 3]
    row2 = [(out[2 * B + k], coef[2 * B + k]) for k in range(B)]
    assert row2 == [(2, 1), (4, -1), (0, 1), (6, 1), (1, -1), (7, -1), (3, 1), (5, -1)]
    assert sum(paths) == 20
    assert sum(1 for c in coef if c < 0) == 24
    assert lib.csmpn_algebra_tables(7, metric, out, coef, grades, paths) == -1
    assert lib.csmpn_param_grad_workspace(10) == 1024 * 10 * 4


def test_product_refuses_cpu_tensors(built_lib):
    import torch

    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models.cegnn_utils import MVLinear

    alg = CliffordAlgebra((1, 1, 1))
    with pytest.raises(RuntimeError, match="no CPU path"):
        alg.geometric_product(torch.randn(2, 8), torch.randn(2, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        MVLinear(alg, 4, 4)(torch.randn(3, 4, 8))


def test_simt_tile_rows_query(built_lib):
    """csmpn_block_simt_resident: rows per shared-memory tile of the SIMT engine (0 = weights would be staged); the host
    side composes blocks from unit kernels below 4 rows (models/fused.py)"""
    from csmpn_b200 import _lib

    l = _lib.lib()
    assert l.csmpn_block_simt_resident(3, 38, 32) >= 8       # md17 edge block
    assert l.csmpn_block_simt_resident(5, 34, 28) >= 4       # hulls, Cl(5,0)
    assert 0 <= l.csmpn_block_simt_resident(3, 70, 64) < 4   # wide block: composed from unit kernels
    assert l.csmpn_block_simt_resident(3, 131, 64) == 0
    assert l.csmpn_block_simt_resident(4, 8, 8) == 0         # unsupported dimension


def test_host_side_modules_import_without_gpu():
    """graphs / pipeline / train_step are importable on a CPU-only box (they touch CUDA only when used)"""
    import importlib

    for name in ("csmpn_b200.graphs", "csmpn_b200.pipeline", "csmpn_b200.train_step", "csmpn_b200.models.fused"):
        importlib.import_module(name)
    from csmpn_b200.models import fused

    assert fused.tc_min_rows() == 4096


def test_bench_accounting_matches_survey_formulas():
    """bench.layer_flops_bytes restates SURVEY.md 8d: 23.6 kB and 2.63 MFLOP per simplex at C=32, B=8, E/N=6"""
    import bench

    flops, nbytes = bench.layer_flops_bytes(1000, 6000, 32, 8)
    assert abs(nbytes / 1000 - 23.6e3) / 23.6e3 < 0.02
    assert abs(flops / 1000 - 2.63e6) / 2.63e6 < 0.02


def test_struct_layouts_match_the_header(tmp_path):
    """The ctypes mirrors of the three C structs (csmpn_block_desc, csmpn_block_grads, csmpn_lift_desc) have the header's
    size and the header's offset for every field: a C program compiled from include/csmpn_b200.h prints them (gcc; no GPU)."""
    import ctypes
    import shutil
    import subprocess

    from csmpn_b200.data.modules.lifting import LiftDesc
    from csmpn_b200.models.fused import BlockDesc, BlockGrads

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    structs = {"csmpn_block_desc": BlockDesc, "csmpn_block_grads": BlockGrads, "csmpn_lift_desc": LiftDesc}
    lines = ["#include <stddef.h>", "#include <stdio.h>", '#include "csmpn_b200.h"', "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    subprocess.run([gcc, "-std=c11", "-I", inc, str(src), "-o", str(exe)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    seen = 0
    for line in filter(None, out):
        cname, fname, val = line.split()
        cls = structs[cname]
        want = ctypes.sizeof(cls) if fname == "size" else getattr(cls, fname).offset
        assert int(val) == want, f"{cname}.{fname}: header {val}, ctypes {want}"
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in structs.values())
