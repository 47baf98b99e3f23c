"""CPU-side checks: the C-ABI library loads and exports every symbol include/svob200.h declares, the
struct layouts the bindings assume match the C sizeof()s, the host-side helpers behave, and creating
a context without a GPU fails loudly (no fallback)."""
import ctypes as C
import os
import re
import numpy as np
import pytest

from android_svo_b200 import capi, synth, frontend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "svob200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(svob200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = capi.load_library()
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), "libsvob200.so does not export %s" % n
    for n in capi.EXPORTED_SYMBOLS:
        assert n in names, "%s is bound in capi.py but not declared in include/svob200.h" % n


def test_every_exported_symbol_is_declared():
    """The library's C ABI is what include/svob200.h declares: no svob200_* function is exported by accident."""
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted({line.split()[-1] for line in out.splitlines() if line.split() and line.split()[-1].startswith("svob200_")})
    assert len(exported) >= 40
    undeclared = sorted(set(exported) - set(declared_symbols()))
    assert not undeclared, "exported by libsvob200.so but not declared in include/svob200.h: %s" % undeclared


def test_abi_struct_layout():
    c_sizes, py_sizes = capi.abi_sizes()
    assert c_sizes == py_sizes


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(capi.Svob200Error):
        capi.Context(0)


def test_round_mode_rule_matches_reference_dispatch():
    lib = capi.load_library()
    # vision.cpp:78 — SSE2 only when in.cols % 16 == 0
    assert [lib.svob200_round_mode_x86(w) for w in (640, 320, 160, 80, 40, 752, 376, 188)] == [1, 1, 1, 1, 0, 1, 0, 0]


def test_matcher_opts_defaults_match_reference():
    o = capi.MatcherOpts()
    capi.load_library().svob200_matcher_opts_default(C.byref(o), 5)
    # matcher.h:75-93
    assert (o.align_1d, o.align_max_iter, o.max_epi_search_steps, o.subpix_refinement, o.epi_search_edgelet_filtering) == (0, 10, 1000, 1, 1)
    assert o.epi_search_edgelet_max_angle == 0.7 and o.max_search_level == 4


def test_synth_is_deterministic_and_consistent(oracle):
    from oracle.pyoracle import Cam
    tex = synth.make_texture(256)
    assert tex.dtype == np.uint8 and tex.min() >= 16 and tex.max() <= 240
    assert np.array_equal(tex, synth.make_texture(256))
    cfg = dict(w=96, h=64, fx=80.0, fy=80.0, cx=47.5, cy=31.5)
    T = synth.trajectory(30, seed=3)[29]
    a = synth.render(tex, cfg, T)
    b = oracle.synth_render(tex, 400.0, 2.0, Cam.make(96, 64, 80.0, 80.0, 47.5, 31.5), T)
    assert np.array_equal(a, b)
    p = synth.backproject_to_plane(cfg, T, (40.0, 20.0))
    assert abs(p[2] - 2.0) < 1e-12
    assert np.allclose(frontend.project(cfg, T, [p])[0], (40.0, 20.0), atol=1e-9)
    assert np.allclose(frontend.project_many(cfg, T, np.array([p]))[0], (40.0, 20.0), atol=1e-9)


def test_select_features_is_cell_ordered():
    cells = np.zeros(6, capi.corner_dt)
    cells["score"] = [5, 30, 11, 10, 50, 12]
    cells["x"] = np.arange(6) * 10
    px, lv = frontend.select_features(cells, 10.0, 3)
    assert list(px[:, 0]) == [10.0, 20.0, 40.0]       # strict >, first come first served in cell order
    with pytest.raises(ValueError):
        frontend.select_features(cells, 10.0, 5)


def test_ldlt_split_bit_identical(tmp_path):
    """ldlt.cuh built for the host: factor + substitution (what the sparse alignment re-uses across the iterations of a level,
    sparse_img_align.cpp:253-262 / nlls_solver_impl.hpp:65) == the one-piece solve, bit for bit, on 50,000 systems."""
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    exe = str(tmp_path / "ldlt_split_check")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-I", os.path.join(here, "..", "android_svo_b200", "csrc"),
                           "-o", exe, os.path.join(here, "ldlt_split_check.cpp"), "-lm"])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "50000 systems, 0 mismatches" in out.stdout
