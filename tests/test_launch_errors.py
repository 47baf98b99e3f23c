"""How the library reports a failed launch, checked on the sources (no GPU needed).

A launch error that is not sticky (no kernel image for the device, an invalid configuration, too many resources) is cleared
by the cudaGetLastError() that reads it.  So every launcher returns the cudaError_t it read, the entry points report that
code, and every raw launch in the tracker is checked where it is made, so that its error is not blamed on the next stage.
"""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "android_svo_b200", "csrc")


def _sources():
    return {f: open(os.path.join(CSRC, f)).read() for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))}


def _balanced(src, i, open_ch, close_ch):
    """src[i] == open_ch: the text up to and including its matching close_ch"""
    depth = 0
    for j in range(i, len(src)):
        depth += (src[j] == open_ch) - (src[j] == close_ch)
        if depth == 0:
            return src[i:j + 1]
    raise AssertionError("unbalanced %s at %d" % (open_ch, i))


def _launcher_definitions():
    """(file, return type, name, body) of every launcher defined in csrc/*.cu"""
    out = []
    for f, src in _sources().items():
        if not f.endswith(".cu"):
            continue
        for m in re.finditer(r"^(?:static )?(\w+) (launch_\w+|seeds_update_impl)\(", src, re.M):
            params = _balanced(src, m.end() - 1, "(", ")")
            rest = src[m.end() - 1 + len(params):]
            if rest.lstrip().startswith(";"):
                continue                                  # a declaration
            out.append((f, m.group(1), m.group(2), _balanced(src, m.end() - 1 + len(params) + rest.index("{"), "{", "}")))
    return out


def test_launchers_return_cuda_error():
    decls = re.findall(r"^(\w+) (launch_\w+)\(", _sources()["kernels.h"], re.M)
    assert len(decls) >= 28
    assert [d for d in decls if d[0] != "cudaError_t"] == []
    defs = _launcher_definitions()
    names = {d[2] for d in defs}
    assert {n for _, n in decls} <= names and {"launch_lk_refine", "launch_fused"} <= names
    assert [(f, n) for f, t, n, _ in defs if t != "cudaError_t"] == []


def test_no_launcher_returns_an_int_code():
    for f, _, name, body in _launcher_definitions():
        assert not re.search(r"\breturn\s*-?\d+\s*;", body), "%s (%s) returns a bare integer" % (name, f)


def test_failures_do_not_read_the_error_again():
    """No fail(...) message is built from cudaGetLastError(): by then a launch error that is not sticky is gone."""
    for f, src in _sources().items():
        for m in re.finditer(r"\bfail\(", src):
            args = _balanced(src, m.end() - 1, "(", ")")
            assert "cudaGetLastError" not in args, "%s: %s" % (f, args[:120])
        assert "if (cudaGetLastError() != cudaSuccess) return fail" not in src, f


def test_tracker_checks_every_raw_launch():
    """Every <<<>>> launch in tracker.cu is counted and then checked by the next statement, under the kernel's name."""
    src = _sources()["tracker.cu"]
    n = 0
    for m in re.finditer(r"(\w+)(?:<[^<>]*>)?<<<", src):
        call = src.index(">>>(", m.end()) + 3
        tail = src[call + len(_balanced(src, call, "(", ")")):]
        c = re.match(r';\s*\+\+ctx->launches;\s*CU_AT\("(tracker_\w+): (\w+)", cudaGetLastError\(\)\);', tail)
        assert c, "unchecked launch of %s: %s" % (m.group(1), tail[:120])
        assert c.group(2) == m.group(1) or m.group(1) == "kernel", (m.group(1), c.group(2))
        n += 1
    assert n >= 17


def test_one_grid_cell_limit():
    """The grid-cell limit is stated once (kMaxGridCells); the launcher does not check it, the entry points do."""
    hits = [(f, line.strip()) for f, src in _sources().items() for line in src.splitlines() if re.search(r"\b8192\b", line)]
    assert hits == [("kernels.h", "constexpr int kMaxGridCells = 8192;")]
    body = {name: b for _, _, name, b in _launcher_definitions()}["launch_reproject_map"]
    assert "kMaxGridCells" not in body
    src = _sources()
    for f, entry in (("capi.cu", "svob200_reproject_map"), ("tracker.cu", "svob200_tracker_set_detector"),
                     ("tracker.cu", "svob200_tracker_add_keyframes"), ("tracker.cu", "svob200_tracker_set_chain")):
        i = src[f].index("int %s(" % entry)
        fn = _balanced(src[f], src[f].index("{", i), "{", "}")
        check = fn.index("> kMaxGridCells) return fail(ctx, SVOB200_ERR_UNSUPPORTED")
        first_work = min(fn.find(k) if fn.find(k) >= 0 else len(fn) for k in ("Stage st", "<<<", "launch_", "new_frame("))
        assert check < first_work, entry
