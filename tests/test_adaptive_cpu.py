"""Adaptive frames (include/sqt.h: sqt_render_retire), the parts that need no GPU: the sqt_retire_params layout, the host build
of the per-pixel retire test against a numpy evaluation of the header's formula, and the CLI's --adaptive argument."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import pysqt
from adaptive import ref as AR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_retire_params_layout_matches_ctypes_and_integration_doc(tmp_path):
    """sqt_retire_params: gcc offsetof, the ctypes mirror and the Storable instance of INTEGRATION.md give the same numbers."""
    src = tmp_path / "retire.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqt.h"\nint main(void){ printf("%zu %zu %zu %zu %zu %zu\\n", '
                   'sizeof(sqt_retire_params), _Alignof(sqt_retire_params), offsetof(sqt_retire_params, rel_tol), '
                   'offsetof(sqt_retire_params, abs_tol), offsetof(sqt_retire_params, min_samples), '
                   'offsetof(sqt_retire_params, reserved)); return 0; }\n')
    exe = tmp_path / "retire"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    R = pysqt.RetireParams
    assert got == [C.sizeof(R), C.alignment(R), R.rel_tol.offset, R.abs_tol.offset, R.min_samples.offset, R.reserved.offset]
    assert got == [16, 4, 0, 4, 8, 12]
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    inst = doc[doc.index("instance Storable SqtRetireParams"):]
    inst = inst[:inst.index("```")]
    m = re.search(r"sizeOf _ = (\d+) ; alignment _ = (\d+)", inst)
    assert m and [int(m.group(1)), int(m.group(2))] == got[:2]
    peek = [l for l in inst.splitlines() if l.strip().startswith("peek p")][0]
    assert [int(x) for x in re.findall(r"peekByteOff p (\d+)", peek)] == got[2:5]
    poke = [l for l in inst.splitlines() if l.strip().startswith("poke p")][0]
    assert [int(x) for x in re.findall(r"pokeByteOff p (\d+)", poke)] == got[2:]


def _case(s1, s2):
    return np.array(s1, np.float32).reshape(-1, 3), np.array(s2, np.float32).reshape(-1, 3)


def _edge_cases():
    """(s1, s2, n, rel, abs) sets that reach every branch of the test."""
    cases = []
    f32 = np.float32
    # n = 2, a converged and a noisy pixel
    cases.append(_case([[1.0, 1.0, 1.0], [0.0, 2.0, 0.0]], [[0.5, 0.5, 0.5], [0.0, 4.0, 0.0]]) + (2, 0.1, 0.0))
    # zero sums (black pixel): retires only with abs_tol > 0
    for ab in (0.0, 1e-6):
        cases.append(_case([[0, 0, 0]], [[0, 0, 0]]) + (8, 0.5, ab))
    # a variance that rounds negative: s2 slightly below s1*s1/n
    x = f32(0.1)
    s1 = f32(x * 3)
    cases.append(_case([[s1, s1, s1]], [[np.nextafter(f32(s1 * s1 / 3), f32(0))] * 3]) + (3, 0.01, 0.0))
    # e2 == t*t exactly: one channel, mu = 1, v = 1 -> e2 = 1/4 with n = 4; t = 0.5 (rel 0.5 * m = 1): strict, not retired
    cases.append(_case([[4.0, 0.0, 0.0]], [[7.0, 0.0, 0.0]]) + (4, 0.5, 0.0))
    cases.append(_case([[4.0, 0.0, 0.0]], [[7.0, 0.0, 0.0]]) + (4, 0.0, 0.5))
    cases.append(_case([[4.0, 0.0, 0.0]], [[7.0, 0.0, 0.0]]) + (4, np.nextafter(f32(0.5), f32(1)), 0.0))
    # zero tolerances: nothing retires, not even a constant pixel
    cases.append(_case([[2.0, 2.0, 2.0]], [[1.0, 1.0, 1.0]]) + (4, 0.0, 0.0))
    # NaN and inf inputs
    nan, inf = float("nan"), float("inf")
    cases.append(_case([[nan, 1, 1], [1, 1, 1], [inf, 1, 1], [inf, 1, 1], [1, 1, 1]],
                       [[1, 1, 1], [nan, 0.25, 0.25], [inf, 1, 1], [1, 1, 1], [inf, 0.25, 0.25]]) + (4, 0.5, 0.1))
    cases.append(_case([[inf, 0, 0], [inf, 0, 0]], [[inf, 0, 0], [1, 0, 0]]) + (4, 0.0, 0.1))
    return cases


def test_retire_test_host_build_matches_numpy_on_edge_cases():
    for i, (s1, s2, n, rel, ab) in enumerate(_edge_cases()):
        want = AR.retire_numpy(s1, s2, n, rel, ab)
        assert np.array_equal(AR.retire_emu(s1, s2, n, rel, ab), want), (i, want)
    # the cases above decide as the header says
    c = _edge_cases()
    assert list(AR.retire_numpy(*c[0])) == [True, False]
    assert not AR.retire_numpy(*c[1])[0] and AR.retire_numpy(*c[2])[0]
    assert AR.retire_numpy(*c[3])[0]                            # negative variance clamps to 0 < t*t
    assert not AR.retire_numpy(*c[4])[0] and not AR.retire_numpy(*c[5])[0] and AR.retire_numpy(*c[6])[0]
    assert not AR.retire_numpy(*c[7])[0]
    # NaN anywhere -> never (inf - inf is NaN too); an infinite mean without a NaN has t = inf and retires -- its value
    # cannot change any more
    assert list(AR.retire_numpy(*c[8])) == [False, False, False, True, False]
    assert not AR.retire_numpy(*c[9]).any()                     # rel_tol * inf with rel_tol = 0 is NaN


@pytest.mark.parametrize("n", [2, 3, 16, 64, 1000])
def test_retire_test_host_build_matches_numpy_on_random_pixels(n):
    """Sums and moments of n samples of a random radiance, at several tolerances: every decision agrees."""
    rng = np.random.default_rng(n)
    P = 20000
    scale = rng.choice([0.0, 1e-3, 1.0, 50.0], size=(P, 1))
    x = (rng.exponential(1.0, size=(n, P, 3)) * rng.random((1, P, 3)) * scale).astype(np.float32)
    const = rng.random(P) < 0.2                           # constant pixels: variances that round to either side of 0
    x[:, const] = x[0, const][None]
    s1 = np.zeros((P, 3), np.float32)
    s2 = np.zeros((P, 3), np.float32)
    for k in range(n):
        s1 += x[k]
        s2 += x[k] * x[k]
    for rel, ab in [(0.0, 0.0), (0.01, 0.0), (0.1, 0.0), (0.5, 1e-3), (0.0, 0.01), (2.0, 0.0)]:
        want = AR.retire_numpy(s1, s2, n, rel, ab)
        got = AR.retire_emu(s1, s2, n, rel, ab)
        assert np.array_equal(got, want), (n, rel, ab, int((got != want).sum()))
        if rel == 0.0 and ab == 0.0:
            assert not want.any()
    assert 0 < AR.retire_numpy(s1, s2, n, 0.1, 0.0).sum() < P


def test_noise_reference_with_counts_reduces_to_uniform():
    import progressive_ref as PR
    rng = np.random.default_rng(3)
    s1 = rng.random((6, 5, 3)).astype(np.float32) * 8
    s2 = (s1 * s1 / 8 + rng.random((6, 5, 3)).astype(np.float32)).astype(np.float32)
    assert AR.noise(s1, s2, np.full((6, 5), 8)) == pytest.approx(PR.noise(s1, s2, 8), rel=1e-15)


CLI = os.path.join(ROOT, "squigly-trace_b200", "squigly-trace")


@pytest.mark.parametrize("args", [
    ["--adaptive=0.1"],                                   # without --progress
    ["--progress=4", "--adaptive="],
    ["--progress=4", "--adaptive=-0.1"],
    ["--progress=4", "--adaptive=nan"],
    ["--progress=4", "--adaptive=inf"],
    ["--progress=4", "--adaptive=1e300"],                 # not a float
    ["--progress=4", "--adaptive=0.1x"],
    ["--progress=4", "--adaptive=0.1,,16"],
    ["--progress=4", "--adaptive=0.1,0,1"],               # MIN < 2
    ["--progress=4", "--adaptive=0.1,0,2.5"],
    ["--progress=4", "--adaptive=0.1,0,16,3"],
    ["--progress=4", "--adaptive=0.1,-1"],
])
def test_cli_rejects_malformed_adaptive(args, tmp_path):
    r = subprocess.run([CLI, "-s", "8", "-d", "16,16", "-p", str(tmp_path / "x.png")] + args, cwd=ROOT, capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 1
    assert "--adaptive" in r.stderr and "Rendering scene" not in r.stdout
    assert not (tmp_path / "x.png").exists()
