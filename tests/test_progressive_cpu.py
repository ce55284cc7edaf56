"""Progressive frames (include/sqt.h), the parts that need no GPU: the sqt_progress layout, the oracle's range render and
the host build of the second-moment accumulation."""
import os
import re
import subprocess

import numpy as np
import pytest

import progressive_ref as PR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_progress_layout_matches_ctypes_and_integration_doc(tmp_path):
    """sqt_progress: gcc offsetof, the ctypes mirror and the Storable instance of INTEGRATION.md give the same numbers."""
    import ctypes as C
    import pysqt
    src = tmp_path / "progress.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqt.h"\nint main(void){ printf("%zu %zu %zu %zu %zu\\n", '
                   'sizeof(sqt_progress), _Alignof(sqt_progress), offsetof(sqt_progress, samples_done), '
                   'offsetof(sqt_progress, samples_total), offsetof(sqt_progress, noise)); return 0; }\n')
    exe = tmp_path / "progress"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    P = pysqt.Progress
    assert got == [C.sizeof(P), C.alignment(P), P.samples_done.offset, P.samples_total.offset, P.noise.offset]
    assert got == [16, 8, 0, 4, 8]
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    inst = doc[doc.index("instance Storable SqtProgress"):]
    inst = inst[:inst.index("```")]
    m = re.search(r"sizeOf _ = (\d+) ; alignment _ = (\d+)", inst)
    assert m and [int(m.group(1)), int(m.group(2))] == got[:2]
    peek = [l for l in inst.splitlines() if l.strip().startswith("peek p")][0]
    assert [int(x) for x in re.findall(r"peekByteOff p (\d+)", peek)] == got[2:]


@pytest.fixture(scope="module")
def small(oracle_scene, camera):
    from oracle import oracle as O
    return oracle_scene, camera, O


@pytest.mark.parametrize("literal", [False, True])
def test_range_render_chunked_equals_one_range_and_orc_render(small, literal):
    scene, cam, O = small
    spp = 11
    p = O.make_params(40, 28, spp, max_depth=4, seed=7, trig=1, literal=literal)
    a1, q1 = PR.render_range(scene, cam, p, 0, spp)
    a, q = PR.render_range(scene, cam, p, 0, 3)
    a, q = PR.render_range(scene, cam, p, 3, 8, a, q)
    a, q = PR.render_range(scene, cam, p, 8, spp, a, q)
    assert np.array_equal(a.view(np.uint32), a1.view(np.uint32))
    assert np.array_equal(q.view(np.uint32), q1.view(np.uint32))
    ref = scene.render(cam, p)
    assert np.array_equal(a1.view(np.uint32), ref["accum"].view(np.uint32))
    assert (q1 > 0).any() and (q1 >= 0).all()


def test_emu_m2_slot_matches_oracle_range(small):
    """accumulate_m2_slot (the function k_accumulate_m2 runs per slot), fed with the oracle's per-sample radiances in rounds of
    uneven size, gives the oracle's sums and second moments bit for bit."""
    scene, cam, O = small
    spp, rows, cols = 9, 24, 32
    p = O.make_params(cols, rows, spp, max_depth=5, seed=2, trig=1)
    # sample k alone, started from +0, is the radiance x_k itself (0 + x = x, 0 + x*x = x*x)
    xs = np.stack([PR.render_range(scene, cam, p, k, k + 1)[0].reshape(-1, 3) for k in range(spp)])
    accum = np.zeros((rows * cols, 3), np.float32)
    m2 = np.zeros((rows * cols, 3), np.float32)
    for k0, k1 in [(0, 4), (4, 5), (5, 9)]:
        PR.accumulate_m2(rows, cols, spp, xs[k0:k1], k0, k1, accum, m2)
    ra, rq = PR.render_range(scene, cam, p, 0, spp)
    assert np.array_equal(accum.view(np.uint32), ra.reshape(-1, 3).view(np.uint32))
    assert np.array_equal(m2.view(np.uint32), rq.reshape(-1, 3).view(np.uint32))
    assert (xs > 0).any()


def test_noise_reference_definition():
    s1 = np.array([[2.0, 0.0, 4.0]], np.float32)
    s2 = np.array([[2.5, 0.0, 9.0]], np.float32)
    n = 4
    mu = s1.astype(np.float64) / n
    var = np.maximum(0, (s2 - s1 * mu) / (n - 1))
    want = np.sqrt((var / n).sum() / 3) / (mu.sum() / 3)
    assert PR.noise(s1, s2, n) == pytest.approx(want, rel=1e-15)
    assert PR.noise(s1, s2, 1) == float("inf")
    assert PR.noise(np.zeros(6), np.zeros(6), 5) == 0.0
