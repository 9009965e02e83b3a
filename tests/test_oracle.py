"""CPU tests: the oracle (oracle/finc_oracle.c + .py) against the reference's own outputs.

Pins the oracle with
  * tests/golden/finc_golden_*.npz -- produced by importing the reference's PaddedConv2d /
    FastFlowUnit and its Cython solver (tests/golden/make_golden.py);
  * the integer known-answer inputs of cuda/cinc_cuda/test_cuda_kernel.py and
    fastflow/test_examples.py (SURVEY.md appendix E) with hand-checkable answers;
  * oracle/_ref: the reference's solve_parallel_mc.pyx compiled from its own source
    (bit-exact comparison in f64);
  * a dense-matrix cross check (cf. misc/solve_mc.py:118-144).
"""
import numpy as np
import pytest

from conftest import Golden, rel_err
from oracle import build_ref
from oracle import finc_oracle as fo

_G = Golden()
FULL = [n for n in _G.names if not n.startswith("kat_")]
KATS = [n for n in _G.names if n.startswith("kat_")]


@pytest.mark.parametrize("name", FULL)
def test_forward_matches_reference(golden, name):
    c = golden.case(name)
    orders = tuple(int(o) for o in c["orders"])
    z64 = fo.forward(c["x"], c["w"], orders, dtype=np.float64)
    z32 = fo.forward(c["x"], c["w"], orders, dtype=np.float32)
    # reference z is torch fp32 CPU conv: only accumulation order differs
    assert rel_err(c["z"], z64) <= 2e-6
    assert rel_err(z32, z64) <= 2e-6


@pytest.mark.parametrize("name", FULL)
def test_backward_matches_reference(golden, name):
    c = golden.case(name)
    orders = tuple(int(o) for o in c["orders"])
    k = c["w"].shape[2:]
    dx = fo.backward_input(c["dz"], c["w"], orders)
    assert rel_err(c["dx"], dx) <= 2e-6
    dw_raw = fo.backward_weight(c["dz"], c["x"], k, orders, apply_mask=False)
    assert rel_err(c["dw_raw"], dw_raw) <= 5e-6
    dw_m = fo.backward_weight(c["dz"], c["x"], k, orders, apply_mask=True)
    assert rel_err(c["dw_masked"], dw_m) <= 5e-6
    # the mask zeroes exactly the entries the reference zeroes (conv.py:81-99)
    assert np.array_equal(c["dw_masked"] == 0, dw_m == 0)
    assert np.array_equal(fo.apply_grad_mask(dw_raw, orders), dw_m)


@pytest.mark.parametrize("name", FULL)
def test_inverse_bit_exact_vs_reference_solver(golden, name):
    """The reference computes the inverse in float64 from the fp32 tensors and casts back
    (conv.py:118-163); same subtraction order => bit-identical."""
    c = golden.case(name)
    orders = tuple(int(o) for o in c["orders"])
    y = fo.inverse(c["zs"], c["w"], orders, dtype=np.float64).astype(np.float32)
    assert np.array_equal(y, c["x_from_zs"])
    y = fo.inverse(c["z"], c["w"], orders, dtype=np.float64).astype(np.float32)
    assert np.array_equal(y, c["x_rt"])
    # and the round trip closes (north_star: <= 1e-4 max-abs)
    assert np.abs(c["x_rt"] - c["x"]).max() <= 1e-4
    # fp32 evaluation of the same recurrence stays within the fp32 tolerance
    y32 = fo.inverse(c["zs"], c["w"], orders, dtype=np.float32)
    assert rel_err(y32, c["x_from_zs"]) <= 1e-5


@pytest.mark.parametrize("name", KATS)
def test_known_answer_vectors(golden, name):
    c = golden.case(name)
    orders = tuple(int(o) for o in c["orders"])
    y = fo.inverse(c["zs"], c["w"], orders, dtype=np.float32)
    assert np.array_equal(y, c["x_from_zs"])  # small integers: exact
    assert np.array_equal(fo.forward(y, c["w"], orders, dtype=np.float32), c["zs"])
    if "z" in c:
        assert np.array_equal(fo.forward(c["x"], c["w"], orders, dtype=np.float32), c["z"])


def test_known_answers_by_hand():
    """SURVEY.md appendix E rows, typed in independently of the fixture file."""
    g = np.arange(1, 17, dtype=np.float64).reshape(1, 1, 4, 4)
    w = np.array([[1, 0], [0, 1]], dtype=np.float64).reshape(1, 1, 2, 2)
    want = [[1, 2, 3, 4], [5, 5, 5, 5], [9, 5, 6, 7], [13, 5, 10, 10]]
    assert np.array_equal(fo.inverse(g, w, (0,))[0, 0], np.array(want, dtype=np.float64))
    w3 = np.eye(3).reshape(1, 1, 3, 3)
    want = [[1, 2, 3, 4], [5, 5, 5, 5], [9, 5, 5, 5], [13, 5, 5, 6]]
    assert np.array_equal(fo.inverse(g, w3, (0,))[0, 0], np.array(want, dtype=np.float64))
    # TR, stored weight [[0,2],[1,0]]: z[h,w] = x[h,w] + 2 x[h-1,w+1]
    x = np.arange(1, 10, dtype=np.float64).reshape(1, 1, 3, 3)
    wtr = np.array([[0, 2], [1, 0]], dtype=np.float64).reshape(1, 1, 2, 2)
    z = fo.forward(x, wtr, (1,))
    assert np.array_equal(z[0, 0], np.array([[1, 2, 3], [8, 11, 6], [17, 20, 9]], dtype=np.float64))
    assert np.array_equal(fo.inverse(z, wtr, (1,)), x)
    # BL, stored weight [[0,1],[1,0]]: z[h,w] = x[h,w] + x[h+1,w-1]
    wbl = np.array([[0, 1], [1, 0]], dtype=np.float64).reshape(1, 1, 2, 2)
    z = fo.forward(x, wbl, (2,))
    assert np.array_equal(z[0, 0], np.array([[1, 6, 8], [4, 12, 14], [7, 8, 9]], dtype=np.float64))
    assert np.array_equal(fo.inverse(z, wbl, (2,)), x)


def test_c_oracle_vs_literal_python_and_dense_matrix():
    rng = np.random.default_rng(7)
    for (C, H, W, k) in [(2, 4, 5, (3, 3)), (3, 5, 4, (2, 3)), (1, 6, 6, (5, 5)), (4, 3, 3, (3, 2))]:
        for order in ("TL", "TR", "BL", "BR"):
            w = fo.init_weight(C, k, order, rng, std=0.2, dtype=np.float64)
            x = rng.normal(size=(2, C, H, W))
            z = fo.forward(x, w, (order,))
            assert np.allclose(z, fo.forward_py(x, w, (order,)), rtol=0, atol=1e-13)
            M = fo.dense_matrix(w, H, W, order)
            assert np.allclose(z.reshape(2, -1), x.reshape(2, -1) @ M.T, rtol=0, atol=1e-13)
            # unit-triangular Jacobian => det 1 => logdet 0 (conv.py:106)
            assert abs(np.linalg.slogdet(M)[1]) < 1e-10
            assert fo.logdet(w, H, W, (order,)) == 0.0
            y = fo.inverse(z, w, (order,))
            assert np.array_equal(y, fo.inverse_py(z, w, (order,)))
            assert np.allclose(y, np.linalg.solve(M, z.reshape(2, -1).T).T.reshape(x.shape),
                               rtol=0, atol=1e-11)
            dz = rng.normal(size=x.shape)
            dx = fo.backward_input(dz, w, (order,))
            assert np.allclose(dx.reshape(2, -1), dz.reshape(2, -1) @ M, rtol=0, atol=1e-13)


def test_oracle_vs_compiled_reference_solver_f64(golden):
    """oracle/_ref = the reference's .pyx compiled from its own source.  Without it (it is built only from a
    reference checkout, FINCFLOW_REFERENCE) the oracle's f64 solve is compared bit for bit with what that
    solver returned for the stored single-convolution cases, which include H < W."""
    ref = build_ref.load()
    if ref is None:
        for name in (n for n in FULL if n.startswith("conv_")):
            c = golden.case(name)
            orders = tuple(int(o) for o in c["orders"])
            assert np.array_equal(fo.inverse(c["zs"], c["w"], orders, dtype=np.float64).astype(np.float32),
                                  c["x_from_zs"]), name
        return
    rng = np.random.default_rng(3)
    for (B, C, H, W, k) in [(3, 4, 14, 14, (3, 3)), (2, 3, 16, 16, (5, 5)), (2, 12, 4, 4, (3, 3)),
                            (2, 3, 5, 9, (2, 3)), (1, 24, 4, 4, (5, 5))]:
        w = fo.init_weight(C, k, "TL", rng, dtype=np.float64)
        z = rng.normal(size=(B, C, H, W))
        want = ref.solve_parallel(z.copy(), w, k)  # mutates its input (.pyx:85)
        assert np.array_equal(fo.inverse(z, w, (0,)), want)


def test_unit_is_four_independent_groups():
    rng = np.random.default_rng(5)
    Cq, H, W, k = 3, 6, 7, (3, 3)
    w = fo.init_unit_weight(Cq, k, rng, dtype=np.float64)
    x = rng.normal(size=(2, 4 * Cq, H, W))
    z = fo.forward(x, w)
    for g in range(4):
        sl = slice(g * Cq, (g + 1) * Cq)
        assert np.array_equal(z[:, sl], fo.forward(x[:, sl], w[sl], (g,)))
    assert rel_err(fo.inverse(z, w), x) < 1e-12


def test_edge_shapes():
    rng = np.random.default_rng(11)
    # empty batch, 1x1 image, kernel larger than the image, H > W (reference's Cython
    # solver is wrong there, solve_parallel_mc.pyx:95-98; the oracle is not)
    w = fo.init_unit_weight(2, (3, 3), rng, dtype=np.float64)
    assert fo.forward(np.zeros((0, 8, 4, 4)), w).shape == (0, 8, 4, 4)
    for (H, W) in [(1, 1), (2, 2), (9, 5), (1, 7)]:
        x = rng.normal(size=(2, 8, H, W))
        assert rel_err(fo.inverse(fo.forward(x, w), w), x) < 1e-12
