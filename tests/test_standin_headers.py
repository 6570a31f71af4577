"""The stand-in Eigen / iDynTree headers (oracle/refbuild/standin) checked ON THEIR OWN against numpy.

The claim "parity is pinned against the reference's own sources" rests on these headers doing what
Eigen and iDynTree document: storage orders and maps, block views, products and their association,
inverses, LLT solve, cross products, aliasing-safe assignment, RPY and the rotation exponential.
oracle/_ref/libstandin_selftest.so (built with assertions enabled) exports one function per group;
none of the reference's code is involved, so it is built wherever the repository is."""
import ctypes as C
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def st():
    from oracle import ref_binding
    ref_binding.build()
    return C.CDLL(os.path.join(ref_binding.REF_DIR, "libstandin_selftest.so"))


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def close(a, b, tol=1e-13):
    return np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max())


def test_dynamic_row_major_products(st):
    rng = np.random.default_rng(0)
    for m, k, n in [(1, 1, 1), (3, 3, 3), (6, 2, 1), (2, 6, 6), (7, 5, 3), (35, 6, 1)]:
        A, B = rng.normal(size=(m, k)), rng.normal(size=(k, n))
        out = np.empty((m, n))
        st.st_matmul(m, k, n, p(A), p(B), p(out))
        assert close(out, A @ B), (m, k, n)


def test_fixed_size_chain_transpose_and_left_to_right_association(st):
    rng = np.random.default_rng(1)
    for _ in range(50):
        A, x = rng.normal(size=(3, 3)), rng.normal(size=3)
        s, t = rng.normal(), rng.normal()
        y = np.empty(3)
        st.st_fixed3_chain(p(A), p(x), C.c_double(s), C.c_double(t), p(y))
        assert close(y, ((s * A) @ A) @ x + t * (A.T @ x))


def test_inverses_and_llt_solve(st):
    rng = np.random.default_rng(2)
    for _ in range(50):
        A = rng.normal(size=(3, 3)) + 3 * np.eye(3)
        out = np.empty((3, 3))
        st.st_inverse3(p(A), p(out))
        assert close(out @ A, np.eye(3), 1e-12) and close(out, np.linalg.inv(A), 1e-12)
    for n in (1, 2, 4, 6, 12, 35):
        A = rng.normal(size=(n, n)) + n * np.eye(n)
        out = np.empty((n, n))
        st.st_inverse_dyn(n, p(A), p(out))
        assert close(out, np.linalg.inv(A), 1e-11), n
        Bm = rng.normal(size=(n, n))
        S = Bm @ Bm.T + n * np.eye(n)
        b, x = rng.normal(size=n), np.empty(n)
        st.st_llt_solve(n, p(S), p(b), p(x))
        assert close(x, np.linalg.solve(S, b), 1e-11), n
    # identity mass matrix: the solve must hand the right-hand side back bit for bit (what the
    # J^T wrench pin relies on, oracle/refbuild/ref_driver.cpp)
    b, x = rng.normal(size=29), np.empty(29)
    st.st_llt_solve(29, p(np.eye(29)), p(b), p(x))
    assert np.array_equal(x, b)


def test_skew_cross_and_colwise_cross(st):
    rng = np.random.default_rng(3)
    for _ in range(50):
        v, w, R = rng.normal(size=3), rng.normal(size=3), rng.normal(size=(3, 3))
        out = np.empty(21)
        st.st_cross_ops(p(v), p(w), p(R), p(out))
        S = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
        assert np.array_equal(out[:9].reshape(3, 3), S)
        assert close(out[9:12], np.cross(v, w))
        assert close(out[12:].reshape(3, 3), np.stack([np.cross(R[:, j], w) for j in range(3)], axis=1))
        assert close(S @ w, np.cross(v, w))


def test_block_views_write_where_eigen_would(st):
    rng = np.random.default_rng(4)
    B, h, t, d = rng.normal(size=(3, 3)), rng.normal(size=3), rng.normal(size=3), 2.5
    g, f, reg = np.empty((6, 6)), np.empty(6), np.empty((6, 2))
    st.st_block_writes(C.c_double(d), p(B), p(h), p(t), p(g), p(f), p(reg))
    want = np.zeros((6, 6))
    want[0, 0] = want[1, 1] = want[2, 2] = d
    want[3:, 3:] = B
    assert np.array_equal(g, want)
    assert np.array_equal(f, np.concatenate([h, t]))
    wr = np.zeros((6, 2))
    wr[:3, 1], wr[3:, 0] = h, t
    assert np.array_equal(reg, wr)


def test_assignment_through_aliasing_maps(st):
    rng = np.random.default_rng(5)
    for pdim, m in [(2, 6), (4, 3), (1, 1)]:
        K, Y, z = rng.normal(size=(pdim, m)), rng.normal(size=(m, pdim)), rng.normal(size=m)
        x0, P0, lam = rng.normal(size=pdim), rng.normal(size=(pdim, pdim)), 0.97
        x, P = x0.copy(), P0.copy()
        st.st_aliasing_update(pdim, m, p(K), p(Y), p(z), C.c_double(lam), p(x), p(P))
        assert close(x, x0 + K @ (z - Y @ x0)) and close(P, (P0 - K @ Y @ P0) / lam)


def test_as_diagonal_rpy_and_exponential(st):
    rng = np.random.default_rng(6)
    v, out = rng.normal(size=5), np.empty((5, 5))
    st.st_as_diagonal(5, p(v), p(out))
    assert np.array_equal(out, np.diag(v))
    for _ in range(20):
        r, pi_, y = rng.uniform(-3, 3, 3)
        R = np.empty((3, 3))
        st.st_rpy(C.c_double(r), C.c_double(pi_), C.c_double(y), p(R))
        cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(pi_), np.sin(pi_), np.cos(y), np.sin(y)
        Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
        Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
        Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
        assert close(R, Rz @ Ry @ Rx)
        w = rng.normal(size=3) * rng.choice([1e-12, 1e-3, 1.0, 3.0])
        E = np.empty((3, 3))
        st.st_exp(p(w), p(E))
        th = np.linalg.norm(w)
        K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
        want = np.eye(3) + (np.sin(th) / th if th > 1e-9 else 1.0) * K + \
            ((1 - np.cos(th)) / th ** 2 if th > 1e-9 else 0.5) * K @ K
        assert close(E, want) and close(E @ E.T, np.eye(3), 1e-12)
