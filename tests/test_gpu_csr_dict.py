"""GPU: the dictionary-encoded CSR stream (Csr::code, one byte per nonzero into a table of (column - row, value)
pairs).  The encoded staged SpMV must be bit-identical to the row-per-thread CSR kernel, and a whole persistent CG
solve on the encoded operator bit-identical to the same solve on the CSR stream (KB200_CSR_DICT=0 at upload)."""
import contextlib
import ctypes as C
import os
import time

import numpy as np
import pytest

from krylov_b200 import _lib
from krylov_b200 import problems as P

pytestmark = pytest.mark.gpu
DT = {np.float64: _lib.KRYLOV_FLOAT64, np.float32: _lib.KRYLOV_FLOAT32}


@contextlib.contextmanager
def csr_stream():
    """Operators uploaded inside keep the CSR stream (the plan reads KB200_CSR_DICT)."""
    old = os.environ.get("KB200_CSR_DICT")
    os.environ["KB200_CSR_DICT"] = "0"
    try:
        yield
    finally:
        if old is None:
            del os.environ["KB200_CSR_DICT"]
        else:
            os.environ["KB200_CSR_DICT"] = old


def distinct_pairs(rp, ci, va):
    rows = np.repeat(np.arange(len(rp) - 1, dtype=np.int64), np.diff(rp))
    off = ci.astype(np.int64) - rows
    bits = va.view(np.uint64 if va.dtype == np.float64 else np.uint32).astype(np.uint64)
    return len(set(zip(off.tolist(), bits.tolist())))


class Dev:
    def __init__(self):
        self.L = _lib.lib()
        self.ctx = self.L.kb200_ctx_create(-1)
        assert self.ctx
        self.bufs = []

    def put(self, a):
        a = np.ascontiguousarray(a)
        p = self.L.kb200_alloc(max(a.nbytes, 8))
        assert p
        self.L.kb200_h2d(p, a.ctypes.data_as(C.c_void_p), a.nbytes)
        self.bufs.append(p)
        return p

    def get(self, p, n, dt):
        out = np.empty(n, dt)
        self.L.kb200_sync(self.ctx)
        self.L.kb200_d2h(out.ctypes.data_as(C.c_void_p), p, out.nbytes)
        return out

    def csr(self, rp, ci, va, base=0, ibytes=4):
        it = np.int32 if ibytes == 4 else np.int64
        rp, ci = np.ascontiguousarray(rp + base, dtype=it), np.ascontiguousarray(ci + base, dtype=it)
        va = np.ascontiguousarray(va)
        h = self.L.kb200_csr_create(self.ctx, DT[va.dtype.type], len(rp) - 1, len(va), rp.ctypes.data_as(C.c_void_p),
                                    ci.ctypes.data_as(C.c_void_p), va.ctypes.data_as(C.c_void_p), base, ibytes, 0)
        assert h, _lib.last_error()
        return h

    def close(self):
        for p in self.bufs:
            self.L.kb200_free(p)
        self.L.kb200_ctx_destroy(self.ctx)


@pytest.fixture()
def dev():
    d = Dev()
    yield d
    d.close()


def encoding_of(kb, dev, csr, n, dt):
    """Dictionary size of a kb200_csr_create operator, read through a workspace it is attached to."""
    ws = kb.CgWorkspace(n, n, dt)
    try:
        assert dev.L.krylov_b200_attach_csr(ws._h, csr) == 0, _lib.last_error()
        return dev.L.krylov_b200_operator_encoding(ws._h)
    finally:
        ws.free()


def check_spmv(kb, dev, rp, ci, va, base=0, ibytes=4):
    """Staged SpMV on the encoded operator == rows kernel; returns the dictionary size."""
    dt = va.dtype.type
    n = len(rp) - 1
    x = np.random.default_rng(n).standard_normal(n).astype(dt)
    px, py1, py2 = dev.put(x), dev.put(np.zeros(n, dt)), dev.put(np.zeros(n, dt))
    csr = dev.csr(rp, ci, va, base, ibytes)
    try:
        nd = encoding_of(kb, dev, csr, n, dt)
        assert dev.L.kb200_spmv_csr(dev.ctx, csr, px, py1, 1) == 0, _lib.last_error()
        assert dev.L.kb200_spmv_csr(dev.ctx, csr, px, py2, 2) == 0, _lib.last_error()
        assert np.array_equal(dev.get(py1, n, dt), dev.get(py2, n, dt)), "encoded staged SpMV differs from the rows kernel"
    finally:
        dev.L.kb200_csr_destroy(csr)
    return nd


def pair_matrix(npairs, dt, n=4096):
    """All 256 (offset, value) pairs of offsets 0..15 and 16 values: row i holds the offsets o = i % 4 (mod 4) with
    value vals[(i // 4 + o) % 16]; every 50th row holds all 16 offsets (rows longer than one gather batch) and every
    97th row is empty.  Rows stay short enough on average for the default 3-CTA/SM tile plan.  npairs = 257 adds the
    pair (16, vals[0]) to row 0."""
    vals = (1.0 + np.arange(16) / 8.0).astype(dt)
    rp, ci, va = [0], [], []
    for i in range(n):
        if i % 97 != 5:
            offs = range(16) if i % 50 == 7 else range(i % 4, 16, 4)
            ent = [(i + o, vals[(i // 4 + o) % 16]) for o in offs if i + o < n]
            if npairs == 257 and i == 0:
                ent.append((16, vals[0]))
            ci += [c for c, _ in ent]
            va += [v for _, v in ent]
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(va, dt)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_encoded_spmv_stencils(kb, dev, dt):
    for rp, ci, va in (P.div_grad_csr(64, dtype=dt), P.kron_unsymmetric_csr(48, dtype=dt)):
        nd = check_spmv(kb, dev, rp, ci, va)
        assert nd == distinct_pairs(rp, ci, va) and 0 < nd <= 7, nd


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_encoded_spmv_dictionary_limit(kb, dev, dt):
    rp, ci, va = pair_matrix(256, dt)
    assert distinct_pairs(rp, ci, va) == 256
    assert check_spmv(kb, dev, rp, ci, va) == 256                 # full dictionary: long rows and empty rows encoded
    rp, ci, va = pair_matrix(257, dt)
    assert distinct_pairs(rp, ci, va) == 257
    assert check_spmv(kb, dev, rp, ci, va) == 0                   # one pair too many: CSR stream


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_encoded_spmv_signed_zeros(kb, dev, dt):
    rp, ci, va = P.div_grad_csr(16, dtype=dt)
    va = va.copy()
    k = rp[3]
    va[k], va[k + 1] = dt(0.0), -dt(0.0)                          # row 3 stores both zeros
    va[rp[100] + 1] = -dt(0.0)                                     # -0.0 at another offset
    nd = check_spmv(kb, dev, rp, ci, va)
    assert nd == distinct_pairs(rp, ci, va) > 7, nd               # 0.0 and -0.0 are different entries


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("base,ibytes", [(1, 4), (0, 8), (1, 8)])
def test_encoded_spmv_after_index_conversion(kb, dev, dt, base, ibytes):
    rp, ci, va = P.div_grad_csr(24, dtype=dt)
    assert check_spmv(kb, dev, rp, ci, va, base, ibytes) == distinct_pairs(rp, ci, va)


def _solve_pair(kb, csr, n, b, M=None):
    out = []
    for encoded in (True, False):
        ws = kb.CgWorkspace(n, n, np.float64)
        if encoded:
            ws.set_operator(csr)
        else:
            with csr_stream():
                ws.set_operator(csr)
        enc = _lib.lib().krylov_b200_operator_encoding(ws._h)
        assert (enc > 0) == encoded, enc
        ws.solve(None, b, M=M, atol=0.0, rtol=0.0, itmax=200, history=True)
        st = ws.stats
        out.append((st.niter, list(st.residuals), ws.x.copy(), ws.vector("r")))
        ws.free()
    (n1, h1, x1, r1), (n2, h2, x2, r2) = out
    assert n1 == n2 == 200
    assert h1 == h2, "residual histories differ"
    assert np.array_equal(x1, x2) and np.array_equal(r1, r2)


def test_persistent_cg_encoded_vs_csr_cfg2(kb):
    """cg! on get_div_grad(215) (the benchmark operator), 200 iterations: the encoded persistent kernel reproduces
    the CSR kernel bit for bit (same grid, same reduction trees), without and with a Jacobi M."""
    N = 215
    csr = P.div_grad_csr(N)
    n = N ** 3
    b = np.ones(n)
    _solve_pair(kb, csr, n, b)
    _solve_pair(kb, csr, n, b, M=1.0 / (6.0 + np.arange(n) % 5))


def test_random_operator_is_not_encoded(kb, dev):
    """The cfg4 random matrix (n = 5e6, ~1e8 nonzeros) has far more than 256 pairs: it keeps the CSR stream, and the
    encoder gives up early (set-up times printed for the record)."""
    rp, ci, va = P.random_csr(5_000_000)
    t = {}
    for label, ctx in (("encoding attempted", contextlib.nullcontext()), ("KB200_CSR_DICT=0", csr_stream())):
        with ctx:
            t0 = time.perf_counter()
            h = dev.csr(rp, ci, va)
            dev.L.kb200_sync(dev.ctx)
            t[label] = time.perf_counter() - t0
        nd = encoding_of(kb, dev, h, len(rp) - 1, np.float32)
        dev.L.kb200_csr_destroy(h)
        assert nd == 0, nd
    print("cfg4 operator upload + plan: " + ", ".join(f"{k} {v:.3f} s" for k, v in t.items()))
