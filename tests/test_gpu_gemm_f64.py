"""GPU: vb_gemm_f64, the float64 DMMA GEMM behind every product of the sqrtm MultivariateT path and of the GLM
plugins' logp_and_grad, element by element against a long-double reference.

Each output must satisfy |C - C_ref| <= 2 (K + 6) u |alpha| (|A'| diag|kscale| |B'|) |rowscale| / |divm + divn| + |bias|
with u = 2^-53 -- the textbook accumulation bound with room for the scalings -- at every (trans_a, trans_b), at
ragged M, N and K around the 64 x 64 tile and the 32-deep K slab, with each fused epilogue alone and all together,
and with leading dimensions wider than the rows.  A, B and their padding are read through views into wider buffers
whose padding holds NaN, so a read outside the operands poisons the result, and C's buffer is filled with a sentinel
that must survive outside the M x N window.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
LD = np.longdouble
MN = [1, 63, 64, 65, 129]
EPILOGUES = ['none', 'kscale', 'rowscale', 'bias', 'div', 'all']
SENTINEL = -7.25e300
MAX_RATIO = [0.0]


@pytest.fixture(scope='module', autouse=True)
def _report():
    yield
    print('[gemm_f64] largest |C - C_ref| / ((K + 6) u |A||B|) = %.3g' % MAX_RATIO[0])


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


def _addr(t, offset=0):
    return t.data_ptr() + 8 * offset


class _Operands:
    """Stored A (K x M if trans_a else M x K) and B (N x K if trans_b else K x N), rows padded with NaN columns."""

    def __init__(self, rs, ta, tb, M, N, K, pad=5):
        self.ta, self.tb, self.M, self.N, self.K = ta, tb, M, N, K
        ra, ca = (K, M) if ta else (M, K)
        rb, cb = (N, K) if tb else (K, N)
        self.lda, self.ldb = ca + pad, cb + pad + 2
        a = np.full((max(ra, 1), self.lda), np.nan)
        b = np.full((max(rb, 1), self.ldb), np.nan)
        a[:ra, :ca] = rs.randn(ra, ca)
        b[:rb, :cb] = rs.randn(rb, cb)
        self.a, self.b = a, b
        self.Ap = a[:ra, :ca].T if ta else a[:ra, :ca]                    # A'(m, k)
        self.Bp = b[:rb, :cb].T if tb else b[:rb, :cb]                    # B'(k, n)
        self.kscale = rs.uniform(-2.0, 2.0, K)
        self.rowscale = rs.uniform(-2.0, 2.0, M)
        self.bias = rs.randn(N)
        self.divm, self.divn = rs.uniform(0.5, 1.5, M), rs.uniform(0.5, 1.5, N)
        self.dev = {k: torch.as_tensor(getattr(self, k), device='cuda')
                    for k in ('a', 'b', 'kscale', 'rowscale', 'bias', 'divm', 'divn')}
        Al, Bl = self.Ap.astype(LD), self.Bp.astype(LD)
        ks = self.kscale.astype(LD)
        self.prod = {False: Al @ Bl, True: (Al * ks) @ Bl}
        self.absprod = {False: np.abs(Al) @ np.abs(Bl), True: (np.abs(Al) * np.abs(ks)) @ np.abs(Bl)}


def _run(vb, op, M, N, epi, alpha, pad_c=(1, 2, 7)):
    """C[M,N] into a sentinel-filled buffer at row offset r0, column offset c0, ldc = N + extra; returns the window
    and asserts nothing else changed."""
    lib, cl = vb._lib.lib, vb._lib
    r0, c0, extra = pad_c
    ldc = N + c0 + extra
    buf = torch.full((M + r0 + 2, ldc), SENTINEL, dtype=torch.float64, device='cuda')
    use = lambda name: op.dev[name] if (epi == 'all' or epi == name or (epi == 'div' and name in ('divm', 'divn'))) else None
    addr = lambda t: None if t is None else t.data_ptr()
    ks, rsc, bias, dm, dn = (use(n) for n in ('kscale', 'rowscale', 'bias', 'divm', 'divn'))
    cl.check(lib.vb_gemm_f64(int(op.ta), int(op.tb), M, N, op.K, alpha, _addr(op.dev['a']), op.lda, _addr(op.dev['b']), op.ldb,
                             _addr(buf, r0 * ldc + c0), ldc, addr(ks), addr(rsc), addr(bias), addr(dm), addr(dn),
                             vb._lib.stream()))
    h = buf.cpu().numpy()
    win = h[r0:r0 + M, c0:c0 + N].copy()
    h[r0:r0 + M, c0:c0 + N] = SENTINEL
    assert (h == SENTINEL).all(), 'gemm_f64 wrote outside the M x N window'
    return win, ks is not None, rsc is not None, bias is not None, dm is not None


def _check(op, M, N, epi, alpha, win, has_ks, has_rs, has_bias, has_div):
    K = op.K
    ref = LD(alpha) * op.prod[has_ks][:M, :N]
    bound = abs(LD(alpha)) * op.absprod[has_ks][:M, :N]
    if has_rs:
        ref = ref * op.rowscale[:M, None].astype(LD)
        bound = bound * np.abs(op.rowscale[:M, None]).astype(LD)
    if has_div:
        den = op.divm[:M, None].astype(LD) + op.divn[None, :N].astype(LD)
        ref, bound = ref / den, bound / den
    if has_bias:
        ref = ref + op.bias[None, :N].astype(LD)
        bound = bound + np.abs(op.bias[None, :N]).astype(LD)
    assert np.isfinite(win).all(), (epi, M, N, K)
    err = np.abs(win.astype(LD) - ref)
    scale = (K + 6) * LD(U) * bound
    bad = err > 2 * scale
    assert not bad.any(), (epi, M, N, K, int(bad.sum()))
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(scale > 0, err / scale, 0.0)
    MAX_RATIO[0] = max(MAX_RATIO[0], float(np.max(r)))


@pytest.mark.parametrize('K', [0, 1, 31, 32, 33, 2048])
@pytest.mark.parametrize('ta,tb', [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_gemm_f64_componentwise(vb, ta, tb, K):
    """Every M, N in {1, 63, 64, 65, 129} with each epilogue alone and all together.  The smaller problems are the
    leading rows / columns of one 129 x 129 problem, so a long-double reference of that one serves them all."""
    rs = np.random.RandomState(100 * K + 10 * ta + tb)
    op = _Operands(rs, bool(ta), bool(tb), max(MN), max(MN), K)
    for M in MN:
        for N in MN:
            for epi in EPILOGUES:
                alpha = -1.25 if epi == 'all' else 0.75
                _check(op, M, N, epi, alpha, *_run(vb, op, M, N, epi, alpha))


@pytest.mark.parametrize('big', ['M', 'N'])
def test_gemm_f64_past_65535_row_tiles(vb, big):
    """M = 4 200 000 (65 625 tiles of 64 rows) with N = K = 3, and the same for N: the tile grid is one-dimensional,
    so neither size is capped at 65 535 tiles.  All epilogues on."""
    n = 4_200_000
    M, N, K = (n, 3, 3) if big == 'M' else (3, n, 3)
    rs = np.random.RandomState(42)
    A = rs.randn(M, K)
    B = rs.randn(K, N)
    ks, rsc, bias = rs.uniform(-2, 2, K), rs.uniform(-2, 2, M), rs.randn(N)
    dm, dn = rs.uniform(0.5, 1.5, M), rs.uniform(0.5, 1.5, N)
    t = lambda a: torch.as_tensor(a, device='cuda')
    Ad, Bd, C = t(A), t(B), torch.full((M, N), float('nan'), dtype=torch.float64, device='cuda')
    dev = [t(x) for x in (ks, rsc, bias, dm, dn)]
    vb._lib.check(vb._lib.lib.vb_gemm_f64(0, 0, M, N, K, 1.5, Ad.data_ptr(), K, Bd.data_ptr(), N, C.data_ptr(), N,
                                          *[x.data_ptr() for x in dev], vb._lib.stream()))
    c = C.cpu().numpy()
    assert np.isfinite(c).all()
    Al = A.astype(LD) * ks.astype(LD)
    den = dm[:, None].astype(LD) + dn[None, :].astype(LD)
    ref = LD(1.5) * (Al @ B.astype(LD)) * rsc[:, None].astype(LD) / den + bias[None, :].astype(LD)
    bound = LD(1.5) * (np.abs(Al) @ np.abs(B).astype(LD)) * np.abs(rsc[:, None]).astype(LD) / den + np.abs(bias[None, :]).astype(LD)
    err = np.abs(c.astype(LD) - ref)
    assert (err <= 2 * (K + 6) * LD(U) * bound).all()
