"""The tensor-core GLM sweep (vb_glm_fast_sweep) element by element against a float64 reference, through the C ABI.

Per-element budgets come from the kernel's numerics (tests/_glm_fast_ref.py): every ll[s], gmu[j] and ge[j] must
stay within its worst-case bound and its statistical bound, at S, d and N around the kernel's branch points, in
every mode (want_grad, ll_total_only, w = NULL / all ones / AlphaDivergence-shaped weights), with the workspace
filled with NaN bytes before each call and sentinels after every output.  Also: probe rows in a million zero rows,
two models sharing one workspace address, C ABI argument errors, and the fused step at its edges."""
import numpy as np
import pytest
import torch

from _glm_fast_ref import CASES, LN2, LN2_F32, Reference, alpha_weights, case_seed, f16_exact, make_case, ratios

pytestmark = pytest.mark.gpu
SENT = -7.25e77            # sentinel after every output array
PAD = 8


def _L():
    from viabel_b200 import _lib
    return _lib


def _dev(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device='cuda')


def _aligned(nbytes, align=1024, offset=0):
    buf = torch.empty(nbytes + 2 * align, dtype=torch.uint8, device='cuda')
    off = (-buf.data_ptr()) % align + offset
    return buf[off:off + nbytes]


class Fast(object):
    """A vb_glm_fast_create handle with its model memory."""

    def __init__(self, X, y, ldx=None):
        L = _L()
        X = np.asarray(X, dtype=np.float64)
        self.N, self.d = X.shape
        ldx = self.d if ldx is None else ldx
        Xp = np.full((self.N, ldx), np.nan)
        Xp[:, :self.d] = X
        self.X, self.y = _dev(Xp), _dev(y)
        self.mem = _aligned(L.lib.vb_glm_fast_model_bytes(self.N, self.d))
        import ctypes
        self.handle = ctypes.c_void_p()
        absmax = ctypes.c_float(0.0)
        self.rc = L.lib.vb_glm_fast_create(ctypes.byref(self.handle), L.ptr(self.X), ldx, L.ptr(self.y), self.N,
                                           self.d, L.LINK_LOGISTIC, L.ptr(self.mem), self.mem.numel(),
                                           ctypes.byref(absmax), L.stream())
        self.absmax = absmax.value

    def ws_bytes(self, S=256):
        return _L().lib.vb_glm_fast_workspace_bytes(self.N, self.d, S)

    def sweep(self, theta, base, w, flags, ws=None, fill=0xFF, debug=None, S=None):
        """One sweep; returns (rc, ll, gmu, ge) as numpy arrays (gmu / ge None without bit 0 of flags).  The
        sentinels after each output must survive; gmu / ge must stay untouched without gradients."""
        L = _L()
        S = theta.shape[0] if S is None else S
        if ws is None:
            ws = _aligned(self.ws_bytes())
        if fill is not None:
            ws.fill_(fill)
        outs = [torch.full((n + PAD,), SENT, dtype=torch.float64, device='cuda') for n in (S, self.d, self.d)]
        th, bs = _dev(theta), (None if base is None else _dev(base))
        wt = None if w is None else _dev(w)
        rc = L.lib.vb_glm_fast_sweep(self.handle, L.ptr(th), L.ptr(bs), L.ptr(wt), S, flags, L.ptr(outs[0]),
                                     L.ptr(outs[1]), L.ptr(outs[2]), L.ptr(ws), ws.numel(), L.ptr(debug), L.stream())
        torch.cuda.synchronize()
        o = [t.cpu().numpy() for t in outs]
        if rc != 0:
            return rc, None, None, None
        assert np.all(o[0][S:] == SENT), 'll written past S'
        assert np.all(np.isfinite(o[0][:S]))
        if flags & 1:
            for a in o[1:]:
                assert np.all(a[self.d:] == SENT), 'gradient written past d'
                assert np.all(np.isfinite(a[:self.d]))
            return rc, o[0][:S], o[1][:self.d], o[2][:self.d]
        assert np.all(o[1] == SENT) and np.all(o[2] == SENT), 'gradient outputs written without want_grad'
        return rc, o[0][:S], None, None

    def __del__(self):
        try:
            _L().lib.vb_glm_fast_destroy(self.handle)
        except Exception:
            pass


def _eq(a, b):
    return a is not None and b is not None and np.array_equal(a, b)


def run_case(N, d, S, general):
    """All modes of one shape; returns {mode: {output: (worst ratio, stat ratio)}}."""
    X, y, theta, base = make_case(N, d, S, case_seed(N, d, S), exact=not general)
    m = Fast(X, y)
    assert m.rc == 0
    ws = _aligned(m.ws_bytes())
    res = {}
    ref = Reference(X, y, theta, base, exact=not general)
    rc, ll, gmu, ge = m.sweep(theta, base, None, 1, ws=ws, fill=0)
    assert rc == 0
    res['main'] = ratios(ref, ll, gmu, ge)
    for _ in range(2):           # NaN-filled workspace, repeated: bitwise the same
        r2 = m.sweep(theta, base, None, 1, ws=ws)
        assert _eq(r2[1], ll) and _eq(r2[2], gmu) and _eq(r2[3], ge), 'repeat / NaN workspace differs'
    r0 = m.sweep(theta, None, None, 0, ws=ws)
    assert r0[0] == 0 and _eq(r0[1], ll), 'want_grad = 0 changes ll'
    rt = m.sweep(theta, base, None, 3, ws=ws)
    assert _eq(rt[2], gmu) and _eq(rt[3], ge), 'll_total_only changes the gradient'
    assert np.all(rt[1] == rt[1][0])
    rt0 = m.sweep(theta, None, None, 2, ws=ws)
    assert _eq(rt0[1], rt[1])
    tot_err = abs(rt[1][0] * S - ref.ll.sum())
    res['total'] = {'ll': (tot_err / ref.total_bound(), 0.0)}
    r1 = m.sweep(theta, base, np.ones(S), 1, ws=ws)
    assert _eq(r1[1], ll) and _eq(r1[2], gmu) and _eq(r1[3], ge), 'all-ones weights differ from w = NULL'
    w = alpha_weights(S, S + d)
    refw = Reference(X, y, theta, base, w=w, exact=not general)
    rw = m.sweep(theta, base, w, 1, ws=ws)
    assert _eq(rw[1], ll), 'weights change ll'
    res['weighted'] = ratios(refw, rw[1], rw[2], rw[3])
    return res


def _check(res, tag):
    for mode, r in res.items():
        for out, (wc, st) in r.items():
            assert wc <= 1.0 and st <= 1.0, (tag, mode, out, wc, st)


def _print(tag, res):
    print('%s: %s' % (tag, ', '.join('%s/%s %.3f/%.3f' % (m, o, w, s) for m, r in res.items()
                                       for o, (w, s) in r.items())))


@pytest.mark.parametrize('N,d,S,general', CASES)
def test_fast_sweep_elementwise(N, d, S, general):
    res = run_case(N, d, S, general)
    _print('pair N=%d d=%d S=%d' % (N, d, S), res)
    _check(res, (N, d, S))


def test_fast_sweep_probe_rows():
    """N = 1 000 003 rows of d = 512 exact zeros except ~40 probe rows at the tile, super-tile, CTA-half and
    persistent-round edges (row 74 * 256 is the first row of pair 0's second round; the last super-tile holds 67 rows,
    so both halves of the one before it are probed) and at columns 0, 255, 256 and d-1.  Zero rows contribute exactly nothing to the gradient,
    so a missing, doubled or misplaced probe is an O(1/40) error; ll is -(N - P) ln 2 (fp32 ln 2 per row, summed
    exactly in the kernel) minus the probe terms."""
    N, d, S = 1000003, 512, 256
    rs = np.random.RandomState(40)
    last = (N - 1) // 256 * 256          # first row of the last super-tile: its 67 rows all lie in the first CTA half
    rows = [0, 1, 127, 128, 255, 256, 74 * 256, 74 * 256 + 128, 2 * 74 * 256, last - 129, last - 128, last - 1, last,
            N - 2, N - 1]
    rows += list(rs.choice(np.arange(257, last - 129), 40 - len(rows), replace=False))
    rows = np.array(sorted(set(int(r) for r in rows)))
    assert rows.min() >= 0 and rows.max() < N
    cols = np.array([0, 1, 127, 128, 255, 256, 383, 384, 510, d - 1])
    Xp = np.zeros((len(rows), d))
    for i in range(len(rows)):
        Xp[i, cols] = rs.randn(len(cols))
        Xp[i, rs.randint(d, size=4)] = rs.randn(4)
    yp = np.where(rs.rand(len(rows)) < 0.5, 1.0, -1.0)
    X = torch.zeros(N, d, dtype=torch.float64, device='cuda')
    y = torch.ones(N, dtype=torch.float64, device='cuda')
    X[torch.as_tensor(rows, device='cuda')] = _dev(Xp)
    y[torch.as_tensor(rows, device='cuda')] = _dev(yp)
    base = f16_exact(rs.randn(S, d))
    theta = 0.3 * rs.randn(d) + 0.2 * base
    import ctypes
    L = _L()
    mem = _aligned(L.lib.vb_glm_fast_model_bytes(N, d))
    h = ctypes.c_void_p()
    assert L.lib.vb_glm_fast_create(ctypes.byref(h), L.ptr(X), d, L.ptr(y), N, d, 0, L.ptr(mem), mem.numel(), None,
                                    L.stream()) == 0
    del X
    m = Fast.__new__(Fast)
    m.N, m.d, m.handle, m.mem = N, d, h, mem
    # the fp8 scales that the sparse data selects (its rms counts the zero rows)
    v = (Xp * yp[:, None]).astype(np.float32).astype(np.float64)
    r = int(np.rint(np.log2(np.sqrt(np.sum(v * v) / (float(N) * d)))))
    sexp = int(np.frexp(np.float32(np.max(np.abs(v))))[1])
    ax, bx = min(2 - r, 26 - sexp), max(8 + r, sexp - 15)
    print('probe rows: %d, fp8 scales ax = %d, bx = %d' % (len(rows), ax, bx))
    ref = Reference(Xp, yp, theta, base, ax=ax)
    rc, ll, gmu, ge = m.sweep(theta, base, None, 1)
    assert rc == 0
    zero_rows = N - len(rows)
    ll_ref = ref.ll - zero_rows * LN2_F32
    wll = ref.bounds()['ll'][0] + 1e-9 * zero_rows
    assert np.all(np.abs(ll - ll_ref) <= wll), np.max(np.abs(ll - ll_ref) / wll)
    assert abs(np.mean(ll) + zero_rows * LN2 - np.mean(ref.ll)) < zero_rows * 2.0 ** -24 + np.max(wll)
    rr = ratios(ref, None, gmu, ge)
    print('probe rows ratios: %s' % rr)
    for o, (wc, st) in rr.items():
        assert wc <= 1.0 and st <= 1.0, (o, wc, st)
    # one probe row less is far outside the budget (what the test would see if a probe were lost)
    _, dg, de = ref.row(len(rows) - 1)
    T = ref.bounds()['gmu'][1]
    assert np.max(np.abs(dg)[T > 0] / T[T > 0]) > 10


def test_fast_sweep_total_only_separated():
    """ll_total_only with S < 64 sums (256 - S) ln 2 of padded columns into the fp32 chunk sums and subtracts them
    afterwards; on well-separated data (per-row softplus << ln 2) the mean must stay within 2^-19 per valid row."""
    N, d = 20000, 64
    rs = np.random.RandomState(3)
    X = rs.randn(N, d)
    beta = rs.randn(d) * 3.0
    y = np.sign(X @ beta)
    m = Fast(X, y)
    for S in (1, 5, 31, 63, 64, 65, 200):
        base = f16_exact(rs.randn(S, d))
        theta = beta + 0.01 * base
        ref = Reference(X, y, theta, base)
        _, ll, _, _ = m.sweep(theta, None, None, 2)
        err = abs(ll[0] - ref.ll.mean())
        print('total-only separated S=%d: mean softplus per row %.2e, error of the mean %.3e = %.3f x 2^-19 N'
              % (S, -ref.ll.mean() / N, err, err / (2.0 ** -19 * N)))
        assert err <= 2.0 ** -19 * N + float(np.mean(ref.bounds()['ll'][0]))


def test_fast_sweep_workspace_reuse():
    """Two models with the same d_pad (d = 300) and different N share one workspace address: every output must equal
    the same model's sweep on a fresh buffer, bitwise.  The cached tensor maps must follow the Theta e5m2 copies,
    whose offset depends on N.  (S = 128, so that a build whose row sums of R depend on the atomics' order is still
    reproducible here; the shared buffer is not refilled, as when the caching allocator hands a block back.)"""
    d, S = 300, 128
    cases = []
    for N in (1000, 20000):
        X, y, theta, base = make_case(N, d, S, case_seed(N, d, S))
        cases.append((Fast(X, y), theta, base))
    own, keep = [], []
    for m, theta, base in cases:
        ws = _aligned(m.ws_bytes())
        keep.append(ws)
        own.append(m.sweep(theta, base, None, 1, ws=ws)[1:])
        own.append(m.sweep(theta, base, None, 3, ws=ws)[1:])
    refs = [Reference(m.X.cpu().numpy(), m.y.cpu().numpy(), theta, base) for m, theta, base in cases]
    shared = _aligned(max(m.ws_bytes() for m, _, _ in cases))
    shared.zero_()
    bad = []
    for rep in range(2):
        for i, (m, theta, base) in enumerate(cases):
            for k, flags in enumerate((1, 3)):
                got = m.sweep(theta, base, None, flags, ws=shared, fill=None)[1:]
                r = ratios(refs[i], None if flags & 2 else got[0], got[1], got[2])
                for name, a, b in zip(('ll', 'gmu', 'ge'), got, own[2 * i + k]):
                    if not np.array_equal(a, b):
                        bad.append(('N=%d' % m.N, 'flags=%d' % flags, name, 'max rel diff %.3e' % np.max(
                            np.abs(a - b) / (np.abs(b) + 1e-300)), 'err/bound %.3g' % r.get(name, (0.0,))[0]))
    assert not bad, bad


def test_fused_step_workspace_reuse():
    """The same through two FusedSteps whose models share nothing but the workspace address."""
    import viabel_b200 as vb
    from viabel_b200.engine import FusedStep
    d, S = 300, 128
    res = {}
    for shared_ws in (False, True):
        shared = None
        out, keep = [], []                    # every model and engine stays alive: no address is reused by accident
        for N in (1000, 20000, 1000, 20000):
            X, y, theta, base = make_case(N, d, S, case_seed(N, d, S))
            model = vb.LogisticRegression(X, y, prior_scale=10.0).enable_fast_path()
            if shared_ws:
                if shared is None:
                    shared = _aligned(max(_L().lib.vb_glm_fast_workspace_bytes(n, d, S) for n in (1000, 20000)))
                h, mem, _ = model._fast
                model._fast = (h, mem, shared)
            eng = FusedStep(vb.ExclusiveKL(vb.MFGaussian(d), model, S), None, inject_base=True)
            mu, ls = np.zeros(d), -1.0 * np.ones(d)
            eng.set_param(np.concatenate([mu, ls]))
            eng.base.copy_(_dev(base))
            eng.run(1, use_graph=False)
            torch.cuda.synchronize()
            out.append(eng.out.cpu().numpy().copy())
            assert max(_fused_ratios(eng, X, y, mu, ls, base)) <= 1.0, (N, shared_ws, _fused_ratios(eng, X, y, mu, ls, base))
            keep.append((model, eng))
        res[shared_ws] = out
    for k, (a, b) in enumerate(zip(res[True], res[False])):
        assert np.array_equal(a, b), (k, 'max rel diff %.3e' % np.max(np.abs(a - b) / (np.abs(b) + 1e-300)))


def _fused_ratios(eng, X, y, mu, ls, base, ps2=100.0):
    """Value and gradient of one fused ExclusiveKL step (prior N(0, ps2)) against the reference sweep: largest
    err / worst-case bound of the value, the mu half and the log-sd half of the gradient."""
    S, d = base.shape
    sig = np.exp(ls)
    theta = mu + sig * base
    value, grad = float(eng.value[0]), eng.grad.cpu().numpy()
    ref = Reference(X, y, theta, base)
    b = ref.bounds()
    logprior = -0.5 * np.sum(theta ** 2, axis=1) / ps2 - 0.5 * d * np.log(2 * np.pi * ps2)
    H = 0.5 * d * (1.0 + np.log(2 * np.pi)) + np.sum(ls)
    v0 = -(np.mean(ref.ll + logprior) + H)
    g_mu = -(ref.gmu - theta.sum(axis=0) / ps2) / S
    g_ls = -sig * (ref.ge - np.sum(theta * base, axis=0) / ps2) / S - 1.0
    tiny = 1e-12 * (1.0 + np.abs(np.concatenate([g_mu, g_ls])))
    e_v = abs(value - v0) / (ref.total_bound() / S + 1e-12 * abs(v0))
    e_mu = np.max(np.abs(grad[:d] - g_mu) / (b['gmu'][0] / S + tiny[:d]))
    e_ls = np.max(np.abs(grad[d:] - g_ls) / (sig * b['ge'][0] / S + tiny[d:]))
    return e_v, e_mu, e_ls


def test_fast_cabi_errors():
    import ctypes
    L = _L()
    N, d, S = 300, 40, 8
    X, y, theta, base = make_case(N, d, S, 1)
    m = Fast(X, y)
    assert m.rc == 0
    ws = _aligned(m.ws_bytes())
    out = [_dev(np.zeros(n)) for n in (300, d, d)]
    th, bs = _dev(theta), _dev(base)

    def call(S_, flags=1, b=bs, w=ws, nbytes=None, t=th):
        return L.lib.vb_glm_fast_sweep(m.handle, L.ptr(t), L.ptr(b), None, S_, flags, L.ptr(out[0]), L.ptr(out[1]),
                                       L.ptr(out[2]), L.ptr(w), w.numel() if nbytes is None else nbytes, None,
                                       L.stream())
    th300 = _dev(np.zeros((300, d)))
    assert call(0) == L.VB_ERR_INVALID_ARG
    assert call(257, t=th300) == L.VB_ERR_UNSUPPORTED
    assert call(S, flags=1, b=None) == L.VB_ERR_INVALID_ARG
    assert call(S, nbytes=m.ws_bytes() - 1) == L.VB_ERR_WORKSPACE
    mis = _aligned(m.ws_bytes(), offset=256)
    assert call(S, w=mis) == L.VB_ERR_INVALID_ARG
    assert call(S) == 0
    # create: d > 2048, ldx < d, a NaN / +-inf entry of X (rejected, never swept), misaligned model memory
    for Xb, code in ((np.zeros((4, 2049)), L.VB_ERR_UNSUPPORTED),):
        assert Fast(Xb, np.ones(4)).rc == code
    for bad in (np.nan, np.inf, -np.inf):
        Xb = X.copy()
        Xb[123, 7] = bad
        assert Fast(Xb, y).rc == L.VB_ERR_UNSUPPORTED, bad
    Xt, yt = _dev(X), _dev(y)
    h = ctypes.c_void_p()
    mem = _aligned(L.lib.vb_glm_fast_model_bytes(N, d))
    assert L.lib.vb_glm_fast_create(ctypes.byref(h), L.ptr(Xt), d - 1, L.ptr(yt), N, d, 0, L.ptr(mem), mem.numel(),
                                    None, L.stream()) == L.VB_ERR_INVALID_ARG
    mis = _aligned(L.lib.vb_glm_fast_model_bytes(N, d), offset=512)
    assert L.lib.vb_glm_fast_create(ctypes.byref(h), L.ptr(Xt), d, L.ptr(yt), N, d, 0, L.ptr(mis), mis.numel(),
                                    None, L.stream()) == L.VB_ERR_INVALID_ARG
    # ldx > d (NaN in the padding columns) gives the contiguous result bitwise
    wide = Fast(X, y, ldx=d + 13)
    assert wide.rc == 0
    a = m.sweep(theta, base, None, 1)
    b = wide.sweep(theta, base, None, 1)
    assert all(np.array_equal(u, v) for u, v in zip(a[1:], b[1:]))


@pytest.mark.parametrize('N,d,S', [(129, 257, 1), (4099, 1, 65), (33000, 2048, 255)])
def test_fused_step_fast_elementwise(N, d, S):
    """mf_pre_kernel packs Theta, E and the e5m2 copies itself: one fused step's value and gradient element by element
    against the reference sweep, through the ExclusiveKL map (prior N(0, 10^2))."""
    import viabel_b200 as vb
    from viabel_b200.engine import FusedStep
    X, y, _, base = make_case(N, d, S, case_seed(N, d, S))
    rs = np.random.RandomState(N + d)
    mu, ls = rs.randn(d) / np.sqrt(d), -1.0 + 0.1 * rs.randn(d)
    model = vb.LogisticRegression(X, y, prior_scale=10.0).enable_fast_path()
    eng = FusedStep(vb.ExclusiveKL(vb.MFGaussian(d), model, S), None, inject_base=True)
    eng.set_param(np.concatenate([mu, ls]))
    eng.base.copy_(_dev(base))
    eng.run(1, use_graph=False)
    torch.cuda.synchronize()
    e_v, e_mu, e_ls = _fused_ratios(eng, X, y, mu, ls, base)
    print('fused N=%d d=%d S=%d: value %.3f, grad mu %.3f, grad log sd %.3f of the worst-case bound' % (N, d, S, e_v, e_mu, e_ls))
    assert e_v <= 1 and e_mu <= 1 and e_ls <= 1
