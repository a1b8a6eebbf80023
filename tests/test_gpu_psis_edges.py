"""PSIS on the device against the oracle on inputs built to reach each branch of csrc/psis.cu (tests/_psis_ref.py):
the sampled run must take the path the host mirror predicts (status, and the exact candidate count on status 0), and
after the exact-mode fallback every output must match oracle.viabel_oracle.psislw_1d -- maximum and shifted cutoff
bit-equal, tail set and rank order bit-exact, k-hat, outputs and moments to 1e-10 -- in the two-pass, exact,
moments-only and unaligned forms, draw-sharded (with and without an output array) and past 2^31 draws."""
import numpy as np
import pytest
import torch

import _psis_ref as P
from _problems import psis_case

pytestmark = pytest.mark.gpu
TOL = 1e-10
R_KHAT, R_SIGMA, R_N2, R_CUTOFF, R_LSE, R_MAX, R_STATUS, R_SUMV, R_SUMEXP2V, R_M, R_NCAND, R_SMOOTHED = range(12)


@pytest.fixture(scope='module')
def psis():
    from viabel_b200 import _psis
    return _psis


_refs = {}


def _oracle(key, lw, reff):
    if key not in _refs:
        _refs[key] = P.oracle(lw, reff)
    return _refs[key]


def _same(a, b):
    """Bit-equal, or both NaN."""
    a, b = np.float64(a), np.float64(b)
    return a.tobytes() == b.tobytes() or (np.isnan(a) and np.isnan(b))


def _close(got, ref, what):
    if np.isfinite(ref):
        assert abs(got - ref) <= TOL * abs(ref) + 1e-300, (what, got, ref)
    else:
        assert _same(got, ref) or got == ref, (what, got, ref)


def _value_order(ti, tr, n2):
    """Tail indices in (value, index) order from the index-ordered list and its value ranks."""
    ti, tr = ti[:n2].cpu().numpy(), tr[:n2].cpu().numpy()
    assert np.all(ti[1:] > ti[:-1])
    order = np.empty(n2, dtype=np.int64)
    order[tr] = ti
    return order


def _check(res, out, ref, tail=None, what=''):
    """One finished (status 0) device run against the oracle."""
    assert res[R_STATUS] == 0, what
    assert _same(res[R_MAX], ref['max']) and _same(res[R_CUTOFF], ref['xcut']), (what, res[R_MAX], res[R_CUTOFF],
                                                                                 ref['max'], ref['xcut'])
    assert int(res[R_N2]) == ref['n2'] and int(res[R_M]) == ref['M'], (what, res[R_N2], ref['n2'])
    if tail is not None:
        assert np.array_equal(tail, ref['tail']), what
    if np.isfinite(ref['k']):
        _close(res[R_KHAT], ref['k'], (what, 'k'))
    else:
        assert res[R_KHAT] == ref['k'], (what, res[R_KHAT], ref['k'])
    _close(res[R_LSE], ref['lse'], (what, 'lse'))
    _close(res[R_SUMV], ref['sumv'], (what, 'sumv'))
    _close(res[R_SUMEXP2V], ref['sumexp2v'], (what, 'sumexp2v'))
    if out is not None:
        np.testing.assert_allclose(out, ref['out'], rtol=TOL, atol=TOL, err_msg=str(what))


def _fallback(psis, t, out, reff, want_tail, exact=False):
    """psislw_device, rerun in exact mode on status 1 (what the public psislw does)."""
    _, res, ti, tr = psis.psislw_device(t, out, reff, want_tail, exact)
    res = res.cpu().numpy()
    if res[R_STATUS] == 1:
        _, res, ti, tr = psis.psislw_device(t, out, reff, want_tail, True)
        res = res.cpu().numpy()
    return res, ti, tr


def _run_matrix(psis, key, lw, reff, variants=True):
    """Sampled run against the mirror, then every form of the finished run against the oracle."""
    pred = P.mirror(lw, reff)
    ref = _oracle(key, lw, reff)
    assert ref['M'] == pred['M']
    t = torch.as_tensor(lw, device='cuda')
    out = torch.empty_like(t)
    _, res, _, _ = psis.psislw_device(t, out, reff, False, False)
    res = res.cpu().numpy()
    assert res[R_STATUS] == pred['status'], (key, res[R_STATUS], pred['status'], sorted(pred['labels']))
    if pred['status'] == 0:
        assert res[R_NCAND] == pred['C'] and res[R_M] == pred['M'], (key, res[R_NCAND], pred['C'])
        _check(res, out.cpu().numpy(), ref, what=(key, 'sampled'))
    # the public fallback (sampled, then exact on status 1), with the tail
    res2, ti, tr = psis._psis_column(t, out, reff, True)
    _check(res2, out.cpu().numpy(), ref, _value_order(ti, tr, int(res2[R_N2])), (key, 'psislw'))
    # exact mode forced
    _, res3, ti, tr = psis.psislw_device(t, out, reff, True, True)
    res3 = res3.cpu().numpy()
    _check(res3, out.cpu().numpy(), ref, _value_order(ti, tr, int(res3[R_N2])), (key, 'exact'))
    # k-hat and moments only (one pass over the draws)
    res4, _, _ = _fallback(psis, t, None, reff, False)
    for slot in (R_KHAT, R_SIGMA, R_N2, R_CUTOFF, R_LSE, R_MAX, R_M, R_SMOOTHED):
        a, b = res4[slot], res2[slot]
        assert _same(a, b) or abs(a - b) <= 1e-12 * abs(b), (key, 'moments-only', slot, a, b)
    _close(res4[R_SUMV], ref['sumv'], (key, 'moments-only sumv'))
    _close(res4[R_SUMEXP2V], ref['sumexp2v'], (key, 'moments-only sumexp2v'))
    if not variants:
        return
    # 8-byte aligned only: the scalar loops of pass A and pass B
    n = lw.size
    buf = torch.zeros(n + 3, device='cuda', dtype=torch.float64)
    obuf = torch.zeros(n + 3, device='cuda', dtype=torch.float64)
    for off in (1, 2, 3):
        buf[off:off + n] = t
        res5, ti, tr = _fallback(psis, buf[off:off + n], obuf[off:off + n], reff, True)
        _check(res5, obuf[off:off + n].cpu().numpy(), ref, _value_order(ti, tr, int(res5[R_N2])), (key, 'offset', off))


@pytest.mark.parametrize('name', list(P.NAMED))
def test_named_cases(psis, name):
    lw = P.named_case(name)
    _run_matrix(psis, name, lw, 1.0)


@pytest.mark.parametrize('name,reff', P.reff_cases())
def test_reff_cases(psis, name, reff):
    """Tail lengths at the kernels' fixed sizes (2048-value GPD chunks, 256-wide loops, 8-term log products,
    n2 <= 4 against 5) and plain values of Reff, which set M, R, the capacity and every tail buffer."""
    _run_matrix(psis, name, psis_case('big_1e6'), reff, variants=name in ('n2_2049', 'reff_0.01'))


@pytest.mark.parametrize('kind', P.SMALL_KINDS)
def test_small_n(psis, kind):
    for n in P.SMALL_N:
        _run_matrix(psis, (kind, n), P.small_case(kind, n), 1.0, variants=n in (2, 3, 17, 64))


# ---- draw-sharded: shards driven in one process, the exchange by hand ------------------------------------------------
def _sharded(psis, x, cuts, reff=1.0):
    """The loop of psislw_sharded: local(sampled), global, apply; every shard reruns exact when any status is 1.
    Each shard also applies without an output array (pass B moments only), which must give the same moments to
    1e-12 (its exp(2 v) is a different polynomial form).
    Returns the outputs, the replicated result, the summed moments and the sampled local status of each shard."""
    n, world = x.numel(), len(cuts) - 1
    shards = [psis.PsisShard(x[cuts[r]:cuts[r + 1]], cuts[r], n, reff, world, r) for r in range(world)]
    local_status = None
    for exact in (False, True):
        recs = torch.cat([s.local(exact) for s in shards])
        if local_status is None:
            heads = recs.view(world, -1)[:, 3].cpu().numpy()
            local_status = [int(-h) if h < 0 else 0 for h in heads]
        outs, res, mom = [], None, np.zeros(2)
        for s in shards:
            s.global_(recs)
            o = torch.empty_like(s.lw)
            rr = s.apply(o).cpu().numpy()
            rm = s.apply(None).cpu().numpy()
            for slot in range(R_SUMV, R_SUMEXP2V + 1):
                a, b = rm[slot], rr[slot]
                assert _same(a, b) or abs(a - b) <= 1e-12 * abs(b), ('apply(None)', slot, a, b)
            mom += rr[R_SUMV:R_SUMEXP2V + 1]
            outs.append(o)
            if res is None:
                res = rr
            else:
                assert np.array_equal(rr[:R_SUMV], res[:R_SUMV], equal_nan=True)
        if res[R_STATUS] == 0:
            return outs, res, mom, local_status
        assert res[R_STATUS] == 1
    raise AssertionError('sharded PSIS did not finish in exact mode')


def _check_sharded(psis, lw, cuts, reff=1.0):
    x = torch.as_tensor(lw, device='cuda')
    o1 = torch.empty_like(x)
    r1, _, _ = _psis_column_res(psis, x, o1, reff)
    outs, res, mom, local_status = _sharded(psis, x, cuts, reff)
    for slot in (R_KHAT, R_SIGMA, R_N2, R_CUTOFF):
        assert _same(res[slot], r1[slot]), (cuts, slot, res[slot], r1[slot])
    np.testing.assert_allclose(torch.cat(outs).cpu().numpy(), o1.cpu().numpy(), rtol=0, atol=1e-11)
    np.testing.assert_allclose(mom, r1[R_SUMV:R_SUMEXP2V + 1], rtol=1e-11)
    return local_status


def _psis_column_res(psis, x, out, reff):
    return psis._psis_column(x, out, reff, False)


@pytest.mark.parametrize('name', [nm for nm in P.NAMED if nm != 'sorted_shard_mix'])
def test_sharded_named(psis, name):
    lw = P.named_case(name)
    n, M = lw.size, P.plan(lw.size)['M']
    _check_sharded(psis, lw, [0, n // 2, n])
    _check_sharded(psis, lw, [0, M // 2, n // 3, n])          # a shard with fewer than M+1 draws: exports all of them


def test_sharded_sorted_shard(psis):
    """One shard sorted, one not: the sorted shard's sampled threshold fails (as the mirror predicts), the other's
    passes, and the rerun in exact mode gives the single-GPU result."""
    lw = P.named_case('sorted_shard_mix')
    n = lw.size
    cuts = [0, n // 2, n]
    pred = [P.mirror(lw[cuts[r]:cuts[r + 1]], 1.0, n, 2)['status'] for r in range(2)]
    assert pred == [0, 1]
    assert _check_sharded(psis, lw, cuts) == pred


# ---- more than 2^31 draws -----------------------------------------------------------------------------------------
def test_more_than_2pow31_draws(psis):
    n = P.BIG_N
    need = 16 * n + (4 << 30)
    free = torch.cuda.mem_get_info()[0]
    if free < need:
        pytest.skip('needs %.1f GB of free device memory, %.1f GB free' % (need / 1e9, free / 1e9))
    pos, vals, body = P.big_piece()
    pred = P.mirror_big()
    sur, reff_s, _ = P.big_surrogate()
    ref = P.oracle(sur, reff_s)
    assert ref['M'] == pred['M'] and np.all(ref['tail'] < pos.size)
    tail = pos[ref['tail']]
    assert tail.max() >= 2 ** 31
    nb = n - pos.size
    v_body = body - ref['max']
    sumv = ref['sumv'] - (sur.size - pos.size) * v_body + nb * v_body
    sume = ref['sumexp2v']                   # exp(2 (body - max)) underflows
    full = dict(ref, sumv=sumv, sumexp2v=sume, tail=tail)
    pos_t, vals_t = torch.as_tensor(pos, device='cuda'), torch.as_tensor(vals, device='cuda')
    lw = torch.full((n,), body, dtype=torch.float64, device='cuda')
    lw[pos_t] = vals_t
    out = torch.empty_like(lw)

    def check_out(res, out, what):
        got = out[pos_t].cpu().numpy()
        np.testing.assert_allclose(got, ref['out'][:pos.size], rtol=TOL, atol=TOL, err_msg=what)
        out[pos_t] = (body - res[R_MAX]) - res[R_LSE]
        assert bool((out == (body - res[R_MAX]) - res[R_LSE]).all()), what

    for exact in (False, True):
        _, res, ti, tr = psis.psislw_device(lw, out, 1.0, True, exact)
        res = res.cpu().numpy()
        if not exact:
            assert res[R_STATUS] == 0 and res[R_NCAND] == pred['C'], (res[R_STATUS], res[R_NCAND], pred['C'])
        _check(res, None, full, _value_order(ti, tr, int(res[R_N2])), ('2^31', exact))
        check_out(res, out, ('2^31', exact))
    single = res
    cut = 2 ** 31 - 5
    outs, res, mom, _ = _sharded(psis, lw, [0, cut, n])
    for slot in (R_KHAT, R_SIGMA, R_N2, R_CUTOFF):
        assert _same(res[slot], single[slot]), slot
    np.testing.assert_allclose(mom, single[R_SUMV:R_SUMEXP2V + 1], rtol=1e-11)
    out[:cut] = outs[0]
    out[cut:] = outs[1]
    del outs
    check_out(res, out, ('2^31', 'sharded'))
