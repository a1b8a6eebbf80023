"""CPU checks of the PSIS host mirror (tests/_psis_ref.py): its plan equals the oracle's tail length and the library's
tail capacity, every named edge case reaches the branches of psis.cu it was built for, and together they reach all of
them.  The GPU side (tests/test_gpu_psis_edges.py) then ties each device run to its predicted branch through the
candidate count."""
import math

import numpy as np
import pytest

import _psis_ref as P
from _problems import psis_case
from oracle import viabel_oracle as vo


def _tail_capacity():
    try:
        from viabel_b200 import _lib
    except (ImportError, OSError):
        return None
    return _lib.lib.vb_psis_tail_capacity


def _plans():
    out = [(n, 1.0) for n in P.SMALL_N]
    out += [(P.named_case(name).size, 1.0) for name in P.NAMED]
    out += [(1000000, reff) for _, reff in P.reff_cases()]
    out += [(P.BIG_N, 1.0)]
    return out


def test_plan_matches_oracle_and_library():
    cap = _tail_capacity()
    for n, reff in _plans():
        p = P.plan(n, reff)
        assert p['M'] == vo.psis_tail_len(n, reff), (n, reff)
        if cap is not None:
            assert cap(n, reff) == p['M'] + 1, (n, reff)
    # the Reff solver hits every tail length it is asked for
    for (name, reff), M in zip(P.reff_cases(), P.REFF_TAILS):
        assert name == 'n2_%d' % M and vo.psis_tail_len(1000000, reff) == M


@pytest.mark.parametrize('name', list(P.NAMED))
def test_named_case_branch(name):
    labels = P.mirror(P.named_case(name))['labels']
    assert labels == P.NAMED[name][1], (name, sorted(labels))


def test_branch_coverage():
    """The union of the branches reached by the named, Reff, small-n and 2^31-draw cases is every branch."""
    seen = set()
    for name in P.NAMED:
        seen |= P.mirror(P.named_case(name))['labels']
    big = psis_case('big_1e6')
    for _, reff in P.reff_cases():
        seen |= P.mirror(big, reff)['labels']
    for kind in P.SMALL_KINDS:
        for n in P.SMALL_N:
            seen |= P.mirror(P.small_case(kind, n))['labels']
    seen |= P.mirror_big()['labels']
    assert seen == set(P.BRANCHES), sorted(set(P.BRANCHES) - seen)


def test_mirror_big_case():
    """More than 2^31 draws: the sampled run resolves with the piece's values alone (no overflow into the body)."""
    r = P.mirror_big()
    assert r['status'] == 0 and 'sample16' in r['labels'] and r["t0"] > P.big_piece()[2]
    assert r['M'] == vo.psis_tail_len(P.BIG_N)
    sur, reff, _ = P.big_surrogate()
    assert vo.psis_tail_len(sur.size, reff) == r['M']


def _off_by_one_changes(x, M):
    """Cutting at rank M or M+2 instead of M+1 changes the shifted cutoff or the tail set, unless the clamped shifted
    value at rank M+1 is tied with a neighbour (None)."""
    with np.errstate(all='ignore'):
        v = x - np.max(x)
    s = np.maximum(np.sort(v)[::-1], math.log(np.finfo(float).tiny))      # cutoffs as clamped by _psis.py:170-173
    if not (s[M - 1] != s[M] and (M + 1 >= s.size or s[M] != s[M + 1])):
        return None

    def cut(rank):
        return s[rank], frozenset(np.flatnonzero(v > s[rank]).tolist())
    ref = cut(M)
    return all(cut(r) != ref for r in (M - 1, M + 1) if r < s.size)


def test_comparisons_discriminate():
    checked = 0
    cases = [P.named_case(name) for name in P.NAMED if P.named_case(name).size <= 2000000]
    cases += [P.small_case('distinct', n) for n in P.SMALL_N if n >= 4]
    for x in cases:
        ok = _off_by_one_changes(x, P.plan(x.size)['M'])
        if ok is None:
            continue
        assert ok
        checked += 1
    big = psis_case('big_1e6')
    for _, reff in P.reff_cases():
        assert _off_by_one_changes(big, P.plan(big.size, reff)['M'])
    assert checked >= 20


def test_oracle_wrapper():
    """The wrapper's lse and cutoff are the oracle's: out + lse normalises, the tail is {x - max > xcut}."""
    x = P.named_case('ulp_above_cutoff')
    r = P.oracle(x)
    assert abs(np.log(np.exp(r['out'] + r['lse']).sum()) - r['lse']) < 1e-12
    assert set(r['tail'].tolist()) == set(np.flatnonzero(x - r['max'] > r['xcut']).tolist())
    assert r['n2'] == r['M'] - 200            # the draws one ulp above the cutoff are not tail
