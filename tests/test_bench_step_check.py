"""The oracle check of bench.py's step (tests/_step_check.py) on a picture small enough for the CPU: device outputs made by the oracle pass,
and a single wrong value of each kind fails, naming its block.  This is what lets test_gpu_bench_step.py fail when the device is wrong."""
import numpy as np
import pytest

import bench
import _step_check as SC
from vvenc_b200.candidates import pyramid_lists

W, H = 256, 184          # 184 = 2 * 64 + 56: parentless 32x32, 16x16 and 8x8 roots below the last 64x64 row


def _noisy(ref, seed, max_amplitude):
    """ref plus uniform noise whose amplitude grows from 0 at the left edge to max_amplitude at the right.  bench.py's pictures quantise to
    all-zero levels at QP 32 (their residual at the best vector is the +-6 noise of the reference); against this one the blocks give zero and
    non-zero levels, many last positions and both RDOQ pre-check decisions."""
    rs = np.random.RandomState(seed)
    amp = np.clip(np.arange(ref.shape[1]) - bench.MARGIN, 0, W) * (max_amplitude / W)
    noise = np.round(rs.uniform(-1.0, 1.0, size=ref.shape) * amp[None, :]).astype(np.int32)
    return np.ascontiguousarray(np.clip(ref.astype(np.int32) + noise, 0, 1023).astype(np.int16))


@pytest.fixture(scope='module')
def levels():
    org, ref, S = bench.synth_picture_pair(99, W, H)
    ref = _noisy(ref, 7, 200)
    pat = bench.refine_pattern()
    out = []
    for n, (xs, ys) in zip(bench.SIZES, pyramid_lists(bench.SIZES[0], len(bench.SIZES), W, H)):
        exp = SC.expected_level(org, ref, S, bench.MARGIN, n, xs, ys, bench.LAMBDA, bench.SEARCH_RANGE, pat, bench.BITDEPTH, bench.QP)
        out.append((n, xs, ys, exp))
    return out


def _copy(exp):
    return {k: v.copy() for k, v in exp.items()}


def test_picture_has_partial_root_rows(levels):
    counts = {n: len(xs) for n, xs, _, _ in levels}
    assert counts == {64: 4 * 2, 32: 4 * 8 + 8, 16: 4 * 40 + 16, 8: 4 * 176 + 32}
    for n, xs, ys, exp in levels:
        # the check sees vectors off the centre, zero and non-zero levels and both RDOQ decisions
        assert (exp['dx'] != 0).any() and (exp['abs_sum'] > 0).any() and (exp['abs_sum'] == 0).any(), n
        assert set(np.unique(exp['need_rdoq'])) == {0, 1}, n


def test_oracle_outputs_pass(levels):
    K = len(bench.refine_pattern())
    for n, xs, ys, exp in levels:
        assert SC.compare_level(n, xs, ys, exp, _copy(exp), K) == [], n


def _fails_naming(n, xs, ys, exp, got, i, what, **kw):
    msgs = SC.compare_level(n, xs, ys, exp, got, len(bench.refine_pattern()), **kw)
    assert len(msgs) == 1 and what in msgs[0], msgs
    assert 'block %d at (%d, %d)' % (i, xs[i], ys[i]) in msgs[0], msgs
    return msgs[0]


def test_one_wrong_value_of_each_kind_fails(levels):
    by_size = {n: (xs, ys, exp) for n, xs, ys, exp in levels}
    K = len(bench.refine_pattern())
    # one dy (a 16x16 block in the parentless row)
    xs, ys, exp = by_size[16]
    i = len(xs) - 3
    got = _copy(exp); got['dy'][i] += 1
    _fails_naming(16, xs, ys, exp, got, i, 'search')
    # one ring cost in the last group of the 8x8 level
    xs, ys, exp = by_size[8]
    i = len(xs) - 1
    got = _copy(exp); got['ring'][i, K - 2] ^= 4
    m = _fails_naming(8, xs, ys, exp, got, i, 'ring', grids={'ring': 3})
    g = i // SC.ring_blocks_per_group(8, K)
    assert 'ring group %d (CTA %d, pass %d)' % (g, g % 3, g // 3) in m and 'ring[%d]' % (K - 2) in m, m
    # one level of a 32x32 TU
    xs, ys, exp = by_size[32]
    i = int(np.flatnonzero(exp['abs_sum'] > 0)[-1])
    got = _copy(exp); got['q'][i, 3, 5] += 1
    m = _fails_naming(32, xs, ys, exp, got, i, 'levels')
    assert 'tc2 tile %d' % (i // SC.tc2_tus_per_tile(32)) in m and 'q[%d]' % (3 * 32 + 5) in m, m
    # one lastPos of a 64x64 TU
    xs, ys, exp = by_size[64]
    i = 5
    got = _copy(exp); got['last_pos'][i] -= 1
    _fails_naming(64, xs, ys, exp, got, i, 'lastPos')
    # one needRdoq flag of an 8x8 TU
    xs, ys, exp = by_size[8]
    i = 301
    got = _copy(exp); got['need_rdoq'][i] ^= 1
    _fails_naming(8, xs, ys, exp, got, i, 'needRdoq')


def test_sampled_blocks_are_named_by_their_level_index(levels):
    n, xs, ys, exp = levels[0]
    idx = np.array([3, 40, 41, len(xs) - 1])
    sub = {k: v[idx] for k, v in exp.items()}
    got = _copy(sub); got['sad'][2] += 1
    msgs = SC.compare_level(n, xs[idx], ys[idx], sub, got, len(bench.refine_pattern()), index=idx)
    assert len(msgs) == 1 and 'sad: 1 of 4 blocks differ; block 41 at (%d, %d)' % (xs[41], ys[41]) in msgs[0], msgs
