"""CPU-only: BASELINE.json configs[0] (and a sample of configs[1], last test) -- 416x240 8-bit, QP 37, "plumbing + bit-exact cost check" -- as a parity case: on a whole synthetic frame of that shape
the oracle and the unmodified reference (AVX2 kernels through oracle/_ref) must agree on every number of the path: full-search vectors and costs for every 8x8
and 16x16 block, the SATD refinement costs around them, the quantised levels / sums / last positions of every residual TU (both slice types), and the MCTF
motion field of the frame pair (unit 8, as vvencCfg.cpp:1495 selects below 720 lines)."""
import ctypes
import os
import sys

import numpy as np
import pytest

from _libs import answered, have_ref_results, oracle, refshim, refshim_reset, P, PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.skipif(not have_ref_results('test_baseline_configs_cpu'), reason='neither oracle/_ref nor a recording of its calls')


@pytest.fixture(autouse=True)
def _fresh_refshim_replay():
    refshim_reset()

W, H, M, BD, QP, RANGE, LAM = 416, 240, 48, 8, 37, 8, 38.0


@pytest.fixture(scope='module')
def frame_pair():
    sys.path.insert(0, ROOT)
    import bench
    org, ref, S = bench.synth_picture_pair(416240, W, H, M)          # natural-like content with a global pan, 10 bit
    rs = np.random.RandomState(37)
    cells = (rs.randint(-60, 61, size=((ref.shape[0] + 3) // 4, (ref.shape[1] + 3) // 4)) * (rs.rand((ref.shape[0] + 3) // 4, (ref.shape[1] + 3) // 4) < 0.3))
    bump = np.kron(cells, np.ones((4, 4), dtype=np.int64))[:ref.shape[0], :ref.shape[1]]                    # 4x4 brightness changes a QP 37 quantiser does not erase
    noisy = np.clip((ref >> 2).astype(np.int64) + bump, 0, 255).astype(np.int16)
    return np.ascontiguousarray(org >> 2), np.ascontiguousarray(noisy), S


def test_whole_frame_search_refinement_and_tu_costs(frame_pair):
    sys.path.insert(0, ROOT)
    import bench
    org, ref, S = frame_pair
    assert int(org.max()) <= 255 and int(ref.max()) <= 255
    O = oracle(); R = refshim(); R.refshim_set_simd(b'AVX2')
    base = M * S + M
    pat = bench.refine_pattern(); K = len(pat)
    for n in (8, 16):
        xs, ys = np.meshgrid(np.arange(0, W - n + 1, n), np.arange(0, H - n + 1, n))
        xs = xs.ravel().astype(np.int32); ys = ys.ravel().astype(np.int32); nb = len(xs)
        blk = np.zeros((nb, 10), dtype=np.int32)
        blk[:, 0] = xs; blk[:, 1] = ys; blk[:, 2] = n; blk[:, 3] = n; blk[:, 4] = -RANGE; blk[:, 5] = RANGE; blk[:, 6] = -RANGE; blk[:, 7] = RANGE
        a = np.zeros((nb, 4), dtype=np.int32); b = np.zeros((nb, 4), dtype=np.int32)
        O.orc_full_search(PO(org, base), S, PO(ref, base), S, P(blk), nb, 0, LAM, 2, 0, P(a), None, 0)
        R.refshim_full_search(1, PO(org, base), S, PO(ref, base), S, P(blk), nb, BD, 0, LAM, 2, 0, P(b), None, 0, 4, 1)
        assert not answered(b) or np.array_equal(a, b), n
        assert (a[:, :2] != 0).any()                                                     # the pan is found
        # SATD of the refinement pattern around every best vector
        desc = np.zeros((nb * K, 6), dtype=np.int32)
        bx = np.repeat(xs, K); by = np.repeat(ys, K)
        desc[:, 0] = bx; desc[:, 1] = by
        desc[:, 2] = bx + np.tile(np.array([p[0] for p in pat], dtype=np.int32), nb) + np.repeat(a[:, 0], K)
        desc[:, 3] = by + np.tile(np.array([p[1] for p in pat], dtype=np.int32), nb) + np.repeat(a[:, 1], K)
        desc[:, 4] = n; desc[:, 5] = n
        ca = np.zeros(nb * K, dtype=np.uint64); cb = np.zeros(nb * K, dtype=np.uint64)
        O.orc_dist_list(2, PO(org, base), S, PO(ref, base), S, P(desc), nb * K, 0, P(ca))
        R.refshim_dist_list(1, 2, PO(org, base), S, PO(ref, base), S, P(desc), nb * K, BD, 0, P(cb), 4)
        assert not answered(cb) or np.array_equal(ca, cb), n
        # residual of the best prediction -> DCT-II + quantiser at QP 37, inter and intra-period rounding
        resi = np.zeros((nb, n, n), dtype=np.int16)
        for i in range(nb):
            x, y, mx, my = int(xs[i]), int(ys[i]), int(a[i, 0]), int(a[i, 1])
            resi[i] = org[M + y:M + y + n, M + x:M + x + n] - ref[M + y + my:M + y + my + n, M + x + mx:M + x + mx + n]
        for irap in (0, 1):
            qa = np.zeros((nb, n, n), dtype=np.int16); sa = np.zeros(nb, dtype=np.int32); la = np.zeros(nb, dtype=np.int32)
            qb = np.zeros((nb, n, n), dtype=np.int16); sb = np.zeros(nb, dtype=np.int32); lb = np.zeros(nb, dtype=np.int32)
            coef = np.zeros((n, n), dtype=np.int32)
            for i in range(nb):
                assert O.orc_transform_quant(0, 0, P(resi[i]), n, n, n, BD, QP, irap, P(coef), P(qa[i]), PO(sa, i), PO(la, i)) == 0
            R.refshim_transform_quant_batch(0, 0, P(resi), nb, n, n, BD, QP, irap, P(qb), P(sb), P(lb), 4)
            assert not answered(qb, sb, lb) or np.array_equal(qa, qb) and np.array_equal(sa, sb) and np.array_equal(la, lb), (n, irap)
        assert (sa > 0).any() and (sa == 0).any()                                        # QP 37: some TUs survive, some quantise to zero


def test_mctf_motion_field_of_the_frame_pair(frame_pair):
    from test_mctf_host import OracleProvider
    from vvenc_b200 import mctf_host as MH
    org, ref, S = frame_pair
    o = np.ascontiguousarray(org[M:M + H, M:M + W]); r = np.ascontiguousarray(ref[M:M + H, M:M + W])
    R = refshim(); R.refshim_set_simd(b'AVX2')
    u = 8
    wb, hb = (W + u - 1) // u, (H + u - 1) // u
    exp = np.zeros((hb, wb, 4), dtype=np.int32)
    R.refshim_mctf_estimate_pyramid(1, P(o), P(r), W, H, BD, u, 0, 0, 0, P(exp))

    def make_provider(po_, pr_):
        a, b = MH.pad_edge(po_, 128), MH.pad_edge(pr_, 128)
        return OracleProvider(a, b, a.shape[1], 128, BD, 0)

    got = MH.estimate_pyramid(make_provider, o, r, u, False, BD, 0)
    assert np.array_equal(got['x'], exp[..., 0]) and np.array_equal(got['y'], exp[..., 1])
    assert np.array_equal(got['error'], exp[..., 2]) and np.array_equal(got['rmsme'].astype(np.int32), exp[..., 3])
    assert (got['x'] != 0).any()


def test_config1_1080p_block_sweep_sample():
    """BASELINE.json configs[1] -- 1920x1080 10-bit, SAD/SATD full-search sweep 4x4..64x64 -- as a CPU parity case on a seeded sample of blocks of every
    size (the whole frame runs on the GPU in tests/test_gpu_parity.py): search range +-16, then SATD at the best vector's neighbourhood"""
    sys.path.insert(0, ROOT)
    import bench
    w1, h1, m1 = 1920, 1080, 80
    org, ref, S = bench.synth_picture_pair(1080, w1, h1, m1)
    O = oracle(); R = refshim(); R.refshim_set_simd(b'AVX2')
    base = m1 * S + m1
    rs = np.random.RandomState(1080)
    pat = bench.refine_pattern(); K = len(pat)
    for n in (4, 8, 16, 32, 64):
        nb = 48
        blk = np.zeros((nb, 10), dtype=np.int32)
        blk[:, 0] = rs.randint(0, (w1 - n) // n + 1, size=nb) * n; blk[:, 1] = rs.randint(0, (h1 - n) // n + 1, size=nb) * n
        blk[:, 2] = n; blk[:, 3] = n; blk[:, 4] = -16; blk[:, 5] = 16; blk[:, 6] = -16; blk[:, 7] = 16
        blk[:, 8] = rs.randint(-20, 21, size=nb); blk[:, 9] = rs.randint(-20, 21, size=nb)
        for ss in ((0, 1) if n > 8 else (0,)):
            a = np.zeros((nb, 4), dtype=np.int32); b = np.zeros((nb, 4), dtype=np.int32)
            O.orc_full_search(PO(org, base), S, PO(ref, base), S, P(blk), nb, ss, 57.0, 2, 0, P(a), None, 0)
            R.refshim_full_search(1, PO(org, base), S, PO(ref, base), S, P(blk), nb, 10, ss, 57.0, 2, 0, P(b), None, 0, 4, 1)
            assert not answered(b) or np.array_equal(a, b), (n, ss)
        desc = np.zeros((nb * K, 6), dtype=np.int32)
        bx = np.repeat(blk[:, 0], K); by = np.repeat(blk[:, 1], K)
        desc[:, 0] = bx; desc[:, 1] = by
        desc[:, 2] = bx + np.tile(np.array([p[0] for p in pat], dtype=np.int32), nb) + np.repeat(a[:, 0], K)
        desc[:, 3] = by + np.tile(np.array([p[1] for p in pat], dtype=np.int32), nb) + np.repeat(a[:, 1], K)
        desc[:, 4] = n; desc[:, 5] = n
        for fam in (1, 2, 3):                                                          # SAD, SATD, fast SATD
            ca = np.zeros(nb * K, dtype=np.uint64); cb = np.zeros(nb * K, dtype=np.uint64)
            O.orc_dist_list(fam, PO(org, base), S, PO(ref, base), S, P(desc), nb * K, 0, P(ca))
            R.refshim_dist_list(1, fam, PO(org, base), S, PO(ref, base), S, P(desc), nb * K, 10, 0, P(cb), 4)
            assert not answered(cb) or np.array_equal(ca, cb), (n, fam)
