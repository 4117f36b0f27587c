"""CPU-only: the host-side replay of the MCTF motion search (vvenc_b200/mctf_host.py) against the reference's OWN MCTF::motionEstimationLuma
(run through oracle/_ref where it exists) and against itself through two providers.  The error numbers come from the CPU oracle here; on the GPU box
the same replay consumes vvb_mctf_search_grid / vvb_mctf_error_batch tables, which tests/test_gpu_parity.py pins to the same oracle."""
import ctypes
import numpy as np
import pytest
from _libs import answered, oracle, refshim, refshim_reset, have_ref_results, P, PO

from vvenc_b200 import mctf_host as MH


@pytest.fixture(autouse=True)
def _fresh_refshim_replay():
    refshim_reset()


class OracleProvider:
    """error tables from oracle/oracle.c on one padded picture pair (margin m, stride S)"""

    def __init__(self, org, ref, S, m, bit_depth=10, tap4=0):
        self.O = oracle(); self.O.orc_mctf_calc_var.restype = ctypes.c_double
        self.org = org; self.ref = ref; self.S = S; self.m = m; self.bd = bit_depth; self.tap4 = tap4

    def errors(self, cands):
        n = len(cands)
        desc = np.stack([cands['x'] + self.m, cands['y'] + self.m, cands['mvx'], cands['mvy'], cands['w'].astype(np.int32), cands['h'].astype(np.int32)], axis=1).astype(np.int32)
        out = np.zeros(n, dtype=np.int32)
        self.O.orc_mctf_err_list(self.tap4, P(self.org), self.S, P(self.ref), self.S, P(np.ascontiguousarray(desc)), n, self.bd, P(out))
        return out

    def grid(self, blocks, step, radius):
        k1 = 2 * radius + 1
        jj, ii = np.mgrid[0:k1, 0:k1]
        c = np.zeros((len(blocks), k1, k1), dtype=MH.CAND_DT)
        for f in ('x', 'y', 'w', 'h'):
            c[f] = blocks[f][:, None, None]
        c['mvx'] = blocks['mvx'][:, None, None] + (ii - radius)[None] * step; c['mvy'] = blocks['mvy'][:, None, None] + (jj - radius)[None] * step
        return self.errors(c.reshape(-1)).reshape(len(blocks), k1, k1)

    def calc_var(self, blocks):
        base = self.m * self.S + self.m
        return np.array([self.O.orc_mctf_calc_var(PO(self.org, base + int(b['y']) * self.S + int(b['x'])), self.S, int(b['w']), int(b['h'])) for b in blocks])


class FakeEngine:
    """same method signatures as vvenc_b200.CostEngine's MCTF calls, numbers from the oracle: exercises EngineProvider without a GPU"""

    def __init__(self, prov):
        self.p = prov

    def mctf_search_grid(self, org_plane, ref_plane, blocks, step, radius, low_res_filter=False):
        return self.p.grid(np.asarray(blocks), step, radius)

    def mctf_error_batch(self, org_plane, ref_plane, cands, low_res_filter=False):
        return self.p.errors(np.asarray(cands))

    def mctf_calc_var(self, plane, blocks):
        return self.p.calc_var(np.asarray(blocks))


def _pictures(seed, W, H, m, shift=(1, -2), noise=6):
    rs = np.random.RandomState(seed)
    S = W + 2 * m
    base = rs.randint(0, 1024, size=(H + 2 * m + 8, S + 8))
    sm = (base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) // 4
    org = np.ascontiguousarray(sm[4:4 + H + 2 * m, 4:4 + S].astype(np.int16))
    a = sm[4 + shift[0]:4 + shift[0] + H + 2 * m, 4 + shift[1]:4 + shift[1] + S]
    b = sm[4 + shift[0]:4 + shift[0] + H + 2 * m, 4 + shift[1] + 1:4 + shift[1] + 1 + S]
    ref = np.ascontiguousarray(np.clip((a + b + 1) // 2 + rs.randint(-noise, noise + 1, size=org.shape), 0, 1023).astype(np.int16))     # half-pel displacement
    return org, ref, S


def mctf_shard_case():
    """one target picture and three neighbour pictures with different displacements (tests/test_bands_gloo.py deals them over two ranks)"""
    rs = np.random.RandomState(77)
    W, H = 128, 96
    base = rs.randint(0, 1024, size=(H + 16, W + 16))
    sm = (base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) // 4
    org = np.ascontiguousarray(sm[8:8 + H, 8:8 + W].astype(np.int16))
    refs = []
    for (dy, dx, noise) in ((1, -2, 4), (-3, 2, 6), (2, 4, 9)):
        refs.append(np.ascontiguousarray(np.clip(sm[8 + dy:8 + dy + H, 8 + dx:8 + dx + W] + rs.randint(-noise, noise + 1, size=org.shape), 0, 1023).astype(np.int16)))
    return org, refs, 8


def _reference_level(opt, org, ref, S, m, W, H, bs, prev, factor, double_res, unit):
    R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    bxn, byn = W // bs, H // bs
    out = np.zeros((byn, bxn, 4), dtype=np.int32); ov = np.zeros((byn, bxn), dtype=np.float64)
    base = m * S + m
    if prev is not None:
        pv = np.ascontiguousarray(np.stack([prev[0], prev[1]], axis=-1).astype(np.int32))
        R.refshim_mctf_estimate_level(opt, PO(org, base), S, PO(ref, base), S, W, H, 10, bs, P(pv), prev[0].shape[1], prev[0].shape[0], factor, int(double_res), 0, unit, P(out), P(ov))
    else:
        R.refshim_mctf_estimate_level(opt, PO(org, base), S, PO(ref, base), S, W, H, 10, bs, None, 0, 0, factor, int(double_res), 0, unit, P(out), P(ov))
    return out, ov


@pytest.mark.skipif(not have_ref_results('test_mctf_host'), reason="neither oracle/_ref nor a recording of its calls")
@pytest.mark.parametrize("opt", [0, 1])
def test_replay_equals_reference_motion_estimation(opt):
    """three chained levels as MCTF::motionEstimationMCTF runs them (coarse without predictors, middle with predictors, final with doubleRes):
    every block's vector, error, rmsme and overlap equal the reference's own search"""
    W, H, m = 192, 128, 40
    org, ref, S = _pictures(5 + opt, W, H, m)
    prov = OracleProvider(org, ref, S, m)
    # level 1: no coarser field, block 32 -> range 8 integer grid
    a = MH.estimate_level(prov, W, H, 32, None, 2, False, 10, 16)
    r, _ = _reference_level(opt, org, ref, S, m, W, H, 32, None, 2, False, 16)
    assert not answered(r) or np.array_equal(a['x'], r[..., 0]) and np.array_equal(a['y'], r[..., 1]) and np.array_equal(a['error'], r[..., 2])
    # level 2: predictors from level 1 (same picture here, the control flow is what is under test), block 16, integer range 5
    prev = (a['x'], a['y'])
    b = MH.estimate_level(prov, W, H, 16, prev, 1, False, 10, 16)
    r, _ = _reference_level(opt, org, ref, S, m, W, H, 16, prev, 1, False, 16)
    assert not answered(r) or np.array_equal(b['x'], r[..., 0]) and np.array_equal(b['y'], r[..., 1]) and np.array_equal(b['error'], r[..., 2])
    # level 3: final level with sub-pel refinement and error scaling; 8x8 blocks so that `previous` is twice as coarse
    prev = (b['x'], b['y'])
    c = MH.estimate_level(prov, W, H, 8, prev, 1, True, 10, 8)
    r, ov = _reference_level(opt, org, ref, S, m, W, H, 8, prev, 1, True, 8)
    assert not answered(r) or np.array_equal(c['x'], r[..., 0]) and np.array_equal(c['y'], r[..., 1])
    assert not answered(r, ov) or np.array_equal(c['error'], r[..., 2]) and np.array_equal(c['rmsme'].astype(np.int32), r[..., 3]) and np.array_equal(c['overlap'], ov)
    assert (c['x'] & 15).any() or (c['y'] & 15).any()          # fractional vectors were chosen somewhere


def test_engine_provider_path_equals_oracle_provider():
    """EngineProvider (the GPU-facing adapter) driven by an oracle-backed engine with CostEngine's signatures gives the same field"""
    W, H, m = 128, 64, 40
    org, ref, S = _pictures(9, W, H, m, shift=(-1, 1))
    prov = OracleProvider(org, ref, S, m)
    eng = MH.EngineProvider(FakeEngine(prov), 0, 1)
    a = MH.estimate_level(prov, W, H, 16, None, 2, False)
    b = MH.estimate_level(eng, W, H, 16, None, 2, False)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    prev = (a['x'], a['y'])
    c = MH.estimate_level(prov, W, H, 8, prev, 1, True, 10, 8)
    d = MH.estimate_level(eng, W, H, 8, prev, 1, True, 10, 8)
    for k in c:
        assert np.array_equal(c[k], d[k]), k


@pytest.mark.skipif(not have_ref_results('test_mctf_host'), reason="neither oracle/_ref nor a recording of its calls")
@pytest.mark.parametrize("add_level,pattern,tap4", [(0, 0, 0), (1, 0, 0), (0, 1, 1), (1, 2, 1), (0, 2, 0)])
def test_pyramid_replay_equals_reference(add_level, pattern, tap4):
    """the whole motion search of one neighbour picture (MCTF::motionEstimationMCTF: 2x2-averaged pyramids + 4 or 5 chained levels) on a picture whose
    size is not a multiple of the coarse block sizes, for the three search patterns (MCTFSpeed 0 / 1-2 / 3-4) and both filter sets: the final field equals
    the reference's, vectors, scaled errors and rmsme"""
    rs = np.random.RandomState(21 + add_level)
    W, H = 208, 136
    base = rs.randint(0, 1024, size=(H + 16, W + 16))
    sm = (base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) // 4
    org = np.ascontiguousarray(sm[8:8 + H, 8:8 + W].astype(np.int16))
    a = sm[8 + 3:8 + 3 + H, 8 - 5:8 - 5 + W]; b = sm[8 + 3:8 + 3 + H, 8 - 4:8 - 4 + W]
    ref = np.ascontiguousarray(np.clip((a + b + 1) // 2 + rs.randint(-5, 6, size=org.shape), 0, 1023).astype(np.int16))
    R = refshim(); R.refshim_set_simd(b'AVX2')
    u = 8
    wb, hb = (W + u - 1) // u, (H + u - 1) // u
    exp = np.zeros((hb, wb, 4), dtype=np.int32)
    R.refshim_mctf_estimate_pyramid(1, P(org), P(ref), W, H, 10, u, add_level, pattern, tap4, P(exp))

    def make_provider(o, r):
        pad = 128
        po, pr = MH.pad_edge(o, pad), MH.pad_edge(r, pad)
        return OracleProvider(po, pr, po.shape[1], pad, 10, tap4)

    got = MH.estimate_pyramid(make_provider, org, ref, u, bool(add_level), 10, pattern)
    assert got['x'].shape == (hb, wb)
    assert np.array_equal(got['x'], exp[..., 0]) and np.array_equal(got['y'], exp[..., 1])
    assert np.array_equal(got['error'], exp[..., 2]) and np.array_equal(got['rmsme'].astype(np.int32), exp[..., 3])
    assert (got['x'] != 0).any() and ((got['x'] & 15).any() or (got['y'] & 15).any())
