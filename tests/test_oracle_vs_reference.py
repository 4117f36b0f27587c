"""CPU-only: a wider random sweep of the oracle against the reference, scalar and AVX2, in the style of test/vvenc_unit_test (tolerance 0).
The reference answers through oracle/_ref where it is built, else from its recorded calls (tests/golden/refshim, see _libs.refshim)."""
import numpy as np
import pytest
import cases as C
import impls
from _libs import answered, have_ref, have_ref_results, refshim_reset

pytestmark = pytest.mark.skipif(not have_ref_results('test_oracle_vs_reference'), reason="neither oracle/_ref nor a recording of its calls")


@pytest.fixture(autouse=True)
def _fresh_refshim_replay():
    refshim_reset()


@pytest.mark.parametrize("opt", [0, 1])
def test_dist_sweep(opt):
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    rs = np.random.RandomState(31 + opt)
    n = 0
    for w in (1, 2, 4, 8, 16, 32, 64, 128):
        for h in (1, 2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128):
            for fam in range(5):
                if fam >= 2 and (w < 2 or h % 2): continue
                if fam == 0 and w == 1 and opt: continue
                if fam == 4 and (w < 4 or h % 4): continue
                so = w if fam == 4 else w + int(rs.randint(0, 64)); sc = w if fam == 4 else w + int(rs.randint(0, 64))
                o = C.pel_block(rs, h, so, 0); c = C.pel_block(rs, h, sc, int(rs.randint(0, 4)))
                ss = int(rs.randint(0, 2)) if fam == 1 and h % 2 == 0 else 0
                assert O.dist(fam, o, so, c, sc, w, h, 10, ss) == R.dist(fam, o, so, c, sc, w, h, 10, ss), (fam, w, h, ss)
                n += 1
    assert n > 300


@pytest.mark.parametrize("opt", [0, 1])
def test_transform_quant_sweep(opt):
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    rs = np.random.RandomState(77 + opt)
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            for (th, tv) in ((0, 0), (2, 2), (1, 2), (2, 1), (1, 1)):
                if (th or tv) and (w > 32 or h > 32): continue
                amp = int(rs.choice([1023, 300, 20, 3])); st = w + int(rs.randint(0, 9))
                resi = rs.randint(-amp, amp + 1, size=(h, st)).astype(np.int16)
                qp = int(rs.randint(0, 64)); irap = int(rs.randint(0, 2))
                a = O.transform_quant(th, tv, resi, st, w, h, 10, qp, irap); b = R.transform_quant(th, tv, resi, st, w, h, 10, qp, irap)
                assert (not answered(b[0], b[1]) or np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])) and a[2:4] == b[2:4], (th, tv, w, h, qp, irap)
                for dq in (0, 1):
                    assert O.need_rdoq(a[0], w, h, 10, qp, dq) == R.need_rdoq(a[0], w, h, 10, qp, dq)


def test_fwd_core_like_reference_unit_test():
    # vvenc_unit_test.cpp:1085-1140: random 8-bit matrix, 11-bit signed src, random line/reducedLine/cutoff/shift
    import ctypes
    from _libs import oracle, refshim, P
    O = oracle(); R = refshim()
    rs = np.random.RandomState(5)
    for tr in (4, 8, 16, 32, 64):
        for rep in range(20):
            line = int(rs.choice([4, 8, 16, 32, 64])); red = line - int(rs.choice([0, line // 2])) ; cut = tr - int(rs.choice([0, tr // 2]))
            shift = int(rs.randint(1, 17))
            tc = C.aligned((tr, tr), np.int16); tc[:] = rs.randint(-128, 128, size=(tr, tr))
            src = C.aligned((line, tr), np.int32); src[:] = rs.randint(-1024, 1024, size=(line, tr))
            d1 = C.aligned((tr, line), np.int32); d2 = C.aligned((tr, line), np.int32)
            R.refshim_fwd_core(tr, P(tc), P(src), P(d1), line, red, cut, shift); O.orc_fwd_core(tr, P(tc), P(src), P(d2), line, red, cut, shift)
            known = answered(d1)
            d1 = d1[:, :red]; d2 = d2[:, :red]      # columns past reducedLine are unspecified (vvenc_unit_test.cpp:1117-1119)
            assert not known or np.array_equal(d1, d2), (tr, line, red, cut, shift)


@pytest.mark.parametrize("opt", [0, 1])
def test_mctf_all_phases(opt):
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    rs = np.random.RandomState(11)
    m = C.MCTF_MARGIN
    for (w, h) in ((8, 8), (16, 16), (32, 24), (64, 64)):
        org = rs.randint(0, 1024, size=(h, w + 3)).astype(np.int16); buf = rs.randint(0, 1024, size=(h + 2 * m, w + 2 * m)).astype(np.int16)
        for tap4 in (0, 1):
            for fx in range(16):
                for fy in range(16):
                    mvx = 16 * int(rs.randint(-2, 3)) + fx; mvy = 16 * int(rs.randint(-2, 3)) + fy
                    a = O.mctf_err(tap4, org, w + 3, buf, w + 2 * m, m, m, mvx, mvy, w, h, 10)
                    b = R.mctf_err(tap4, org, w + 3, buf, w + 2 * m, m, m, mvx, mvy, w, h, 10)
                    assert a == b, (w, h, tap4, mvx, mvy)


@pytest.mark.parametrize("opt", [0, 1])
def test_affine(opt):
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    for row in C.affine_cases():
        w, h, ps, ds, six, seed = [int(v) for v in row]
        pred, resi, gx, gy = C.affine_inputs(row)
        for vert in (0, 1):
            r = R.sobel(vert, pred, ps, ds, w, h)
            assert not answered(r) or np.array_equal(O.sobel(vert, pred, ps, ds, w, h), r)
        r = R.equal_coeff(six, resi, ps, gx, gy, ds, w, h)
        assert not answered(r) or np.array_equal(O.equal_coeff(six, resi, ps, gx, gy, ds, w, h), r)


@pytest.mark.parametrize("opt", [0, 1])
def test_full_search_with_tables(opt):
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    sc = C.search_case(seed=991)
    for ss in (0, 1):
        a, ta = O.full_search(sc, ss, True); b, tb = R.full_search(sc, ss, True)
        assert not answered(b, tb) or np.array_equal(a, b) and np.array_equal(ta, tb)


def test_tables_match_reference():
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))
    import gen_tables as g
    from _libs import refshim, P
    R = refshim()
    for (t, N), m in g.matrices().items():
        ref = np.zeros((N, N), dtype=np.int16)
        assert R.refshim_tr_matrix(t, N, P(ref)) == 0
        assert not answered(ref) or np.array_equal(ref, m), (t, N)
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            a = np.zeros(1024, dtype=np.int32); b = np.zeros(1024, dtype=np.int32)
            from _libs import oracle
            assert R.refshim_scan_order(w, h, P(a)) == oracle().orc_scan_order(w, h, P(b)) and (not answered(a) or np.array_equal(a, b))


@pytest.mark.parametrize("opt", [0, 1])
def test_inverse_path_sweep(opt):
    """dequant + inverse transform (TrQuant::invTransformNxN), random levels over the full QP range, 8/10/12 bit"""
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    rs = np.random.RandomState(177 + opt)
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            for (th, tv) in ((0, 0), (2, 2), (1, 2), (2, 1), (1, 1)):
                if (th or tv) and (w > 32 or h > 32): continue
                for bd in (8, 10, 12):
                    amp = int(rs.choice([32767, 2000, 40, 2])); qp = int(rs.randint(-6 * (bd - 8), 64)); st = w + int(rs.randint(0, 9))
                    q = rs.randint(-amp - 1, amp + 1, size=(h, w)).astype(np.int16)
                    q[rs.rand(h, w) < 0.5] = 0
                    a = O.inv_transform_quant(th, tv, q, w, h, bd, qp, st); b = R.inv_transform_quant(th, tv, q, w, h, bd, qp, st)
                    assert not answered(b[0]) or np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), (th, tv, w, h, bd, qp)


@pytest.mark.parametrize("opt", [0, 1])
def test_tu_roundtrip_sweep(opt):
    """residual -> transformNxN -> invTransformNxN -> reconstruct -> SSE, as xIntraCodingTUBlock chains them"""
    O = impls.OracleImpl(); R = impls.RefImpl(opt)
    rs = np.random.RandomState(277 + opt)
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            for (th, tv) in ((0, 0), (2, 2), (2, 1)):
                if (th or tv) and (w > 32 or h > 32): continue
                amp = int(rs.choice([400, 60, 8])); qp = int(rs.randint(4, 56)); irap = int(rs.randint(0, 2)); so = w + int(rs.randint(0, 9)); ps = w + int(rs.randint(0, 9))
                org = rs.randint(0, 1024, size=(h, so)).astype(np.int16)
                pred = np.zeros((h, ps), dtype=np.int16)
                pred[:, :w] = np.clip(org[:, :w] + rs.randint(-amp, amp + 1, size=(h, w)), 0, 1023)
                a = O.tu_roundtrip(th, tv, org, so, pred, ps, w, h, 10, qp, irap); b = R.tu_roundtrip(th, tv, org, so, pred, ps, w, h, 10, qp, irap)
                assert not answered(b[0], b[1]) or np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2], (th, tv, w, h, qp, irap, a[2], b[2])


@pytest.mark.parametrize("opt", [0, 1])
def test_mctf_apply_stage(opt):
    """applyFrac + applyPlanarCorrection + applyBlock chained per block as xFinalizeBlkLine does: oracle == reference (float results included)"""
    from _libs import oracle, refshim
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    for (seed, W, H, refs, bs, bd, tap4, planar) in C.MCTF_APPLY_CASES:
        case = C.mctf_apply_case(seed, W, H, 24, refs, bs, bd)
        a = impls.mctf_apply_expected(O, 'orc', case, tap4, planar)
        known = np.ones(a.shape, dtype=bool)
        b = impls.mctf_apply_expected(R, 'refshim', case, tap4, planar, opt, known)
        assert np.array_equal(a[known], b[known]), (seed, np.abs(a.astype(int) - b)[known].max())
        assert np.any(a != case['org'][24:24 + H, 24:24 + W])           # the filter does something


@pytest.mark.parametrize("opt", [0, 1])
def test_mctf_calc_var(opt):
    import ctypes
    from _libs import oracle, refshim, P
    O = oracle(); R = refshim()
    O.orc_mctf_calc_var.restype = ctypes.c_double; R.refshim_mctf_calc_var.restype = ctypes.c_double
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(88)
    for (w, h) in ((8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 8)):
        for bd in (8, 10):
            org = C.aligned((h, w + 16), np.int16); org[:] = rs.randint(0, 1 << bd, size=(h, w + 16))
            assert O.orc_mctf_calc_var(P(org), w + 16, w, h) == R.refshim_mctf_calc_var(opt, P(org), w + 16, w, h), (w, h, bd)


@pytest.mark.parametrize("opt", [0, 1])
def test_two_pass_interpolation(opt):
    """filterHor(isLast=false) + filterVer(isFirst=false, isLast=true), every quarter-pel phase pair, the 8/6/4-tap ME filter sets and the
    alternative half-pel filter, 8 and 10 bit, extreme content included"""
    from _libs import oracle, refshim, P, PO
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(11 + opt)
    for bd in (8, 10, 12):
        mx = (1 << bd) - 1
        for (w, h) in ((8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (64, 32)):
            S = w + 32
            src = rs.randint(0, mx + 1, size=(h + 24, S)).astype(np.int16)
            if (w, h) == (8, 8):
                src[:] = np.where(rs.randint(0, 2, size=src.shape) > 0, mx, 0)
            for (rt, alt) in ((0, 0), (1, 0), (2, 0), (0, 1), (2, 1)):
                for fx in range(4):
                    for fy in range(4):
                        d1 = np.zeros((h, w), np.int16); d2 = np.zeros((h, w), np.int16)
                        O.orc_if_two_pass(PO(src, 8 * S + 12), S, w, h, fx, fy, bd, rt, alt, P(d1), w)
                        R.refshim_if_two_pass(opt, PO(src, 8 * S + 12), S, w, h, fx, fy, bd, rt, alt, P(d2), w)
                        assert not answered(d2) or np.array_equal(d1, d2), (bd, w, h, rt, alt, fx, fy)


@pytest.mark.parametrize("opt", [0, 1])
def test_full_search_against_the_reference_member_function(opt, golden):
    """InterSearch::xPatternSearch itself (called as a member on an InterSearch whose only live members are the ones it reads) against the oracle's
    replay and the golden argmins; sub-sampling through RdCost::setDistParam's own subShiftMode rule (mode 2: every second row when h > 8)"""
    from _libs import refshim, P, PO
    R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    O = impls.OracleImpl()
    sc = C.search_case()
    n = len(sc['blk']); S = sc['stride']; base = sc['margin'] * S + sc['margin']
    for ss, mode in ((0, 0), (1, 2)):
        out = np.zeros((n, 4), dtype=np.int32)
        R.refshim_pattern_search_member(opt, PO(sc['org'], base), S, PO(sc['ref'], base), S, P(sc['blk']), n, 10, mode, sc['lam'], sc['cost_scale'], sc['imv_shift'], P(out))
        same = [i for i in range(n) if ss == 0 or sc['blk'][i][3] > 8]
        assert len(same) >= 20
        assert np.array_equal(out[same], O.full_search(sc, ss)[same])
        assert np.array_equal(out[same], golden['search_best_ss%d' % ss][same])


@pytest.mark.parametrize("opt", [0, 1])
def test_mctf_apply_against_the_reference_member_function(opt):
    """MCTF::bilateralFilter -> xFinalizeBlkLine called as members on whole small pictures (unit 8 and 16, QP on both sides of the planar-correction
    threshold, 6-tap and 4-tap apply filters, clipped edge blocks): the oracle chain fed with the same strengths / sigma gives the same picture"""
    import ctypes
    from _libs import oracle, refshim, P
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(303 + opt)
    for (W, H, unit, nrefs, qp, tap4, reorder) in ((96, 64, 16, 4, 22, 0, 1), (72, 40, 8, 6, 40, 0, 1), (64, 48, 16, 2, 32, 1, 0), (48, 32, 8, 8, 27, 0, 1)):
        base = rs.randint(0, 1024, size=(H + 8, W + 8))
        sm = (base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) // 4
        org = np.ascontiguousarray(sm[4:4 + H, 4:4 + W].astype(np.int16))
        refs = []
        for a in ([3, 12, 60, 300] * 2)[:nrefs]:
            dy = int(rs.randint(-1, 2)); dx = int(rs.randint(-1, 2))
            refs.append(np.ascontiguousarray(np.clip(sm[4 + dy:4 + dy + H, 4 + dx:4 + dx + W] + rs.randint(-a, a + 1, size=org.shape), 0, 1023).astype(np.int16)))
        wb, hb = (W + unit - 1) // unit, (H + unit - 1) // unit
        mv = np.zeros((nrefs, hb * wb, 4), dtype=np.int32)
        mv[..., 0] = rs.randint(-16 * 5, 16 * 5 + 1, size=(nrefs, hb * wb)); mv[..., 1] = rs.randint(-16 * 5, 16 * 5 + 1, size=(nrefs, hb * wb))
        mv[..., 2] = rs.choice([3, 20, 49, 50, 75, 100, 101, 400], size=(nrefs, hb * wb)); mv[..., 3] = rs.choice([0, 1, 5, 22, 60], size=(nrefs, hb * wb))
        idx = np.array([i % 6 for i in range(nrefs)], dtype=np.int32)
        ptrs = (ctypes.c_void_p * nrefs)(*[r.ctypes.data for r in refs])
        got = np.zeros((H, W), dtype=np.int16); strg = np.zeros(nrefs, dtype=np.float64); sig = ctypes.c_double()
        overall = 0.95
        R.refshim_mctf_bilateral_filter(opt, P(org), ptrs, nrefs, P(np.ascontiguousarray(mv)), P(idx), W, H, 10, unit, qp, ctypes.c_double(overall), reorder, tap4,
                                        P(got), P(strg), ctypes.byref(sig))
        assert sig.value == 9.0 * (128.0 + 3.0 / 256.0 * qp * qp * qp)                      # 10 bit: bitDepthDiffWeighting = 1
        if not answered(got, strg):
            continue
        pad = 128
        case = dict(org=np.ascontiguousarray(np.pad(org, pad, mode='edge')), refs=[np.ascontiguousarray(np.pad(r, pad, mode='edge')) for r in refs],
                    stride=W + 2 * pad, margin=pad, W=W, H=H, mvs=mv, strengths=strg, ws=overall * 0.4, sigma=sig.value, bs=unit, bd=10, num_refs=nrefs)
        exp = impls.mctf_apply_expected(O, 'orc', case, tap4, 1 if qp <= 32 else 0)
        assert np.array_equal(got, exp), (W, H, unit, nrefs, qp, int(np.abs(got.astype(int) - exp).max()))
        assert np.any(got != org)


@pytest.mark.parametrize("opt", [0, 1])
def test_fractional_refinement_against_the_reference_member_function(opt):
    """InterSearch::xPatternSearchFracDIF itself (xExtDIFUpSamplingH/Q + both rounds of xPatternRefinement, m_fastSubPel = 0) against the replay of the two
    rounds on the oracle's 7x7 quarter-pel table: the chosen half / quarter offsets and the final cost agree -- for the 8-, 6- and 4-tap ME filter sets,
    SATD and SAD, and vectors of both parities.  This pins (a) that every filtered block of the encoder is the two-pass interpolation the table holds and
    (b) the host-side selection in vvenc_b200.candidates.subpel_refinement."""
    import ctypes
    from _libs import oracle, refshim, P, PO
    from vvenc_b200 import candidates as cand
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    R.refshim_frac_search_member.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    O.orc_mv_cost.restype = ctypes.c_uint64
    case = C.frac_case(5151 + opt)
    S = case['stride']; base = case['margin'] * S + case['margin']
    rs = np.random.RandomState(17)
    lam = 57.25
    checked = 0
    for (w, h) in ((8, 8), (16, 16), (32, 32), (64, 64)):
        n = 5
        blk = np.zeros((n, 8), dtype=np.int32)
        for k in range(n):
            blk[k] = (int(rs.randint(0, case['W'] - w + 1)), int(rs.randint(0, case['H'] - h + 1)), w, h, int(rs.randint(-6, 7)), int(rs.randint(-6, 7)),
                      int(rs.randint(-40, 41)), int(rs.randint(-40, 41)))
        for (rt, had, alt) in ((2, 1, 0), (0, 1, 0), (1, 1, 0), (2, 0, 0), (2, 1, 1)):
            out = np.zeros((n, 6), dtype=np.int32)
            R.refshim_frac_search_member(opt, PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk)), n, 10, lam, rt, had, alt, 0, P(out))
            tab = np.zeros((n, 7, 7), dtype=np.uint32)
            b6 = np.ascontiguousarray(blk[:, :6])
            O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(b6), n, 2 if had else 1, 10, rt, alt, P(tab))
            for k in range(n):
                ph, pv = int(blk[k, 6]), int(blk[k, 7])
                half, quarter, cost = cand.subpel_refinement(tab[k], (int(blk[k, 4]), int(blk[k, 5])), lambda x, y, cs: int(O.orc_mv_cost(lam, x, y, ph, pv, cs, 0)),
                                                             quarter_round=not alt)
                got_cost = (int(out[k, 4]) & 0xffffffff) | (int(out[k, 5]) << 32)
                assert (half, quarter, cost) == ((int(out[k, 0]), int(out[k, 1])), (int(out[k, 2]), int(out[k, 3])), got_cost), (w, h, rt, had, alt, k, half, quarter, cost, out[k])
                checked += 1
    assert checked == 100
    # rectangular PUs: SATD built from the 16x8 / 8x16 / 8x4 / 4x8 tiles (RdCost.cpp:1840-1905, fp64 normalisation) -- not offered by vvb_frac_cost_grid yet, the
    # oracle's table already equals what the member sees
    for (w, h) in ((16, 8), (8, 16), (32, 16), (16, 32), (8, 4), (4, 8), (4, 4), (64, 32)):
        n = 4
        blk = np.zeros((n, 8), dtype=np.int32)
        for k in range(n):
            blk[k] = (int(rs.randint(0, case['W'] - w + 1)), int(rs.randint(0, case['H'] - h + 1)), w, h, int(rs.randint(-6, 7)), int(rs.randint(-6, 7)),
                      int(rs.randint(-40, 41)), int(rs.randint(-40, 41)))
        out = np.zeros((n, 6), dtype=np.int32)
        R.refshim_frac_search_member(opt, PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk)), n, 10, lam, 2, 1, 0, 0, P(out))
        tab = np.zeros((n, 7, 7), dtype=np.uint32)
        O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk[:, :6])), n, 2, 10, 2, 0, P(tab))
        for k in range(n):
            ph, pv = int(blk[k, 6]), int(blk[k, 7])
            half, quarter, cost = cand.subpel_refinement(tab[k], (int(blk[k, 4]), int(blk[k, 5])), lambda x, y, cs: int(O.orc_mv_cost(lam, x, y, ph, pv, cs, 0)))
            got_cost = (int(out[k, 4]) & 0xffffffff) | (int(out[k, 5]) << 32)
            assert (half, quarter, cost) == ((int(out[k, 0]), int(out[k, 1])), (int(out[k, 2]), int(out[k, 3])), got_cost), ('rect', w, h, k)
    # m_fastHad (the faster / fast presets): xPatternRefinement asks for DF_HAD_fast -- the 16x16_fast tiles on square blocks that are multiples of 32, the plain
    # tiles elsewhere (RdCost.cpp:1818-1938).  The same replay on the oracle's table of that family gives the member's offsets and cost.
    for (w, h) in ((16, 16), (32, 32), (64, 64)):
        n = 5
        blk = np.zeros((n, 8), dtype=np.int32)
        for k in range(n):
            blk[k] = (int(rs.randint(0, case['W'] - w + 1)), int(rs.randint(0, case['H'] - h + 1)), w, h, int(rs.randint(-6, 7)), int(rs.randint(-6, 7)),
                      int(rs.randint(-40, 41)), int(rs.randint(-40, 41)))
        out = np.zeros((n, 6), dtype=np.int32)
        R.refshim_frac_search_member(opt, PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk)), n, 10, lam, 2, 2, 0, 0, P(out))
        tab = np.zeros((n, 7, 7), dtype=np.uint32); plain = np.zeros((n, 7, 7), dtype=np.uint32)
        O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk[:, :6])), n, 3, 10, 2, 0, P(tab))
        O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk[:, :6])), n, 2, 10, 2, 0, P(plain))
        assert np.array_equal(tab, plain) == (w < 32)                      # the fast tiles only exist from 32x32 upwards
        for k in range(n):
            ph, pv = int(blk[k, 6]), int(blk[k, 7])
            half, quarter, cost = cand.subpel_refinement(tab[k], (int(blk[k, 4]), int(blk[k, 5])), lambda x, y, cs: int(O.orc_mv_cost(lam, x, y, ph, pv, cs, 0)))
            got_cost = (int(out[k, 4]) & 0xffffffff) | (int(out[k, 5]) << 32)
            assert (half, quarter, cost) == ((int(out[k, 0]), int(out[k, 1])), (int(out[k, 2]), int(out[k, 3])), got_cost), ('fastHad', w, h, k)
    # the preset control (m_fastSubPel = 1): positions are skipped by the encoder's own heuristics, but whatever position it ends on, its cost must be the
    # table entry of that position plus the vector rate -- the half-pel blocks filtered inside xPatternRefinement and the partial xExtDIFUpSamplingQ planes
    # are the same two-pass interpolations
    for (w, h) in ((8, 8), (16, 16), (32, 32)):
        n = 8
        blk = np.zeros((n, 8), dtype=np.int32)
        for k in range(n):
            blk[k] = (int(rs.randint(0, case['W'] - w + 1)), int(rs.randint(0, case['H'] - h + 1)), w, h, int(rs.randint(-6, 7)), int(rs.randint(-6, 7)),
                      int(rs.randint(-40, 41)), int(rs.randint(-40, 41)))
        out = np.zeros((n, 6), dtype=np.int32)
        R.refshim_frac_search_member(opt, PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk)), n, 10, lam, 2, 1, 0, 1, P(out))
        tab = np.zeros((n, 7, 7), dtype=np.uint32)
        O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk[:, :6])), n, 2, 10, 2, 0, P(tab))
        for k in range(n):
            ph, pv = int(blk[k, 6]), int(blk[k, 7]); mx, my = int(blk[k, 4]), int(blk[k, 5])
            hx, hy, qx, qy = [int(v) for v in out[k, :4]]
            got_cost = (int(out[k, 4]) & 0xffffffff) | (int(out[k, 5]) << 32)
            c_half = int(tab[k][2 * hy + 3][2 * hx + 3]) + int(O.orc_mv_cost(lam, 2 * mx + hx, 2 * my + hy, ph, pv, 1, 0))
            ok = got_cost == c_half
            if abs(qx) <= 1 and abs(qy) <= 1:
                c_q = int(tab[k][2 * hy + qy + 3][2 * hx + qx + 3]) + int(O.orc_mv_cost(lam, 2 * (2 * mx + hx) + qx, 2 * (2 * my + hy) + qy, ph, pv, 0, 0))
                ok = ok or got_cost == c_q
            assert ok, (w, h, k, out[k], c_half)


@pytest.mark.parametrize("opt", [0, 1])
def test_fast_subpel_replay_equals_the_reference_member(opt):
    """m_fastSubPel = 1 (every preset between `fast` and `slow`): candidates.subpel_refinement_fast -- the early stops of the half-pel round, the pattern id and the
    skip table of the quarter-pel round, the carried-over threshold -- on the oracle's 7x7 table gives the offsets and the cost of InterSearch::xPatternSearchFracDIF
    itself, for square and rectangular PUs, SATD / fast SATD / SAD, and a lambda range that moves the decision between distortion and rate"""
    import ctypes
    from _libs import oracle, refshim, P, PO
    from vvenc_b200 import candidates as cand
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    R.refshim_frac_search_member.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    O.orc_mv_cost.restype = ctypes.c_uint64
    case = C.frac_case(7171 + opt)
    S = case['stride']; base = case['margin'] * S + case['margin']
    rs = np.random.RandomState(29)
    checked = 0; quarter_rounds = 0; early = 0; dirs = set()
    for (w, h, had) in ((8, 8, 1), (16, 16, 1), (32, 32, 2), (64, 64, 2), (16, 8, 1), (8, 16, 1), (32, 16, 2), (8, 4, 1), (4, 8, 1), (16, 16, 0), (64, 32, 1)):
        for lam in (4.0, 57.25, 900.0):
            n = 10
            blk = np.zeros((n, 8), dtype=np.int32)
            for k in range(n):
                blk[k] = (int(rs.randint(0, case['W'] - w + 1)), int(rs.randint(0, case['H'] - h + 1)), w, h, int(rs.randint(-6, 7)), int(rs.randint(-6, 7)),
                          int(rs.randint(-40, 41)), int(rs.randint(-40, 41)))
            out = np.full((n, 6), -99, dtype=np.int32)
            R.refshim_frac_search_member(opt, PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk)), n, 10, lam, 2, had, 0, 1, P(out))
            tab = np.zeros((n, 7, 7), dtype=np.uint32)
            O.orc_frac_cost_grid(PO(case['org'], base), S, PO(case['ref'], base), S, P(np.ascontiguousarray(blk[:, :6])), n, 3 if had == 2 else (2 if had else 1), 10, 2, 0, P(tab))
            for k in range(n):
                ph, pv = int(blk[k, 6]), int(blk[k, 7])
                half, quarter, cost = cand.subpel_refinement_fast(tab[k], (int(blk[k, 4]), int(blk[k, 5])), lambda x, y, cs: int(O.orc_mv_cost(lam, x, y, ph, pv, cs, 0)))
                got_cost = (int(out[k, 4]) & 0xffffffff) | (int(out[k, 5]) << 32)
                assert half == (int(out[k, 0]), int(out[k, 1])) and cost == got_cost, (w, h, had, lam, k, half, quarter, cost, out[k])
                if quarter is None:
                    assert (int(out[k, 2]), int(out[k, 3])) == (0, 0), (w, h, k, out[k])        # the probe passes a zero rcMvQter; the member leaves it alone
                    early += 1
                else:
                    assert quarter == (int(out[k, 2]), int(out[k, 3])), (w, h, had, lam, k, quarter, out[k])
                    quarter_rounds += 1
                dirs.add(half)
                checked += 1
    assert checked == 330 and quarter_rounds > 100 and len(dirs) >= 5, (checked, quarter_rounds, early, dirs)


@pytest.mark.parametrize("opt", [0, 1])
def test_sign_bit_hiding_against_the_reference(opt):
    """Quant::quant with slice->signDataHidingEnabled (the RDOQ = 2 presets run the plain quantiser next to sign hiding, vvencCfg.cpp:2675-2677): xSignBitHidingHDQ
    (Quant.cpp:377-518) on top of QuantCore -- levels, absSum and lastPos of the oracle equal the reference for every TU shape, transform pair, QP and slice type,
    and hiding changes levels in a good share of the cases"""
    import ctypes
    from _libs import oracle, refshim, P
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rows = C.tq_cases()
    changed = 0; moved_last = 0; n = 0
    for row in rows[::2] if opt else rows:
        th, tv, w, h, st, amp, qp, irap, bd, seed = [int(v) for v in row]
        resi = C.tq_inputs(row)
        for sh in (1,):
            coefR = np.zeros((h, w), dtype=np.int32); qR = np.zeros((h, w), dtype=np.int16); sR = ctypes.c_int32(); lR = ctypes.c_int32()
            rc = R.refshim_transform_quant_sdh(th, tv, P(resi), st, w, h, bd, qp, irap, sh, P(coefR), P(qR), ctypes.byref(sR), ctypes.byref(lR))
            if rc:
                continue
            coefO = np.zeros((h, w), dtype=np.int32); qO = np.zeros((h, w), dtype=np.int16); sO = ctypes.c_int32(); lO = ctypes.c_int32()
            assert O.orc_transform_quant_ex(th, tv, P(resi), st, w, h, bd, qp, irap, sh, P(coefO), P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
            assert (not answered(qR) or np.array_equal(qO, qR)) and sO.value == sR.value and lO.value == lR.value, (row, int((qO != qR).sum()), sO.value, sR.value, lO.value, lR.value)
            q0 = np.zeros((h, w), dtype=np.int16); s0 = ctypes.c_int32(); l0 = ctypes.c_int32()
            O.orc_transform_quant_ex(th, tv, P(resi), st, w, h, bd, qp, irap, 0, P(coefO), P(q0), ctypes.byref(s0), ctypes.byref(l0))
            changed += int(not np.array_equal(q0, qO)); moved_last += int(l0.value != lO.value); n += 1
            assert s0.value == sO.value                                # uiAbsSum is QuantCore's sum, hiding does not update it
    assert n > 100 and changed > n // 4, (n, changed, moved_last)


@pytest.mark.parametrize("opt", [0, 1])
def test_lfnst_forward_against_the_reference(opt):
    """TrQuant::transformNxN for intra TUs with an LFNST index (xT with the LFNST zero-out, xFwdLfnst, plain quantiser on coefficient group 0, xNeedRDOQ): the
    oracle's restatement gives the reference's coefficients, levels, absSum, lastPos and RDOQ flag for every TU shape that can carry LFNST, both indices, intra
    modes of all four kernel sets with and without transposition, wide-angle remapping on rectangular TUs, with and without sign-bit hiding"""
    import ctypes
    from _libs import oracle, refshim, P
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(31 + opt)
    sets = set(); n = 0
    for (w, h) in ((4, 4), (8, 8), (4, 8), (8, 4), (16, 16), (4, 16), (16, 4), (8, 16), (32, 32), (32, 8), (64, 64), (16, 64)):
        for mode in (0, 1, 2, 10, 18, 23, 34, 35, 44, 50, 58, 66):
            for idx in (1, 2):
                amp = int(rs.choice([1023, 200, 30]))
                qp = int(rs.randint(18, 46)); irap = int(rs.randint(0, 2)); sh = int(rs.randint(0, 2))
                resi = rs.randint(-amp, amp + 1, size=(h, w)).astype(np.int16)
                cR = np.zeros((h, w), dtype=np.int32); qR = np.zeros((h, w), dtype=np.int16); sR = ctypes.c_int32(); lR = ctypes.c_int32(); nR = ctypes.c_int32()
                st = np.zeros(2, dtype=np.int32)
                assert R.refshim_transform_quant_lfnst(P(resi), w, w, h, 10, qp, irap, sh, mode, idx, P(cR), P(qR), ctypes.byref(sR), ctypes.byref(lR), ctypes.byref(nR), P(st)) == 0
                cO = np.zeros((h, w), dtype=np.int32); qO = np.zeros((h, w), dtype=np.int16); sO = ctypes.c_int32(); lO = ctypes.c_int32()
                assert O.orc_transform_quant_lfnst(P(resi), w, w, h, 10, qp, irap, sh, int(st[0]), idx, int(st[1]), P(cO), P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
                assert not answered(cR) or np.array_equal(cO, cR), (w, h, mode, idx, st, np.argwhere(cO != cR)[:4])
                assert (not answered(qR) or np.array_equal(qO, qR)) and sO.value == sR.value and lO.value == lR.value, (w, h, mode, idx, qp, sh)
                assert O.orc_need_rdoq(P(cO), w, h, 10, qp, 0) == nR.value
                sets.add((int(st[0]), int(st[1]))); n += 1
    assert n == 288 and len(sets) >= 6, (n, sets)


def test_dep_quant_scan_tables_equal_the_reference_rom():
    """ScanInfo / NbInfoSbb / NbInfoOut of DQIntern::Rom (DepQuant.cpp:75-342) for all 25 luma shapes: the tables the library uploads are the reference's"""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            nc = min(w, 32) * min(h, 32)
            a = np.zeros(nc * 24, np.uint8); b = np.zeros(nc * 16, np.uint8); c = np.zeros(nc * 24, np.uint8); d = np.zeros(nc * 16, np.uint8)
            assert R.refshim_dep_quant_tables(w, h, P(a), P(b)) == nc and O.orc_dep_quant_tables(w, h, P(c), P(d)) == nc
            assert not answered(a, b) or np.array_equal(a, c) and np.array_equal(b, d), (w, h)


@pytest.mark.parametrize("opt", [0, 1])
def test_dep_quant_against_the_reference_member(opt):
    """DepQuant::xQuantDQ on the probe's TU rig (CABAC contexts initialised for the slice QP) against the restatement fed with the rate tables the reference's
    RateEstimator derived: levels, absSum, lastPos for every TU shape class, 8 / 10 bit, QP 17..51, explicit MTS and SBT zero-out, LFNST position limit, intra and
    inter CUs; opt 0 = the scalar members (checkAllRdCosts, updateStates, ... of DepQuant.cpp), 1 = what initDepQuantX86 installs.  Also the Quantizer constants."""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    rs = np.random.RandomState(500 + opt)
    n = 0; nonzero = 0; big = 0
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (64, 64), (8, 4), (4, 16), (32, 8), (16, 64), (64, 32), (32, 16), (4, 32), (64, 4), (8, 16), (16, 4)]:
        for bd in (10, 8):
            for qp in (17, 22, 27, 32, 37, 42, 51):
                for trial in range(5):
                    lam = float(rs.choice([3.0, 11.7, 30.0, 57.3, 120.0, 800.0, 4000.0]))
                    scale = float(rs.choice([5, 20, 60, 200, 600, 2000, 30000]))
                    dec = float(rs.choice([0.1, 0.5, 1.0, 1.5]))
                    coef = rs.laplace(0, scale, size=(h, w)) * (1.0 / (1 + np.add.outer(np.arange(h), np.arange(w))) ** dec)
                    coef = np.clip(coef, -32768, 32767).astype(np.int32)
                    if w > 32: coef[:, 32:] = 0
                    if h > 32: coef[32:, :] = 0
                    mts = int(rs.choice([0, 0, 2, 3, 5])) if (w <= 32 and h <= 32) else 0
                    lf = int(rs.choice([0, 0, 0, 1, 2])) if mts == 0 else 0
                    sbt = int(rs.choice([0, 0, 0, 1])) if (mts == 0 and lf == 0) else 0
                    intra = 1 if lf else (0 if sbt else int(rs.randint(2)))
                    zo = 1 if (mts > 1 or (sbt and w <= 32 and h <= 32)) else 0
                    thr = int(rs.choice([8, 8, 4, 16]))
                    qR = np.zeros((h, w), np.int16); sR = ctypes.c_int32(); lR = ctypes.c_int32(); rates = np.zeros(266, np.int32); kR = np.zeros(9, np.int64)
                    assert R.refshim_dep_quant(P(coef), w, h, bd, qp, mts, intra, lf, sbt, lam, thr, opt, int(rs.randint(17, 52)), trial % 3, P(qR), ctypes.byref(sR), ctypes.byref(lR),
                                               P(rates), P(kR)) == 0
                    n += 1; nonzero += int(lR.value >= 0); big += int(np.abs(qR).max() > 127)
                    if not answered(qR, rates, kR):                           # replay: levels, rate tables and constants of the recorded sample
                        continue
                    kO = np.zeros(9, np.int64)
                    assert O.orc_dep_quant_constants(w, h, bd, qp, lam, thr, P(kO)) == 0 and np.array_equal(kO, kR), (w, h, bd, qp, lam, kO, kR)
                    qO = np.zeros((h, w), np.int16); sO = ctypes.c_int32(); lO = ctypes.c_int32()
                    assert O.orc_dep_quant(w, h, bd, qp, lam, thr, zo, lf, 1 - opt, P(rates), P(coef), 1, P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
                    assert np.array_equal(qO, qR) and sO.value == sR.value and lO.value == lR.value, (w, h, bd, qp, lam, scale, mts, lf, sbt, int((qO != qR).sum()))
    assert n == 1050 and nonzero > 500 and (big > 10 or not have_ref()), (n, nonzero, big)      # big reads every level array: the live probe only


@pytest.mark.parametrize("opt", [0, 1])
def test_rdoq_against_the_reference_member(opt):
    """QuantRDOQ2::xRateDistOptQuant (what m_RDOQ == 2 runs for a TU that is not transform skipped) on the probe's TU rig against the restatement fed with the fractional
    bits the reference read from its CABAC contexts: levels, absSum, lastPos for every TU shape class, 8 / 10 bit, QP 17..51, luma / Cb / Cr (Cr with and without a coded
    Cb: last-position table reuse and the coded-block-flag context), sign-bit hiding, LFNST scan limit, SBT bin budget, intra and inter CUs, thrVal 4 / 8 / 16;
    opt 0 = the scalar build of the routine's threshold pre-test, 1 = its SSE form (QuantRDOQ2.cpp:601-637).  Also the per-call constants (error scale)."""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(700 + opt)
    n = 0; nonzero = 0; hidden = 0; zeroed_cg = 0
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (64, 64), (8, 4), (4, 16), (32, 8), (16, 64), (64, 32), (32, 16), (4, 32), (64, 4), (8, 16), (16, 4)]:
        for bd in (10, 8):
            for qp in (17, 22, 27, 32, 37, 42, 51):
                for trial in range(5):
                    lam = float(rs.choice([3.0, 11.7, 30.0, 57.3, 120.0, 800.0, 4000.0]))
                    scale = float(rs.choice([5, 20, 60, 200, 600, 2000, 30000]))
                    dec = float(rs.choice([0.1, 0.5, 1.0, 1.5]))
                    coef = rs.laplace(0, scale, size=(h, w)) * (1.0 / (1 + np.add.outer(np.arange(h), np.arange(w))) ** dec)
                    coef = np.clip(coef, -32768, 32767).astype(np.int32)
                    if w > 32: coef[:, 32:] = 0
                    if h > 32: coef[32:, :] = 0
                    comp = int(rs.choice([0, 0, 1, 2]))
                    lf = int(rs.choice([0, 0, 0, 1, 2]))
                    sbt = int(rs.choice([0, 0, 0, 1])) if (lf == 0 and comp == 0) else 0
                    intra = 1 if lf else (0 if sbt else int(rs.randint(2)))
                    sh = int(rs.randint(2)); cb = int(rs.randint(2)) if comp == 2 else 0
                    thr = int(rs.choice([8, 8, 4, 16]))
                    qR = np.zeros((h, w), np.int16); sR = ctypes.c_int32(); lR = ctypes.c_int32(); rates = np.zeros(190, np.int32); kR = np.zeros(7, np.int32)
                    assert R.refshim_rdoq(comp, P(coef), w, h, bd, qp, intra, lf, sbt, sh, cb, lam, thr, int(rs.randint(17, 52)), trial % 3, P(qR), ctypes.byref(sR), ctypes.byref(lR),
                                          P(rates), P(kR)) == 0
                    n += 1; nonzero += int(lR.value >= 0); hidden += int(sh and lR.value >= 0)
                    if not answered(qR, rates, kR):
                        continue
                    kO = np.zeros(7, np.int32)
                    assert O.orc_rdoq_constants(w, h, bd, qp, int(comp > 0), lf, sbt, thr, P(kO)) == 0 and np.array_equal(kO, kR), (w, h, bd, qp, comp, lf, sbt, kO, kR)
                    qO = np.zeros((h, w), np.int16); sO = ctypes.c_int32(); lO = ctypes.c_int32()
                    assert O.orc_rdoq(w, h, bd, qp, int(comp > 0), lf, sbt, sh, lam, thr, P(rates), P(coef), 1, P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
                    assert np.array_equal(qO, qR) and sO.value == sR.value and lO.value == lR.value, (w, h, bd, qp, comp, lf, sbt, intra, sh, cb, lam, scale, int((qO != qR).sum()))
                    q2 = np.zeros((h, w), np.int16); s2 = ctypes.c_int32(); l2 = ctypes.c_int32()        # the second engine (accumulated templates, cost tables)
                    assert O.orc_rdoq_v2(w, h, bd, qp, int(comp > 0), lf, sbt, sh, lam, thr, P(rates), P(coef), 1, P(q2), ctypes.byref(s2), ctypes.byref(l2)) == 0
                    assert np.array_equal(q2, qR) and s2.value == sR.value and l2.value == lR.value, ('engine 2', w, h, bd, qp, comp, lf, sbt, intra, sh, cb, lam, scale, int((q2 != qR).sum()))
    R.refshim_set_simd(b'AVX2')
    assert n == 1050 and nonzero > 450 and hidden > 150, (n, nonzero, hidden)


@pytest.mark.parametrize("opt", [0, 1])
def test_rdoq_ts_against_the_reference_member(opt):
    """QuantRDOQ::rateDistOptQuantTS (transform-skipped TUs, Quant::m_useRDOQTS) on the probe's TU rig against the restatement fed with the fractional bits of the
    transform-skip context sets the reference read: signed levels and absSum for 12 shapes up to 32 x 32, 8 / 10 bit, QP 2..51 (the QP floor of skipped transforms incl.
    internalMinusInputBitDepth), luma and Cb, dense / laplacian / sparse residuals from 2 to full amplitude (so that the budget of context-coded bins runs out in some
    TUs and all three rate branches are taken); costs are doubles: the comparison is exact"""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(900 + opt)
    n = 0; nonzero = 0; big = 0
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (8, 4), (4, 16), (32, 8), (16, 32), (32, 16), (4, 32), (8, 16), (16, 4)]:
        for bd in (10, 8):
            for qp in (17, 22, 27, 32, 37, 42, 51, 2):
                for trial in range(6):
                    lam = float(rs.choice([3.0, 11.7, 30.0, 57.3, 120.0, 800.0, 4000.0]))
                    amp = int(rs.choice([2, 6, 20, 60, 200, 1023]))
                    kind = trial % 3
                    if kind == 0: resi = rs.randint(-amp, amp + 1, size=(h, w))
                    elif kind == 1: resi = rs.laplace(0, amp / 3.0 + 0.5, size=(h, w)).astype(np.int64)
                    else:
                        resi = rs.randint(-amp, amp + 1, size=(h, w)); resi[rs.rand(h, w) < 0.7] = 0
                    coef = (np.clip(resi, -1023, 1023) << ((5 if bd == 10 else 7) if trial & 1 else 0)).astype(np.int32)     # xTransformSkip copies the residual unscaled; the shifted rows reach large levels
                    comp = int(rs.randint(2)); intra = int(rs.randint(2)); delta = int(rs.choice([0, 0, 2])) if bd == 10 else 0
                    qR = np.zeros((h, w), np.int16); sR = ctypes.c_int32(); rates = np.zeros(44, np.int32); kR = np.zeros(3, np.int32); eR = ctypes.c_double()
                    assert R.refshim_rdoq_ts(comp, P(coef), w, h, bd, qp, delta, intra, lam, int(rs.randint(17, 52)), trial % 3, P(qR), ctypes.byref(sR), P(rates), P(kR), ctypes.byref(eR)) == 0
                    n += 1; nonzero += int(sR.value > 0); big += int(np.abs(qR).max() > 9)
                    if not answered(qR, rates):
                        continue
                    kO = np.zeros(3, np.int32); eO = ctypes.c_double()
                    assert O.orc_rdoq_ts_constants(w, h, bd, qp, delta, P(kO), ctypes.byref(eO)) == 0 and np.array_equal(kO, kR) and eO.value == eR.value, (w, h, bd, qp, delta, kO, kR)
                    qO = np.zeros((h, w), np.int16); sO = ctypes.c_int32()
                    assert O.orc_rdoq_ts(w, h, bd, qp, delta, lam, P(rates), P(coef), 1, P(qO), ctypes.byref(sO)) == 0
                    assert np.array_equal(qO, qR) and sO.value == sR.value, (w, h, bd, qp, comp, intra, delta, lam, amp, kind, int((qO != qR).sum()))
    R.refshim_set_simd(b'AVX2')
    assert n == 1152 and nonzero > 600 and (big > 150 or not have_ref()), (n, nonzero, big)      # big reads every level array: the live probe only


@pytest.mark.parametrize("opt", [0, 1])
def test_rdoq_bdpcm_against_the_reference_member(opt):
    """QuantRDOQ::forwardRDPCM (BDPCM TUs: horizontal and vertical direction) on the probe's TU rig against the restatement: the reconstruction chain (xDequantSample of the
    level just chosen + its prediction), the BDPCM context variants, the member's scanPos-indexed refresh after a zeroed group; same inputs as the transform-skip test"""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    rs = np.random.RandomState(950 + opt)
    n = 0; nonzero = 0
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (8, 4), (4, 16), (32, 8), (16, 32), (32, 16), (4, 32), (8, 16), (16, 4)]:
        for bd in (10, 8):
            for qp in (17, 22, 27, 32, 37, 42, 51, 2):
                for trial in range(6):
                    lam = float(rs.choice([3.0, 11.7, 30.0, 57.3, 120.0, 800.0, 4000.0]))
                    amp = int(rs.choice([2, 6, 20, 60, 200, 1023]))
                    kind = trial % 3
                    if kind == 0: resi = rs.randint(-amp, amp + 1, size=(h, w))
                    elif kind == 1: resi = rs.laplace(0, amp / 3.0 + 0.5, size=(h, w)).astype(np.int64)
                    else:
                        resi = rs.randint(-amp, amp + 1, size=(h, w)); resi[rs.rand(h, w) < 0.7] = 0
                    coef = (np.clip(resi, -1023, 1023) << ((5 if bd == 10 else 7) if trial & 1 else 0)).astype(np.int32)
                    comp = int(rs.randint(2)); delta = int(rs.choice([0, 0, 2])) if bd == 10 else 0; dm = 1 + int(rs.randint(2))
                    qR = np.zeros((h, w), np.int16); sR = ctypes.c_int32(); rates = np.zeros(44, np.int32)
                    assert R.refshim_rdoq_bdpcm(comp, P(coef), w, h, bd, qp, delta, 1, dm, lam, int(rs.randint(17, 52)), trial % 3, P(qR), ctypes.byref(sR), P(rates)) == 0
                    n += 1; nonzero += int(sR.value > 0)
                    if not answered(qR, rates):
                        continue
                    qO = np.zeros((h, w), np.int16); sO = ctypes.c_int32()
                    assert O.orc_rdoq_bdpcm(w, h, bd, qp, delta, dm, lam, P(rates), P(coef), 1, P(qO), ctypes.byref(sO)) == 0
                    assert np.array_equal(qO, qR) and sO.value == sR.value, (w, h, bd, qp, comp, delta, dm, lam, amp, kind, int((qO != qR).sum()))
    R.refshim_set_simd(b'AVX2')
    assert n == 1152 and nonzero > 700, (n, nonzero)


@pytest.mark.parametrize("opt", [0, 1])
def test_transform_skip_and_chroma_against_the_reference(opt):
    """TrQuant::xTransformSkip + Quant::quant with the transform-skip QP (floor 4 + 6 * internalMinusInputBitDepth, no transform shift), Quant::xNeedRDOQ in full
    (dependent-quantisation QP only for non-skipped transforms, the transform shift it keeps for skipped ones, 256 for chroma components), Quant::dequant +
    xITransformSkip: the oracle's restatements against the members on the probe's rig (luma, and Cb on a 4:4:4 rig), with and without sign-bit hiding"""
    import ctypes
    from _libs import oracle, refshim, P
    import cases as C
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    I32 = ctypes.c_int32
    n = 0; nts = 0; ninv = 0
    for row in C.ts_cases():
        w, h, st, bd, amp, qp, irap, sh, dq, ts, delta, comp, seed = [int(v) for v in row]
        resi = C.ts_inputs(row)
        cR = np.zeros((h, w), np.int32); qR = np.zeros((h, w), np.int16); sR = I32(); lR = I32(); nR = I32()
        assert R.refshim_transform_quant_ts(P(resi), st, w, h, bd, qp, irap, sh, dq, ts, delta, comp, P(cR), P(qR), ctypes.byref(sR), ctypes.byref(lR), ctypes.byref(nR)) == 0
        cO = np.zeros((h, w), np.int32); qO = np.zeros((h, w), np.int16); sO = I32(); lO = I32()
        if ts:
            assert O.orc_transform_quant_ts(P(resi), st, w, h, bd, qp, irap, sh, delta, P(cO), P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
        else:
            assert O.orc_transform_quant_ex(0, 0, P(resi), st, w, h, bd, qp, irap, sh, P(cO), P(qO), ctypes.byref(sO), ctypes.byref(lO)) == 0
        assert (not answered(cR, qR) or np.array_equal(cO, cR) and np.array_equal(qO, qR)) and sO.value == sR.value and lO.value == lR.value, [int(v) for v in row]
        assert O.orc_need_rdoq_ex(P(cO), w, h, bd, qp, dq, ts, delta, comp) == nR.value, [int(v) for v in row]
        n += 1; nts += ts
        if ts and sR.value > 0:
            rR = np.zeros((h, st), np.int16); rO = np.zeros((h, st), np.int16); dR = np.zeros((h, w), np.int32); dO = np.zeros((h, w), np.int32)
            assert R.refshim_inv_transform_quant_ts(P(qR), w, h, bd, qp, delta, P(dR), P(rR), st) == 0
            assert O.orc_inv_transform_quant_ts(P(qR), w, h, bd, qp, delta, P(dO), P(rO), st) == 0
            assert not answered(dR, rR) or np.array_equal(dR, dO) and np.array_equal(rR[:, :w], rO[:, :w]), [int(v) for v in row]
            ninv += 1
    assert n == 220 and nts >= 80 and ninv > 40, (n, nts, ninv)


@pytest.mark.parametrize("opt", [0, 1])
def test_dep_quant_chroma_against_the_reference_member(opt):
    """DepQuant::xQuantDQ on the Cb component of a 4:4:4 rig: chroma scan tables (compared with the reference's Rom entry by entry) and chroma rate tables"""
    import ctypes
    from _libs import dq_oracle, refshim, P
    O = dq_oracle(); R = refshim()
    for w in (4, 8, 16, 32, 64):
        for h in (4, 8, 16, 32, 64):
            nc = min(w, 32) * min(h, 32)
            a = np.zeros(nc * 24, np.uint8); b = np.zeros(nc * 16, np.uint8); c = np.zeros(nc * 24, np.uint8); d = np.zeros(nc * 16, np.uint8)
            assert R.refshim_dep_quant_tables_ex(1, w, h, P(a), P(b)) == nc and O.orc_dep_quant_tables_ex(1, w, h, P(c), P(d)) == nc
            assert not answered(a, b) or np.array_equal(a, c) and np.array_equal(b, d), (w, h)
    rs = np.random.RandomState(700 + opt); n = 0; nz = 0
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (8, 4), (4, 16), (32, 8), (16, 32), (64, 64), (16, 4)]:
        for bd in (10, 8):
            for qp in (17, 27, 37, 47):
                for trial in range(5):
                    lam = float(rs.choice([3.0, 11.7, 57.3, 800.0])); scale = float(rs.choice([5, 20, 200, 2000, 30000])); dec = float(rs.choice([0.1, 0.5, 1.0]))
                    coef = rs.laplace(0, scale, size=(h, w)) * (1.0 / (1 + np.add.outer(np.arange(h), np.arange(w))) ** dec)
                    coef = np.clip(coef, -32768, 32767).astype(np.int32)
                    if w > 32: coef[:, 32:] = 0
                    if h > 32: coef[32:, :] = 0
                    q = np.zeros((h, w), np.int16); s = ctypes.c_int32(); l = ctypes.c_int32(); rates = np.zeros(266, np.int32)
                    assert R.refshim_dep_quant_comp(1, P(coef), w, h, bd, qp, 0, int(rs.randint(2)), 0, 0, lam, 8, opt, int(rs.randint(17, 52)), trial % 3, P(q), ctypes.byref(s), ctypes.byref(l), P(rates), None) == 0
                    n += 1; nz += int(l.value >= 0)
                    if not answered(q, rates):
                        continue
                    q2 = np.zeros((h, w), np.int16); s2 = ctypes.c_int32(); l2 = ctypes.c_int32()
                    assert O.orc_dep_quant_chroma(w, h, bd, qp, lam, 8, 0, 1 - opt, P(rates), P(coef), 1, P(q2), ctypes.byref(s2), ctypes.byref(l2)) == 0
                    assert np.array_equal(q, q2) and s.value == s2.value and l.value == l2.value, (w, h, bd, qp, lam, scale)
    assert n == 400 and nz > 150, (n, nz)


@pytest.mark.parametrize("opt", [0, 1])
def test_dep_quant_dequantiser_against_the_reference(opt):
    """DepQuant::dequant -> Quantizer::dequantBlock (state machine over the scan, qIdx at QP + 1) followed by TrQuant::xIT: dequantised coefficients and residual"""
    from _libs import oracle, refshim, P
    import cases as C
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    n = 0
    for row in C.dqd_cases():
        th, tv, w, h, bd, qp, amp, seed = [int(v) for v in row]
        so = np.zeros(1024, np.int32); O.orc_scan_order(w, h, P(so))
        q, last = C.dqd_inputs(row, so)
        cR = np.zeros((h, w), np.int32); rR = np.zeros((h, w), np.int16); cO = np.zeros((h, w), np.int32); rO = np.zeros((h, w), np.int16)
        assert R.refshim_inv_transform_quant_dq(th, tv, P(q), last, w, h, bd, qp, P(cR), P(rR), w) == 0
        assert O.orc_inv_transform_quant_dq(th, tv, P(q), w, h, bd, qp, P(cO), P(rO), w) == 0
        assert not answered(cR, rR) or np.array_equal(cR, cO) and np.array_equal(rR, rO), [int(v) for v in row]
        n += 1
    assert n == 168


@pytest.mark.parametrize("opt", [0, 1])
def test_lfnst_inverse_against_the_reference(opt):
    """TrQuant::invTransformNxN for intra TUs with an LFNST index (dequantiser of either quantiser, xInvLfnst on the first 16 scan positions, xIT over the
    top-left 8x8 / 4x4): the oracle's restatement (the inverse kernel read as the transpose of the forward one) gives the reference's residual for every TU
    shape that can carry LFNST, both indices, intra modes of all four kernel sets with and without transposition, plain and dependent quantisation"""
    from _libs import oracle, refshim, P
    import cases as C
    O = oracle(); R = refshim()
    R.refshim_set_simd(b'AVX2' if opt else b'SCALAR')
    n = 0; sets = set(); nz = 0
    for row in C.ilf_cases():
        w, h, bd, qp, mode, idx, dq, amp, seed = [int(v) for v in row]
        so = np.zeros(1024, np.int32); O.orc_scan_order(w, h, P(so))
        q, last = C.ilf_inputs(row, so)
        cR = np.zeros((h, w), np.int32); rR = np.zeros((h, w), np.int16); st = np.zeros(2, np.int32)
        assert R.refshim_inv_transform_quant_lfnst(P(q), w, h, bd, qp, dq, last, mode, idx, P(cR), P(rR), w, P(st)) == 0
        cO = np.zeros((h, w), np.int32); rO = np.zeros((h, w), np.int16)
        assert O.orc_inv_transform_quant_lfnst(P(q), w, h, bd, qp, dq, int(st[0]), idx, int(st[1]), P(cO), P(rO), w) == 0
        assert not answered(rR) or np.array_equal(rR, rO), [int(v) for v in row]
        k = 8 if (w >= 8 and h >= 8) else 4
        assert not answered(cR) or np.array_equal(cR[:k, :k], cO[:k, :k]), [int(v) for v in row]       # what xIT reads
        sets.add((int(st[0]), int(st[1]))); n += 1; nz += int(rR.any())
    assert n == 288 and len(sets) >= 6 and (nz > 200 or not have_ref()), (n, sets, nz)      # nz reads every residual: the live probe only
