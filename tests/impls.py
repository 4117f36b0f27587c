"""Adapters that give the CPU oracle and the live reference probe one calling convention, so the same seeded case
loops (tests/cases.py) drive: oracle-vs-golden, oracle-vs-reference and (tests/test_gpu_*.py) CUDA-vs-oracle."""
import ctypes
import numpy as np
import cases as C
from _libs import answered, oracle, refshim, P, PO

I32 = ctypes.c_int32


class OracleImpl:
    name = 'oracle'

    def __init__(self):
        self.L = oracle()

    def dist(self, fam, o, so, c, sc, w, h, bd, ss):
        return int(self.L.orc_dist(fam, P(o), so, P(c), sc, w, h, ss))

    def transform_quant(self, th, tv, resi, st, w, h, bd, qp, irap, dq=0):
        coef = np.zeros((h, w), dtype=np.int32); q = np.zeros((h, w), dtype=np.int16); s = I32(); lp = I32()
        assert self.L.orc_transform_quant(th, tv, P(resi), st, w, h, bd, qp, irap, P(coef), P(q), ctypes.byref(s), ctypes.byref(lp)) == 0
        return coef, q, s.value, lp.value, self.need_rdoq(coef, w, h, bd, qp, dq)

    def need_rdoq(self, coef, w, h, bd, qp, dq):
        return int(self.L.orc_need_rdoq(P(coef), w, h, bd, qp, dq))

    def inv_transform_quant(self, th, tv, q, w, h, bd, qp, stride):
        """-> (dequantised coefficients int32 [h][w], residual int16 [h][w])"""
        coef = np.zeros((h, w), dtype=np.int32); resi = np.zeros((h, stride), dtype=np.int16)
        assert self.L.orc_inv_transform_quant(th, tv, P(q), w, h, bd, qp, P(coef), P(resi), stride) == 0
        return coef, np.ascontiguousarray(resi[:, :w])

    def tu_roundtrip(self, th, tv, org, so, pred, ps, w, h, bd, qp, irap):
        """-> (levels [h][w], reco [h][w], [dist_reco, dist_resi, dist_zero, abs_sum, last_pos])"""
        q = np.zeros((h, w), dtype=np.int16); reco = np.zeros((h, w), dtype=np.int16); o4 = np.zeros(4, dtype=np.uint64)
        assert self.L.orc_tu_roundtrip(th, tv, P(org), so, P(pred), ps, w, h, bd, qp, irap, P(q), P(reco), w, P(o4)) == 0
        return q, reco, [int(o4[0]), int(o4[1]), int(o4[2]), int(o4[3]) & 0xffffffff, np.int32(np.uint32(int(o4[3]) >> 32)).item()]

    def mctf_err(self, tap4, org, so, buf, sb, x, y, mvx, mvy, w, h, bd):
        desc = np.array([[x, y, mvx, mvy, w, h]], dtype=np.int32); out = np.zeros(1, dtype=np.int32)
        self.L.orc_mctf_err_list(tap4, PO(org, -(y * so + x)), so, P(buf), sb, P(desc), 1, bd, P(out))
        return int(out[0])

    def sobel(self, vert, pred, ps, ds, w, h):
        d = np.zeros((h, ds), dtype=np.int16)
        self.L.orc_sobel(vert, P(pred), ps, P(d), ds, w, h)
        return d

    def equal_coeff(self, six, resi, rs, gx, gy, ds, w, h):
        e = np.zeros(49, dtype=np.int64)
        self.L.orc_equal_coeff(six, P(resi), rs, P(gx), P(gy), ds, w, h, P(e))
        return e

    def full_search(self, sc, ss, want_table=False):
        n = len(sc['blk']); S = sc['stride']; base = sc['margin'] * S + sc['margin']
        out = np.zeros((n, 4), dtype=np.int32)
        ts = int(max((b[5] - b[4] + 1) * (b[7] - b[6] + 1) for b in sc['blk']))
        tab = np.zeros((n, ts), dtype=np.uint32) if want_table else None
        self.L.orc_full_search(PO(sc['org'], base), S, PO(sc['ref'], base), S, P(sc['blk']), n, ss, sc['lam'], sc['cost_scale'], sc['imv_shift'],
                               P(out), P(tab) if want_table else None, ts)
        return (out, tab) if want_table else out

    def mv_bits(self, *a):
        return int(self.L.orc_mv_bits(*a))

    def mv_cost(self, lam, *a):
        return int(self.L.orc_mv_cost(lam, *a))


class RefImpl(OracleImpl):
    """the unmodified reference through oracle/_ref (opt=1: SIMD table, opt=0: scalar table)"""

    def __init__(self, opt=1, simd=b'AVX2'):
        self.L = refshim(); self.opt = opt; self.simd = simd
        self.name = 'reference-%s' % (simd.decode() if opt else 'scalar')

    def _simd(self):
        self.L.refshim_set_simd(self.simd if self.opt else b'SCALAR')

    def dist(self, fam, o, so, c, sc, w, h, bd, ss):
        return int(self.L.refshim_dist(self.opt, fam, P(o), so, P(c), sc, w, h, bd, ss))

    def transform_quant(self, th, tv, resi, st, w, h, bd, qp, irap, dq=0):
        self._simd()
        coef = np.zeros((h, w), dtype=np.int32); q = np.zeros((h, w), dtype=np.int16); s = I32(); lp = I32()
        assert self.L.refshim_transform_quant(th, tv, P(resi), st, w, h, bd, qp, irap, P(coef), P(q), ctypes.byref(s), ctypes.byref(lp)) == 0
        return coef, q, s.value, lp.value, self.need_rdoq(coef, w, h, bd, qp, dq)

    def need_rdoq(self, coef, w, h, bd, qp, dq):
        self._simd()
        return int(self.L.refshim_need_rdoq(P(coef), w, h, bd, qp, dq))

    def inv_transform_quant(self, th, tv, q, w, h, bd, qp, stride):
        self._simd()
        coef = np.zeros((h, w), dtype=np.int32); resi = np.zeros((h, stride), dtype=np.int16)
        assert self.L.refshim_inv_transform_quant(th, tv, P(q), w, h, bd, qp, P(coef), P(resi), stride) == 0
        return coef, np.ascontiguousarray(resi[:, :w])

    def tu_roundtrip(self, th, tv, org, so, pred, ps, w, h, bd, qp, irap):
        self._simd()
        q = np.zeros((h, w), dtype=np.int16); reco = np.zeros((h, w), dtype=np.int16); o4 = np.zeros(4, dtype=np.uint64)
        assert self.L.refshim_tu_roundtrip(self.opt, th, tv, P(org), so, P(pred), ps, w, h, bd, qp, irap, P(q), P(reco), w, P(o4)) == 0
        return q, reco, [int(o4[0]), int(o4[1]), int(o4[2]), int(o4[3]) & 0xffffffff, np.int32(np.uint32(int(o4[3]) >> 32)).item()]

    def mctf_err(self, tap4, org, so, buf, sb, x, y, mvx, mvy, w, h, bd):
        desc = np.array([[x, y, mvx, mvy, w, h]], dtype=np.int32); out = np.zeros(1, dtype=np.int32)
        self.L.refshim_mctf_err_list(self.opt, tap4, PO(org, -(y * so + x)), so, P(buf), sb, P(desc), 1, bd, P(out), 1)
        return int(out[0])

    def sobel(self, vert, pred, ps, ds, w, h):
        d = np.zeros((h, ds), dtype=np.int16)
        self.L.refshim_sobel(self.opt, vert, P(pred), ps, P(d), ds, w, h)
        return d

    def equal_coeff(self, six, resi, rs, gx, gy, ds, w, h):
        e = np.zeros(49, dtype=np.int64)
        self.L.refshim_equal_coeff(self.opt, six, P(resi), rs, P(gx), P(gy), ds, w, h, P(e))
        return e

    def full_search(self, sc, ss, want_table=False):
        n = len(sc['blk']); S = sc['stride']; base = sc['margin'] * S + sc['margin']
        out = np.zeros((n, 4), dtype=np.int32)
        ts = int(max((b[5] - b[4] + 1) * (b[7] - b[6] + 1) for b in sc['blk']))
        tab = np.zeros((n, ts), dtype=np.uint32) if want_table else None
        self.L.refshim_full_search(self.opt, PO(sc['org'], base), S, PO(sc['ref'], base), S, P(sc['blk']), n, 10, ss, sc['lam'], sc['cost_scale'],
                                   sc['imv_shift'], P(out), P(tab) if want_table else None, ts, 2, 0)
        return (out, tab) if want_table else out

    def mv_bits(self, *a):
        return int(self.L.refshim_mv_bits(*a))

    def mv_cost(self, lam, *a):
        return int(self.L.refshim_mv_cost(lam, *a))


# ---------------------------------------------------------------------------------------------------------------
# case loops: each returns a list of mismatch descriptions (empty == parity)

def run_dist(impl, rows, expect):
    bad = []
    for row, e in zip(rows, expect):
        fam, w, h, so, sc, ss, ko, kc, bd, seed = [int(v) for v in row]
        o, c = C.dist_inputs(row)
        g = impl.dist(fam, o, so, c, sc, w, h, bd, ss)
        if g != int(e):
            bad.append(('dist', row.tolist(), g, int(e)))
    return bad


def run_tq(impl, rows, coef, q, meta):
    bad = []; off = 0
    for i, row in enumerate(rows):
        th, tv, w, h, st, amp, qp, irap, bd, seed = [int(v) for v in row]
        resi = C.tq_inputs(row)
        c, qq, s, lp, nr = impl.transform_quant(th, tv, resi, st, w, h, bd, qp, irap, seed & 1)
        ec = coef[off:off + w * h].reshape(h, w); eq = q[off:off + w * h].reshape(h, w); off += w * h
        if not (np.array_equal(c, ec) and np.array_equal(qq, eq) and s == meta[i][0] and lp == meta[i][1] and nr == meta[i][2]):
            bad.append(('tq', row.tolist(), bool(np.array_equal(c, ec)), bool(np.array_equal(qq, eq)), s, lp, nr, meta[i].tolist()))
    return bad


def run_itq(impl, rows, coef, resi):
    """inverse path: dequantised coefficients (where the implementation exposes them) and the residual"""
    bad = []; off = 0
    for row in rows:
        th, tv, w, h, st, kind, qp, bd, seed = [int(v) for v in row]
        q = C.itq_inputs(row)
        c, r = impl.inv_transform_quant(th, tv, q, w, h, bd, qp, st)
        ec = coef[off:off + w * h].reshape(h, w); er = resi[off:off + w * h].reshape(h, w); off += w * h
        if not ((c is None or np.array_equal(c, ec)) and np.array_equal(r, er)):
            bad.append(('itq', row.tolist(), c is None or bool(np.array_equal(c, ec)), bool(np.array_equal(r, er))))
    return bad


def run_rt(impl, rows, q, reco, meta):
    bad = []; off = 0
    for i, row in enumerate(rows):
        th, tv, w, h, so, ps, amp, qp, irap, bd, seed = [int(v) for v in row]
        org, pred = C.rt_inputs(row)
        gq, gr, gm = impl.tu_roundtrip(th, tv, org, so, pred, ps, w, h, bd, qp, irap)
        eq = q[off:off + w * h].reshape(h, w); er = reco[off:off + w * h].reshape(h, w); off += w * h
        if not (np.array_equal(gq, eq) and np.array_equal(gr, er) and [int(v) for v in gm] == [int(v) for v in meta[i]]):
            bad.append(('rt', row.tolist(), bool(np.array_equal(gq, eq)), bool(np.array_equal(gr, er)), gm, meta[i].tolist()))
    return bad


def mctf_apply_expected(L, prefix, case, tap4, planar, opt=None, known=None):
    """filtered picture [H][W] through the oracle (prefix 'orc') or the reference probe (prefix 'refshim', opt = 0/1), block by block;
    `known` (bool [H][W]) is cleared over the blocks whose reference values a replayed probe could not give (see _libs.answered)"""
    S = case['stride']; m = case['margin']; W = case['W']; H = case['H']; bs = case['bs']; base = m * S + m
    out = np.zeros((H, W), dtype=np.int16)
    n = case['num_refs']
    ptrs = (ctypes.c_void_p * n)(*[r.ctypes.data + base * 2 for r in case['refs']])
    bxn = (W + bs - 1) // bs
    for by in range(0, H, bs):
        for bx in range(0, W, bs):
            b = (by // bs) * bxn + bx // bs
            w = min(bs, W - bx); h = min(bs, H - by)
            mv4 = np.ascontiguousarray(case['mvs'][:, b, :])
            if prefix == 'orc':
                L.orc_mctf_finalize_block(PO(case['org'], base), S, ptrs, S, n, P(mv4), bx, by, w, h, case['bd'], tap4, planar, P(case['strengths']),
                                          ctypes.c_double(case['ws']), ctypes.c_double(case['sigma']), P(out), W)
            else:
                L.refshim_mctf_finalize_block(opt, PO(case['org'], base), S, ptrs, S, n, P(mv4), W, H, bx, by, w, h, case['bd'], tap4, planar, P(case['strengths']),
                                              ctypes.c_double(case['ws']), ctypes.c_double(case['sigma']), P(out), W)
                if known is not None and not answered(out):
                    known[by:by + h, bx:bx + w] = False
    return out


def run_mctf(impl, rows, expect):
    bad = []
    m = C.MCTF_MARGIN
    for row, e in zip(rows, expect):
        w, h, mvx, mvy, tap4, bd, seed = [int(v) for v in row]
        org, buf = C.mctf_inputs(row)
        g = impl.mctf_err(tap4, org, org.shape[1], buf, buf.shape[1], m, m, mvx, mvy, w, h, bd)
        if g != int(e):
            bad.append(('mctf', row.tolist(), g, int(e)))
    return bad


def run_affine(impl, rows, sobel, eqs):
    bad = []; off = 0
    for i, row in enumerate(rows):
        w, h, ps, ds, six, seed = [int(v) for v in row]
        pred, resi, gx, gy = C.affine_inputs(row)
        for vert in (0, 1):
            d = impl.sobel(vert, pred, ps, ds, w, h)[:, :w]
            e = sobel[off:off + w * h].reshape(h, w); off += w * h
            if not np.array_equal(d, e):
                bad.append(('sobel', row.tolist(), vert))
        g = impl.equal_coeff(six, resi, ps, gx, gy, ds, w, h)
        if not np.array_equal(g, eqs[i]):
            bad.append(('equal_coeff', row.tolist()))
    return bad


class GpuImpl:
    """the CUDA product through its C ABI (vvenc_b200.CostEngine); same calling convention as OracleImpl"""
    name = 'gpu'

    def __init__(self, device=0):
        import vvenc_b200 as V
        self.V = V
        self.eng = V.CostEngine(device)

    def dist(self, fam, o, so, c, sc, w, h, bd, ss):
        return self.eng.dist_block(fam, o, so, c, sc, w, h, bd, ss)

    def transform_quant(self, th, tv, resi, st, w, h, bd, qp, irap, dq=0):
        par = self.eng.tu_par(w, h, th, tv, bd, qp, bool(irap), bool(dq))
        r = self.eng.fwd_trquant(par, np.ascontiguousarray(resi[:, :w]).reshape(1, h, w))
        return r['coef'][0], r['q'][0], int(r['abs_sum'][0]), int(r['last_pos'][0]), int(r['need_rdoq'][0])

    def inv_transform_quant(self, th, tv, q, w, h, bd, qp, stride):
        par = self.eng.tu_par(w, h, th, tv, bd, qp, False, False)
        return None, self.eng.inv_trquant(par, q.reshape(1, h, w))[0]

    def tu_roundtrip(self, th, tv, org, so, pred, ps, w, h, bd, qp, irap):
        par = self.eng.tu_par(w, h, th, tv, bd, qp, bool(irap), False)
        r = self.eng.tu_roundtrip(par, np.ascontiguousarray(org[:, :w]).reshape(1, h, w), np.ascontiguousarray(pred[:, :w]).reshape(1, h, w))
        x = r['res'][0]
        return r['q'][0], r['reco'][0], [int(x['dist_reco']), int(x['dist_resi']), int(x['dist_zero']), int(x['abs_sum']), int(x['last_pos'])]

    def mctf_err(self, tap4, org, so, buf, sb, x, y, mvx, mvy, w, h, bd):
        m = min(x, y)
        orgp = np.zeros_like(buf)
        orgp[y:y + h, x:x + w] = org[:h, :w]
        self.eng.upload_plane(0, np.ascontiguousarray(orgp), buf.shape[1] - 2 * m, buf.shape[0] - 2 * m, m, bd)
        self.eng.upload_plane(1, np.ascontiguousarray(buf), buf.shape[1] - 2 * m, buf.shape[0] - 2 * m, m, bd)
        c = np.zeros(1, dtype=self.V.MCTF_DT)
        c['x'] = x - m; c['y'] = y - m; c['mvx'] = mvx; c['mvy'] = mvy; c['w'] = w; c['h'] = h
        return int(self.eng.mctf_error_batch(0, 1, c, bool(tap4))[0])

    def sobel(self, vert, pred, ps, ds, w, h):
        return self.eng.affine_sobel(vert, pred, ps, ds, w, h)

    def equal_coeff(self, six, resi, rs, gx, gy, ds, w, h):
        return self.eng.affine_equal_coeff(six, resi, rs, gx, gy, ds, w, h)

    def upload_search_case(self, sc):
        m = sc['margin']
        self.eng.upload_plane(0, sc['org'], sc['W'], sc['H'], m, 10)
        self.eng.upload_plane(1, sc['ref'], sc['W'], sc['H'], m, 10)

    def full_search(self, sc, ss, want_table=False):
        self.upload_search_case(sc)
        blk = sc['blk']; n = len(blk)
        out = np.zeros((n, 4), dtype=np.int32)
        ts = int(max((b[5] - b[4] + 1) * (b[7] - b[6] + 1) for b in blk))
        tab = np.zeros((n, ts), dtype=np.uint32)
        par = self.eng.me_par(sc['lam'], sc['cost_scale'], sc['imv_shift'], ss)
        # one launch per distinct block shape (the C ABI takes uniform-shape batches)
        shapes = sorted(set((int(b[2]), int(b[3])) for b in blk))
        for (w, h) in shapes:
            idx = [i for i in range(n) if (int(blk[i][2]), int(blk[i][3])) == (w, h)]
            B = np.zeros(len(idx), dtype=self.V.BLOCK_DT)
            for k, i in enumerate(idx):
                b = blk[i]
                B[k] = (b[0], b[1], b[4], b[5], b[6], b[7], b[8], b[9], 0, 0)
            best, t = self.eng.sad_search(0, 1, B, w, h, par, want_tables=True)
            for k, i in enumerate(idx):
                out[i] = (best[k]['dx'], best[k]['dy'], int(best[k]['cost']) & 0xffffffff, int(best[k]['cost']) >> 32)
                tab[i, :t.shape[1]] = t[k]
        return (out, tab) if want_table else out
