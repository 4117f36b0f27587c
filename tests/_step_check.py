"""Oracle check of the step that bench.py times (bench.Job.run): for the blocks of one level, the dense search, the Hadamard ring around
the best vector and the transform + quantisation of the best residual, computed by the CPU oracle and compared with the device's results.

Everything here takes and returns numpy arrays, so that a test without a GPU can show that each comparison fails when a single value is
wrong (test_bench_step_check.py); test_gpu_bench_step.py runs the same comparisons on what the device returned."""
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from _libs import oracle, PO

UNREACHABLE = 0xFFFFFFFF      # ring cost of a point outside the block's search range (had8_direct_kernel, search_kernels.cuh)
FAMILY_SAD, FAMILY_HAD = 1, 2  # orc_dist families of DF_SAD and DF_HAD

# the comparisons, in the order they are reported: name -> fields of the level dicts that make it up
CHECKS = (('search (dx, dy, cost)', ('dx', 'dy', 'cost')), ('sad', ('sad',)), ('ring', ('ring',)), ('levels', ('q',)),
          ('absSum', ('abs_sum',)), ('lastPos', ('last_pos',)), ('needRdoq', ('need_rdoq',)))


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def ring_blocks_per_group(n, K):
    """blocks per group of had8_direct_kernel (vvb_cost_pattern_dev): at most 512 (block, point, 8x8 tile) items, 32 blocks"""
    return max(1, min(32, 512 // max(1, K * (n // 8) ** 2)))


def tc2_tus_per_tile(n):
    """TUs per tile of fwd_trquant_tc2_kernel (Tc2Shape::TPT): the 128 stage-2 rows hold min(n, 32) rows of each TU"""
    return 128 // min(n, 32)


def _chunked(fn, count, threads, per_thread=8):
    """fn(start, end) over [0, count) in chunks on a thread pool (the oracle's ctypes calls release the GIL); returns fn's results"""
    step = max(1, -(-count // (threads * per_thread)))
    with ThreadPoolExecutor(threads) as ex:
        return list(ex.map(lambda s: fn(s, min(count, s + step)), range(0, count, step)))


def expected_level(org, ref, stride, margin, n, xs, ys, lam, search_range, pattern, bit_depth, qp, threads=None, timing=None, best=None):
    """The oracle's results for the n x n blocks at (xs, ys) of a padded picture pair (predictor 0, cost scale 2, no sub-sampling, DCT-II,
    not IRAP, no DepQuant): dict of dx, dy, cost, sad (at the winning vector), ring [nb][K] (orc_had at best + pattern[k], UNREACHABLE
    outside +-search_range), q [nb][n][n], abs_sum, last_pos, need_rdoq.  best = (dx, dy): no search, ring and TU around these vectors
    (the dict then has no search fields).  timing: optional dict that collects seconds per stage."""
    O = oracle()
    threads = threads or host_threads()
    timing = {} if timing is None else timing
    xs = np.asarray(xs, dtype=np.int32); ys = np.asarray(ys, dtype=np.int32)
    nb, K, R = len(xs), len(pattern), search_range
    base = margin * stride + margin
    po, pr = PO(org, base), PO(ref, base)
    res = {}

    t0 = time.perf_counter()
    if best is None:
        blk = np.zeros((nb, 10), dtype=np.int32)
        blk[:, 0] = xs; blk[:, 1] = ys; blk[:, 2] = n; blk[:, 3] = n; blk[:, 4] = -R; blk[:, 5] = R; blk[:, 6] = -R; blk[:, 7] = R
        out = np.zeros((nb, 4), dtype=np.int32)
        _chunked(lambda s, e: O.orc_full_search(po, stride, pr, stride, PO(blk, 10 * s), e - s, 0, lam, 2, 0, PO(out, 4 * s), None, 0), nb, threads)
        dx, dy = out[:, 0].copy(), out[:, 1].copy()
        cost = out[:, 2].view(np.uint32).astype(np.uint64) | (out[:, 3].view(np.uint32).astype(np.uint64) << np.uint64(32))
        desc = np.stack([xs, ys, xs + dx, ys + dy, np.full(nb, n), np.full(nb, n)], axis=1).astype(np.int32)
        sad = np.zeros(nb, dtype=np.uint64)
        _chunked(lambda s, e: O.orc_dist_list(FAMILY_SAD, po, stride, pr, stride, PO(desc, 6 * s), e - s, 0, PO(sad, s)), nb, threads)
        res.update(dx=dx, dy=dy, cost=cost, sad=sad)
    else:
        dx, dy = (np.asarray(v, dtype=np.int32) for v in best)
    t1 = time.perf_counter()

    pdx = np.array([p[0] for p in pattern], dtype=np.int32); pdy = np.array([p[1] for p in pattern], dtype=np.int32)
    mx = dx[:, None] + pdx[None, :]; my = dy[:, None] + pdy[None, :]
    rdesc = np.zeros((nb, K, 6), dtype=np.int32)
    rdesc[..., 0] = xs[:, None]; rdesc[..., 1] = ys[:, None]; rdesc[..., 2] = xs[:, None] + mx; rdesc[..., 3] = ys[:, None] + my; rdesc[..., 4] = n; rdesc[..., 5] = n
    had = np.zeros(nb * K, dtype=np.uint64)
    _chunked(lambda s, e: O.orc_dist_list(FAMILY_HAD, po, stride, pr, stride, PO(rdesc, 6 * s), e - s, 0, PO(had, s)), nb * K, threads)
    had = had.reshape(nb, K)
    inside = (np.abs(mx) <= R) & (np.abs(my) <= R)
    assert (had[inside] < UNREACHABLE).all()
    ring = np.where(inside, had, UNREACHABLE).astype(np.uint32)
    t2 = time.perf_counter()

    pos = np.stack([xs, ys, dx, dy], axis=1).astype(np.int32)
    q = np.zeros((nb, n, n), dtype=np.int16); asum = np.zeros(nb, dtype=np.int32); last = np.zeros(nb, dtype=np.int32); nr = np.zeros(nb, dtype=np.uint8)
    rcs = _chunked(lambda s, e: O.orc_transform_quant_blocks(0, 0, po, stride, pr, stride, PO(pos, 4 * s), e - s, n, n, bit_depth, qp, 0, 0,
                                                             PO(q, s * n * n), PO(asum, s), PO(last, s), PO(nr, s)), nb, threads)
    assert not any(rcs), rcs
    t3 = time.perf_counter()
    for k, v in (('search', t1 - t0), ('ring', t2 - t1), ('tu', t3 - t2)):
        timing[k] = timing.get(k, 0.0) + v
    res.update(ring=ring, q=q, abs_sum=asum, last_pos=last, need_rdoq=nr)
    return res


def device_level(best, ring, q, abs_sum, last_pos, need_rdoq):
    """the same dict from the device's outputs of a level: best as a BEST_DT array (None: no search), ring [nb][K] costs, q [nb][n][n] levels"""
    d = dict(ring=np.asarray(ring).view(np.uint32), q=q, abs_sum=abs_sum, last_pos=last_pos, need_rdoq=need_rdoq)
    if best is not None:
        d.update(dx=best['dx'].astype(np.int32), dy=best['dy'].astype(np.int32), cost=best['cost'], sad=best['sad'])
    return d


def compare_level(n, xs, ys, exp, got, K, index=None, grids=None):
    """every check of CHECKS on the blocks of one level; returns one message per failing check, naming how many blocks differ and the first
    of them: index in the level, position, ring group or transform tile (with grids = {'ring': ctas, 'tu': ctas}: the CTA and the pass of
    its loop that ran it), expected and got.  index: position of each compared block in the level list (default: all blocks in order)."""
    nb = len(xs)
    index = np.arange(nb) if index is None else np.asarray(index)
    grids = grids or {}
    msgs = []
    for name, fields in CHECKS:
        if any(f not in exp for f in fields):
            continue
        bad = np.zeros(nb, dtype=bool)
        for f in fields:
            e = np.asarray(exp[f]).reshape(nb, -1).astype(np.int64); g = np.asarray(got[f]).reshape(nb, -1).astype(np.int64)
            bad |= (e != g).any(axis=1)
        if not bad.any():
            continue
        where = []
        for i in np.flatnonzero(bad)[:3]:
            j = int(index[i])
            if name == 'ring':
                unit, per = 'ring group', ring_blocks_per_group(n, K)
            elif name in ('search (dx, dy, cost)', 'sad'):
                unit, per = None, 1
            else:
                unit, per = 'tc2 tile', tc2_tus_per_tile(n)
            loc = ''
            if unit:
                u = j // per
                loc = ', %s %d' % (unit, u)
                ctas = grids.get('ring' if name == 'ring' else 'tu')
                if ctas:
                    loc += ' (CTA %d, pass %d)' % (u % ctas, u // ctas)
            diff = []
            for f in fields:
                e = np.asarray(exp[f]).reshape(nb, -1)[i]; g = np.asarray(got[f]).reshape(nb, -1)[i]
                for k in np.flatnonzero(e.astype(np.int64) != g.astype(np.int64))[:2]:
                    diff.append('%s%s expected %d got %d' % (f, '[%d]' % k if e.size > 1 else '', int(e[k]), int(g[k])))
            where.append('block %d at (%d, %d)%s: %s' % (j, int(xs[i]), int(ys[i]), loc, ', '.join(diff)))
        msgs.append('%dx%d %s: %d of %d blocks differ; %s' % (n, n, name, int(bad.sum()), nb, '; '.join(where)))
    return msgs
