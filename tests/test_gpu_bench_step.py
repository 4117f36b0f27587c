"""The step bench.py times (bench.Job.run: SAD pyramid at +-32 over 8/16/32/64 blocks, the 18-point Hadamard ring around each best vector,
DCT-II + quantisation of the best residual at QP 32) at the size it is timed, 3840x2160 10-bit, against the CPU oracle for every block of
the four levels (-m gpu).

At this size the persistent kernels of the step loop: fwd_trquant_tc2_kernel takes several tiles per CTA and had8_direct_kernel several
block groups, which no smaller oracle comparison reaches; the picture height leaves a row of parentless 32x32 and one of 16x16 roots.  The
other search engines, the window staging without TMA, the CUDA-core transform and the one-call chain (vvb_search_refine_tu) must give the
same outputs on the device.  A 7680x4320 picture (BASELINE configs[4]) is compared on its bottom root row, its right-hand root column and a
seeded sample.  The comparisons themselves are tests/_step_check.py; test_bench_step_check.py shows without a GPU that they fail."""
import ctypes
import json
import math
import os
import re
import tempfile
import time

import numpy as np
import pytest

import bench
import _step_check as SC
from vvenc_b200.candidates import pyramid_lists

pytestmark = pytest.mark.gpu

SIZES = bench.SIZES
PATTERN = bench.refine_pattern()
K = len(PATTERN)
P_ = ctypes.c_void_p


def _env(torch, V, eng):
    """the env dict of bench.main (bench.py:692-707), without the entries of the multi-rank legs, which Job.run does not read"""
    lib = eng.lib
    pat_np = np.zeros(K, dtype=V.MV_DT)
    pat_np['dx'] = [p[0] for p in PATTERN]; pat_np['dy'] = [p[1] for p in PATTERN]

    def dev(a):
        return torch.from_numpy(np.frombuffer(a.tobytes(), dtype=np.uint8).copy()).cuda()

    def chk(rc):
        if rc != 0:
            raise RuntimeError('vvenc_b200: ' + lib.vvb_last_error(eng.h).decode())
    return {'torch': torch, 'V': V, 'eng': eng, 'lib': lib, 'chk': chk, 'me': eng.me_par(bench.LAMBDA, 2, 0, 0, 1, 2), 'nx': 2 * bench.SEARCH_RANGE + 1,
            'dev': dev, 'KP': K, 'd_pat': dev(pat_np), 'pat_np': pat_np,
            'tu_par': {n: eng.tu_par(n, n, V.DCT2, V.DCT2, bench.BITDEPTH, bench.QP, False, False) for n in SIZES}}


def _bind(torch, eng, org, ref, S, w, h, ids):
    """the picture pair as bench.main binds it (bench.py:717-721); returns the device planes, which must outlive their use"""
    dorg = torch.from_numpy(org).cuda(); dref = torch.from_numpy(ref).cuda()
    base = (bench.MARGIN * S + bench.MARGIN) * 2
    eng.bind_plane_dev(ids[0], dorg.data_ptr() + base, S, w, h, bench.MARGIN, bench.BITDEPTH)
    eng.bind_plane_dev(ids[1], dref.data_ptr() + base, S, w, h, bench.MARGIN, bench.BITDEPTH)
    torch.cuda.synchronize()
    return dorg, dref


def _run(step, job, planes=(0, 1), direct=False):
    """one Job.run, synchronised; returns every output of every level as numpy arrays"""
    torch, V, eng, env = step['torch'], step['V'], step['eng'], step['env']
    job.run(env, planes[0], planes[1], direct)
    eng.synchronize(); torch.cuda.synchronize()
    out = {}
    for n in SIZES:
        nb = job.counts[n]
        out[n] = dict(best=np.frombuffer(job.d_best[n][:nb * 16].cpu().numpy().tobytes(), dtype=V.BEST_DT),
                      ring=job.d_satd[n][:nb * K].cpu().numpy().view(np.uint32).reshape(nb, K),
                      q=job.d_q[n][:nb * n * n].cpu().numpy().reshape(nb, n, n), abs_sum=job.d_sum[n][:nb].cpu().numpy(),
                      last_pos=job.d_last[n][:nb].cpu().numpy(), need_rdoq=job.d_nr[n][:nb].cpu().numpy())
    return out


def _device_level(o, index=slice(None)):
    return SC.device_level(o['best'][index], o['ring'][index], o['q'][index], o['abs_sum'][index], o['last_pos'][index], o['need_rdoq'][index])


def _first_difference(a, b):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    if a.dtype.names:
        a = a.view(np.uint8).reshape(len(a), -1); b = b.view(np.uint8).reshape(len(b), -1)
    if a.shape != b.shape:
        return 'shape %s vs %s' % (a.shape, b.shape)
    bad = np.flatnonzero((a.reshape(len(a), -1) != b.reshape(len(b), -1)).any(axis=1))
    return None if len(bad) == 0 else '%d blocks differ, first %d' % (len(bad), bad[0])


@pytest.fixture(scope='module')
def step():
    import torch
    import vvenc_b200 as V
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    eng = V.CostEngine(0)
    env = _env(torch, V, eng)
    org, ref, S = bench.synth_picture_pair(1234)                  # picture set 0 of bench.main
    planes = _bind(torch, eng, org, ref, S, bench.W, bench.H, (0, 1))
    job = bench.Job(env, bench.W, pyramid_lists(SIZES[0], len(SIZES), bench.W, bench.H), 'test')
    torch.cuda.synchronize()
    st = dict(torch=torch, V=V, eng=eng, env=env, org=org, ref=ref, S=S, planes=planes, job=job, grids={})
    st['out'] = _run(st, job)
    yield st
    eng.synchronize()
    eng.close()


def test_gpu_bench_step_persistent_launches_loop(step):
    """precondition of the comparisons below: at 2160p every ring launch has more block groups, and every tensor-core TU launch more tiles,
    than CTAs, so that the CTAs run their loops.  The grids are read from a profile of one step and bounded by the SM count."""
    from torch.profiler import profile, ProfilerActivity
    torch, job = step['torch'], step['job']
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _run(step, job)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'step.json')
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)['traceEvents']
    kernels = sorted((e for e in events if e.get('cat') == 'kernel'), key=lambda e: e['ts'])
    ring = [e['args']['grid'][0] for e in kernels if 'had8_direct_kernel' in e['name']]
    tc2 = {}
    for e in kernels:
        m = re.search(r'fwd_trquant_tc2_kernel<(\d+), ?1>', e['name'])
        if m:
            tc2[int(m.group(1))] = e['args']['grid'][0]
    assert len(ring) == len(SIZES) and sorted(tc2) == list(SIZES), ([e['name'] for e in kernels], ring, tc2)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for n, ring_grid in zip(SIZES, ring):
        nb = job.counts[n]
        groups = math.ceil(nb / SC.ring_blocks_per_group(n, K)); tiles = math.ceil(nb / SC.tc2_tus_per_tile(n))
        print('%dx%d: %d blocks; ring %d groups on %d CTAs; tc2 %d tiles on %d CTAs (%d SMs)' % (n, n, nb, groups, ring_grid, tiles, tc2[n], sms))
        assert ring_grid <= 8 * sms and groups > ring_grid, (n, groups, ring_grid)
        assert tc2[n] <= 8 * sms and tiles > tc2[n], (n, tiles, tc2[n])
        step['grids'][n] = {'ring': ring_grid, 'tu': tc2[n]}


def test_gpu_bench_step_2160p_every_block_vs_oracle(step):
    """every block of the four levels: (dx, dy, cost) == orc_full_search (predictor 0, +-32, lambda 57.9, cost scale 2), sad == orc_sad at the
    winning vector, the 18 ring costs == orc_had at best + pattern[k], levels / absSum / lastPos / needRdoq == orc_transform_quant + orc_need_rdoq"""
    job, timing, msgs = step['job'], {}, []
    t0 = time.perf_counter()
    # the picture's edge: 2160 = 33 * 64 + 48 leaves a row of parentless 32x32 roots at y = 2112 and of 16x16 roots at y = 2144
    assert job.counts == {8: 129600, 16: 32400, 32: 8040, 64: 1980}
    for n in SIZES:
        b = job.blocks_np[n]
        exp = SC.expected_level(step['org'], step['ref'], step['S'], bench.MARGIN, n, b['x'], b['y'], bench.LAMBDA, bench.SEARCH_RANGE, PATTERN,
                                bench.BITDEPTH, bench.QP, timing=timing)
        msgs += SC.compare_level(n, b['x'], b['y'], exp, _device_level(step['out'][n]), K, grids=step['grids'].get(n))
    print('oracle on %d host threads: %.1f s (search %.1f s, ring %.1f s, TU %.1f s); blocks compared per level and check: %s'
          % (SC.host_threads(), time.perf_counter() - t0, timing['search'], timing['ring'], timing['tu'], job.counts))
    assert msgs == [], '\n'.join(msgs)


def test_gpu_bench_step_ring_and_tu_at_spread_vectors_vs_oracle(step):
    """the ring and TU stages of the step on the same blocks with seeded start vectors across the window (half of the blocks keep their best
    vector).  bench.py's pictures quantise to all-zero levels at QP 32; at these vectors the residuals give zero and non-zero levels, both
    RDOQ pre-check decisions and ring points outside the window (cost 0xFFFFFFFF)"""
    torch, V, eng, env, job = step['torch'], step['V'], step['eng'], step['env'], step['job']
    lib, chk, R = env['lib'], env['chk'], bench.SEARCH_RANGE
    rs = np.random.RandomState(2160)
    msgs, seen = [], {'nonzero': 0, 'zero': 0, 'rdoq': 0, 'unreachable': 0}
    t0 = time.perf_counter()
    for n in SIZES:
        nb = job.counts[n]
        b = job.blocks_np[n].copy()
        best = step['out'][n]['best']
        spread = rs.rand(nb) < 0.5
        b['start_x'] = np.where(spread, rs.randint(-R, R + 1, nb), best['dx']); b['start_y'] = np.where(spread, rs.randint(-R, R + 1, nb), best['dy'])
        d_b = env['dev'](b)
        ring = torch.empty(nb * K, dtype=torch.int32, device='cuda'); q = torch.empty(nb * n * n, dtype=torch.int16, device='cuda')
        s = torch.empty(nb, dtype=torch.int32, device='cuda'); last = torch.empty(nb, dtype=torch.int32, device='cuda'); nr = torch.empty(nb, dtype=torch.uint8, device='cuda')
        torch.cuda.synchronize()
        chk(lib.vvb_cost_pattern_dev(eng.h, V.DF_HAD, 0, 1, P_(d_b.data_ptr()), nb, n, n, P_(env['d_pat'].data_ptr()), K, ctypes.byref(env['me']), P_(ring.data_ptr()), None))
        chk(lib.vvb_fwd_trquant_planes_dev(eng.h, ctypes.byref(env['tu_par'][n]), 0, 1, P_(d_b.data_ptr()), nb, None, P_(q.data_ptr()), P_(s.data_ptr()),
                                           P_(last.data_ptr()), P_(nr.data_ptr())))
        eng.synchronize(); torch.cuda.synchronize()
        got = SC.device_level(None, ring.cpu().numpy().reshape(nb, K), q.cpu().numpy().reshape(nb, n, n), s.cpu().numpy(), last.cpu().numpy(), nr.cpu().numpy())
        exp = SC.expected_level(step['org'], step['ref'], step['S'], bench.MARGIN, n, b['x'], b['y'], bench.LAMBDA, R, PATTERN, bench.BITDEPTH, bench.QP,
                                best=(b['start_x'], b['start_y']))
        msgs += SC.compare_level(n, b['x'], b['y'], exp, got, K, grids=step['grids'].get(n))
        seen['nonzero'] += int((exp['abs_sum'] > 0).sum()); seen['zero'] += int((exp['abs_sum'] == 0).sum())
        seen['rdoq'] += int(exp['need_rdoq'].sum()); seen['unreachable'] += int((exp['ring'] == SC.UNREACHABLE).any(axis=1).sum())
    print('spread vectors: %s blocks of %d; oracle %.1f s' % (seen, sum(job.counts.values()), time.perf_counter() - t0))
    assert msgs == [], '\n'.join(msgs)
    assert seen['nonzero'] and seen['zero'] and seen['rdoq'] and seen['unreachable'], seen


def test_gpu_bench_step_engines_agree(step):
    """at full size on the device: the per-size direct search (bench.py's direct_search row), the per-quad pyramid engine, the window staging
    without TMA and the CUDA-core transform give the resident step's outputs, every field of every block"""
    eng, job, ref = step['eng'], step['job'], step['out']
    variants = (('direct search', dict(direct=True)), ('direct search, TMA staging 0', dict(direct=True, tma=0)),
                ('pyramid engine 0', dict(pyramid=0)), ('pyramid engine 0, TMA staging 0', dict(pyramid=0, tma=0)),
                ('tensor transform 0', dict(tensor=0)))
    bad = []
    for name, v in variants:
        eng.set_pyramid_engine(v.get('pyramid', 1)); eng.set_tma_staging(v.get('tma', 2)); eng.set_tensor_transform(v.get('tensor', 3))
        try:
            got = _run(step, job, direct=v.get('direct', False))
        finally:
            eng.set_pyramid_engine(1); eng.set_tma_staging(2); eng.set_tensor_transform(3)
        for n in SIZES:
            for field in ref[n]:
                d = _first_difference(got[n][field], ref[n][field])
                if d:
                    bad.append('%s, %dx%d %s: %s' % (name, n, n, field, d))
    assert bad == [], '\n'.join(bad)


def test_gpu_bench_step_chain_call_equals_resident(step):
    """vvb_search_refine_tu (one host call: search -> ring -> TU, asynchronous, levels also packed to lastPos) on the same picture and blocks
    returns the resident step's outputs"""
    import vvenc_b200._lib as VL
    V, eng, env, job, ref = step['V'], step['eng'], step['env'], step['job'], step['out']
    io = (VL.vvb_level_io * len(SIZES))(); keep = []
    for l, n in enumerate(SIZES):
        nb = job.counts[n]
        o = dict(blk=np.ascontiguousarray(job.blocks_np[n]), best=np.zeros(nb, dtype=V.BEST_DT), ring=np.zeros((nb, K), dtype=np.uint32),
                 q=np.zeros((nb, n, n), dtype=np.int16), abs_sum=np.zeros(nb, dtype=np.int32), last_pos=np.zeros(nb, dtype=np.int32),
                 need_rdoq=np.zeros(nb, dtype=np.uint8), pq=np.zeros(nb * n * n, dtype=np.int16), off=np.zeros(nb + 1, dtype=np.int32))
        keep.append(o)
        io[l].blocks = o['blk'].ctypes.data; io[l].count = nb; io[l].best = o['best'].ctypes.data; io[l].refine_cost = o['ring'].ctypes.data
        io[l].q = o['q'].ctypes.data; io[l].abs_sum = o['abs_sum'].ctypes.data; io[l].last_pos = o['last_pos'].ctypes.data; io[l].need_rdoq = o['need_rdoq'].ctypes.data
        io[l].packed_q = o['pq'].ctypes.data; io[l].packed_offsets = o['off'].ctypes.data
        io[l].tu = env['tu_par'][n]
    eng.set_async(True)
    try:
        rc = eng.lib.vvb_search_refine_tu(eng.h, 0, 1, len(SIZES), io, SIZES[0], ctypes.byref(env['me']), env['nx'], env['nx'], V.DF_HAD,
                                          env['pat_np'].ctypes.data_as(P_), K)
        assert rc == 0, eng.lib.vvb_last_error(eng.h)
        eng.synchronize()
    finally:
        eng.set_async(False)
    bad = []
    for o, n in zip(keep, SIZES):
        nb = job.counts[n]
        for field in ref[n]:
            d = _first_difference(o[field], ref[n][field])
            if d:
                bad.append('%dx%d %s: %s' % (n, n, field, d))
        so = np.zeros(min(n, 32) ** 2, dtype=np.int32)
        assert eng.lib.vvb_scan_order(n, n, so.ctypes.data_as(P_)) == 0
        off = o['off'].astype(np.int64); lens = np.maximum(o['last_pos'].astype(np.int64) + 1, 0)
        assert off[0] == 0 and np.array_equal(np.diff(off), lens), n
        full = np.zeros((nb, n * n), dtype=np.int16)
        full[np.repeat(np.arange(nb), lens), so[np.arange(int(off[nb])) - np.repeat(off[:nb], lens)]] = o['pq'][:int(off[nb])]
        d = _first_difference(full.reshape(nb, n, n), ref[n]['q'])
        if d:
            bad.append('%dx%d packed levels: %s' % (n, n, d))
    assert bad == [], '\n'.join(bad)


def test_gpu_bench_step_4320p_edges_and_sample_vs_oracle(step):
    """7680x4320 (BASELINE configs[4], the whole-picture job of bench.strong_4320p): 4320 = 67 * 64 + 32, so the bottom root row is parentless
    32x32 blocks.  Every block of that row and of the right-hand root column, and a seeded sample of 1000 blocks per level, against the oracle"""
    torch, eng, env = step['torch'], step['eng'], step['env']
    w4, h4 = 2 * bench.W, 2 * bench.H
    org, ref, S = bench.synth_picture_pair(777, w4, h4)
    planes = _bind(torch, eng, org, ref, S, w4, h4, (50, 51))
    lists = pyramid_lists(SIZES[0], len(SIZES), w4, h4)
    job = bench.Job(env, w4, lists, 'test4320')
    torch.cuda.synchronize()
    try:
        out = _run(step, job, planes=(50, 51))
    finally:
        eng.free_plane(50); eng.free_plane(51)
    del planes
    bottom, right = (h4 // 64) * 64, w4 - 64
    assert bottom == 4288 and int((lists[2][1] == bottom).sum()) == w4 // 32 and not (lists[3][1] >= bottom).any()
    msgs, compared, timing = [], {}, {}
    t0 = time.perf_counter()
    for n, (xs, ys) in zip(SIZES, lists):
        edge = np.flatnonzero((ys >= bottom) | (xs >= right))
        idx = np.union1d(edge, np.random.RandomState(n).choice(len(xs), size=1000, replace=False))
        exp = SC.expected_level(org, ref, S, bench.MARGIN, n, xs[idx], ys[idx], bench.LAMBDA, bench.SEARCH_RANGE, PATTERN, bench.BITDEPTH, bench.QP,
                                timing=timing)
        msgs += SC.compare_level(n, xs[idx], ys[idx], exp, _device_level(out[n], idx), K, index=idx)
        compared[n] = (len(edge), len(idx))
    print('4320p: (edge blocks, blocks compared) per level %s; oracle %.1f s' % (compared, time.perf_counter() - t0))
    assert msgs == [], '\n'.join(msgs)
