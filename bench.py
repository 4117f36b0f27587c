#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 block-cost path (contract: see DESIGN.md section "Measurement").

Workload `2160p10_fullsearch_me_rdo` (BASELINE.json: candidate-blocks/s (SAD+SATD+DCT-quant) on 2160p10):
one 3840x2160 10-bit luma picture against one reference picture; for every block of the quad-tree depths
8x8, 16x16, 32x32, 64x64 tiling the picture
    1. integer full search, +-32 window (4225 SAD candidates, MV rate, raster tie-break)   InterSearch::xPatternSearch
    2. Hadamard (SATD) refinement over an 18-point ring pattern around the best vector      InterSearch.cpp:2582-2630 style
    3. residual = org - pred(best), forward DCT-II + quantise + RDOQ pre-check              TrQuant::transformNxN
A "step" is one BATCH of PICTURES_PER_STEP such pictures (a GOP's worth of candidate evaluation; the timed region of the default
run is then seconds, not milliseconds); units = candidate-blocks = SAD candidates + SATD candidates + TUs.

  value : whole-job candidate-blocks/s, inputs resident in HBM, K steps timed with CUDA events on the context stream
  e2e   : same step through the host-buffer C ABI (pictures + block lists uploaded, costs / vectors / levels downloaded
          for every picture), pinned host memory
  --impl reference : the reference's own AVX2 path (oracle/_ref, else the oracle port) on the host cores, bounded sample

N > 1 (torchrun): CTU-row bands (vvenc_b200.bands.split_ctu_rows) of ONE picture that is N times taller (weak scaling: 3840 x 2160*N, replicated on
every rank); every rank runs the kernels on its band; one NCCL all-gather of the per-block result tables per picture (bands.BandGather); after the
timed region rank 0 recomputes every band alone and requires the gathered tables to be bit-identical.  extra.strong_4320p: BASELINE configs[4] -- one
7680x4320 picture, CTU rows over the N ranks, gathered table == single-GPU table, strong-scaling efficiency from the same run.
"""
import argparse, ctypes, json, math, os, statistics, subprocess, sys, threading, time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, MARGIN, BITDEPTH = 3840, 2160, 80, 10
SIZES = (8, 16, 32, 64)
SEARCH_RANGE = 32
QP = 32
LAMBDA = 57.9          # ~ 0.57 * 2^((QP-12)/3), the encoder's lambda scale at QP 32
N_PICTURE_SETS = 4     # rotated between pictures: 4 x (org+ref) = 4 x 36.6 MB planes + outputs > 126 MB L2
PICTURES_PER_STEP = 40
CTU = 128


def refine_pattern():
    # centre + 8 neighbours at distance 1 + 8 at distance 2 + centre again at the end (18 points, integer-pel Hadamard refinement)
    pts = [(0, 0)] + [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if dx or dy] + [(dx, dy) for dy in (-2, 0, 2) for dx in (-2, 0, 2) if dx or dy] + [(0, 0)]
    return pts


def synth_picture_pair(seed, w=W, h=H, margin=MARGIN):
    """natural-like 10-bit luma: low-pass noise, reference = panned copy + noise (SURVEY 8d distribution ii)"""
    rs = np.random.RandomState(seed)
    S = w + 2 * margin
    Hh = h + 2 * margin
    base = rs.randint(0, 1024, size=(Hh // 4 + 3, S // 4 + 3)).astype(np.float32)
    up = np.kron(base, np.ones((4, 4), dtype=np.float32))[:Hh + 8, :S + 8]
    sm = (up[:-4, :-4] + up[4:, :-4] + up[:-4, 4:] + up[4:, 4:] + 2 * up[2:-2, 2:-2]) / 6.0
    sm = sm[:Hh + 4, :S + 4]
    tex = rs.randint(-24, 25, size=sm.shape)
    full = np.clip(sm + tex, 0, 1023)
    org = full[2:2 + Hh, 2:2 + S].astype(np.int16)
    ref = np.clip(full[2 + 1:2 + 1 + Hh, 2 - 2:2 - 2 + S] + rs.randint(-6, 7, size=org.shape), 0, 1023).astype(np.int16)
    return np.ascontiguousarray(org), np.ascontiguousarray(ref), S


def tall_picture(plane, n_bands, h=H, margin=MARGIN):
    """a picture n_bands times taller than `plane` (margins kept): band b carries the picture rolled 16*b pels to the left, so that bands differ"""
    if n_bands == 1:
        return plane
    inner = plane[margin:margin + h]
    parts = [plane[:margin]] + [np.roll(inner, -16 * b, axis=1) for b in range(n_bands)] + [plane[margin + h:]]
    return np.ascontiguousarray(np.concatenate(parts, axis=0))


_GRID_CACHE = {}


def block_grid(n, w=W, h=H):
    # quad-tree order of the encoder's partitioner: block j of size 2n is the parent of blocks 4j..4j+3 of size n (vvenc_b200.candidates.pyramid_lists)
    if (w, h) not in _GRID_CACHE:
        from vvenc_b200.candidates import pyramid_lists
        _GRID_CACHE[(w, h)] = pyramid_lists(SIZES[0], len(SIZES), w, h)
    return _GRID_CACHE[(w, h)][SIZES.index(n)]


def units_of(counts):
    """candidate-blocks of one picture (or band) with counts[size] blocks per size"""
    K = len(refine_pattern())
    u = {'sad': 0, 'satd': 0, 'tu': 0}
    for n in SIZES:
        u['sad'] += counts[n] * (2 * SEARCH_RANGE + 1) ** 2
        u['satd'] += counts[n] * K
        u['tu'] += counts[n]
    return u


def units_per_picture():
    return units_of({n: len(block_grid(n)[0]) for n in SIZES})


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index = index; self.proc = None; self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons), 'samples': len(sm)}




def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_dram_traffic(kernel_substr, profiles=('profiles/r02p_ncu_step_kernels.txt', 'profiles/r02_ncu_step_kernels.txt', 'profiles/r01_v8_ncu_step_kernels.txt')):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes per launch) of the first capture whose kernel name contains `kernel_substr`, from the committed
    `ncu --set full` summaries; (None, None) when no file holds the kernel"""
    unit = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    for profile in profiles:
        try:
            for blk in open(os.path.join(ROOT, profile)).read().split('-' * 100):
                name = [l for l in blk.split('\n') if l.startswith('Kernel Name')]
                if not name or kernel_substr not in name[0]:
                    continue
                tot = 0.0; seen = 0
                for l in blk.split('\n'):
                    if l.startswith('dram__bytes_read.sum') or l.startswith('dram__bytes_write.sum'):
                        f = l.split()
                        tot += float(f[1].replace(',', '')) * unit[f[2]]; seen += 1
                if seen == 2:
                    return tot, profile
        except Exception:
            continue
    return None, None


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores (oracle/_ref), else the oracle port
# ---------------------------------------------------------------------------------------------------------------
def host_cpus():
    """CPUs this process may actually use: scheduler affinity capped by the cgroup CPU quota (v2 cpu.max, v1 cfs_quota_us); os.cpu_count() alone
    reports the machine, not the container (round 1: two boxes both said 128 and differed 3.2x)"""
    info = {'os_cpu_count': os.cpu_count()}
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    info['affinity'] = aff
    quota = None
    try:
        f = open('/sys/fs/cgroup/cpu.max').read().split()
        if f and f[0] != 'max':
            quota = float(f[0]) / float(f[1])
    except Exception:
        try:
            q = float(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read()); p = float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    info['cgroup_quota_cpus'] = quota
    n = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    info['usable'] = n
    try:
        model = [l.split(':', 1)[1].strip() for l in open('/proc/cpuinfo') if l.startswith('model name')]
        info['model'] = model[0] if model else None
    except Exception:
        info['model'] = None
    return n, info


_THREAD_CHOICE = {}
_CPU_CACHE = {}


def pick_threads(run_probe, usable):
    """thread sweep {usable/2, usable, 2*usable}: keeps the count with the best probe rate (SMT siblings / quota make either end win on some hosts)"""
    if 'n' in _THREAD_CHOICE:
        return _THREAD_CHOICE['n'], _THREAD_CHOICE['sweep']
    sweep = {}
    for t in sorted({max(1, usable // 2), usable, 2 * usable}):
        run_probe(t)                                  # warm
        c0 = time.process_time(); w0 = time.perf_counter()
        units = run_probe(t)
        w = time.perf_counter() - w0; c = time.process_time() - c0
        sweep[t] = {'rate': units / w, 'cpu_seconds_per_wall_second': c / w}
    best = max(sweep, key=lambda t: sweep[t]['rate'])
    _THREAD_CHOICE['n'] = best; _THREAD_CHOICE['sweep'] = {str(k): v for k, v in sweep.items()}
    return best, _THREAD_CHOICE['sweep']


def cpu_arm(sample_budget_s=12.0, threads=None, quiet=False):
    """times a bounded sample of the SAME per-picture workload on the host; returns dict(value cand-blocks/s, kind, cores, sample, per-leg rates)"""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from _libs import have_ref, refshim, oracle, P, PO
    kind = 'reference' if have_ref() else 'port'
    if 'pic' not in _CPU_CACHE:
        _CPU_CACHE['pic'] = synth_picture_pair(1234)
    org, ref, S = _CPU_CACHE['pic']
    base = MARGIN * S + MARGIN
    K = len(refine_pattern()); pat = refine_pattern()
    legs = {}
    R = refshim() if kind == 'reference' else None
    O = oracle()
    usable, cpu_info = host_cpus()
    sweep = None
    if kind == 'port':
        threads = 1
    elif threads is None:
        xs16, ys16 = block_grid(16)
        def probe(t):
            cnt = min(len(xs16), 6 * t)
            blk = np.zeros((cnt, 10), dtype=np.int32)
            blk[:, 0] = xs16[:cnt]; blk[:, 1] = ys16[:cnt]; blk[:, 2] = 16; blk[:, 3] = 16
            blk[:, 4] = -SEARCH_RANGE; blk[:, 5] = SEARCH_RANGE; blk[:, 6] = -SEARCH_RANGE; blk[:, 7] = SEARCH_RANGE
            out = np.zeros((cnt, 4), dtype=np.int32)
            R.refshim_full_search(1, PO(org, base), S, PO(ref, base), S, P(blk), cnt, BITDEPTH, 0, LAMBDA, 2, 0, P(out), None, 0, t, 1)
            return cnt
        threads, sweep = pick_threads(probe, usable)
    u = units_per_picture()
    per_leg_budget = sample_budget_s / (3 * len(SIZES))
    sample_desc = []
    t_step = 0.0
    cpu_s = 0.0; wall_s = 0.0
    for n in SIZES:
        xs, ys = block_grid(n)
        nb_all = len(xs)
        # ---- SAD full search: calibrate on a few blocks, then size the sample to the budget
        def run_search(idx):
            blk = np.zeros((len(idx), 10), dtype=np.int32)
            blk[:, 0] = xs[idx]; blk[:, 1] = ys[idx]; blk[:, 2] = n; blk[:, 3] = n
            blk[:, 4] = -SEARCH_RANGE; blk[:, 5] = SEARCH_RANGE; blk[:, 6] = -SEARCH_RANGE; blk[:, 7] = SEARCH_RANGE
            out = np.zeros((len(idx), 4), dtype=np.int32)
            t0 = time.perf_counter()
            if R is not None:
                R.refshim_full_search(1, PO(org, base), S, PO(ref, base), S, P(blk), len(idx), BITDEPTH, 0, LAMBDA, 2, 0, P(out), None, 0, threads, 1)
            else:
                O.orc_full_search(PO(org, base), S, PO(ref, base), S, P(blk), len(idx), 0, LAMBDA, 2, 0, P(out), None, 0)
            return time.perf_counter() - t0, out
        rs = np.random.RandomState(n)
        probe = rs.choice(nb_all, size=min(nb_all, 4 * threads), replace=False)
        tp, _ = run_search(probe)
        cnt = int(min(nb_all, max(len(probe), len(probe) * per_leg_budget / max(tp, 1e-6))))
        idx = rs.choice(nb_all, size=cnt, replace=False)
        c0 = time.process_time()
        ts, best = run_search(idx)
        cpu_s += time.process_time() - c0; wall_s += ts
        t_sad = ts / cnt * nb_all
        # ---- SATD refinement around the best vectors of the sample
        desc = np.zeros((cnt * K, 6), dtype=np.int32)
        bx = np.repeat(xs[idx], K); by = np.repeat(ys[idx], K)
        ddx = np.tile(np.array([p[0] for p in pat], dtype=np.int32), cnt) + np.repeat(best[:, 0], K)
        ddy = np.tile(np.array([p[1] for p in pat], dtype=np.int32), cnt) + np.repeat(best[:, 1], K)
        desc[:, 0] = bx; desc[:, 1] = by; desc[:, 2] = bx + ddx; desc[:, 3] = by + ddy; desc[:, 4] = n; desc[:, 5] = n
        outc = np.zeros(cnt * K, dtype=np.uint64)
        t0 = time.perf_counter()
        if R is not None:
            R.refshim_dist_list(1, 2, PO(org, base), S, PO(ref, base), S, P(desc), cnt * K, BITDEPTH, 0, P(outc), threads)
        else:
            O.orc_dist_list(2, PO(org, base), S, PO(ref, base), S, P(desc), cnt * K, 0, P(outc))
        t_satd = (time.perf_counter() - t0) / cnt * nb_all
        # ---- TU: residual of the best prediction, DCT-II + quantise
        resi = np.zeros((cnt, n, n), dtype=np.int16)
        for i in range(cnt):
            x, y = int(xs[idx[i]]), int(ys[idx[i]]); mx, my = int(best[i, 0]), int(best[i, 1])
            resi[i] = org[MARGIN + y:MARGIN + y + n, MARGIN + x:MARGIN + x + n] - ref[MARGIN + y + my:MARGIN + y + my + n, MARGIN + x + mx:MARGIN + x + mx + n]
        q = np.zeros((cnt, n, n), dtype=np.int16); s = np.zeros(cnt, dtype=np.int32); lp = np.zeros(cnt, dtype=np.int32)
        t0 = time.perf_counter()
        if R is not None:
            R.refshim_transform_quant_batch(0, 0, P(resi), cnt, n, n, BITDEPTH, QP, 0, P(q), P(s), P(lp), threads)
        else:
            coef = np.zeros((n, n), dtype=np.int32)
            for i in range(cnt):
                O.orc_transform_quant(0, 0, P(resi[i]), n, n, n, BITDEPTH, QP, 0, P(coef), P(q[i]), PO(s, i), PO(lp, i))
        t_tu = (time.perf_counter() - t0) / cnt * nb_all
        legs[n] = {'sad_s': t_sad, 'satd_s': t_satd, 'tu_s': t_tu, 'sample_blocks': cnt}
        sample_desc.append('%dx%d:%d/%d blocks' % (n, n, cnt, nb_all))
        t_step += t_sad + t_satd + t_tu
    total_units = u['sad'] + u['satd'] + u['tu']
    return {'value': total_units / t_step, 'unit': 'candidate-blocks/s', 'cores': threads, 'kind': kind,
            'sample': ('random block sample per size, full-picture time extrapolated per leg (' + ', '.join(sample_desc) + '); AVX2, early exit on; %d threads chosen by a sweep over '
                       '{usable/2, usable, 2x usable} of %d usable CPUs (affinity %s, cgroup quota %s, os.cpu_count %s)'
                       % (threads, usable, cpu_info['affinity'], cpu_info['cgroup_quota_cpus'], cpu_info['os_cpu_count'])) if kind == 'reference'
                      else 'scalar oracle port, ' + ', '.join(sample_desc),
            'cpu_s_per_picture': t_step, 'legs': legs, 'value_per_thread': total_units / t_step / threads,
            'host': cpu_info, 'thread_sweep': sweep, 'search_cpu_seconds_per_wall_second': (cpu_s / wall_s) if wall_s > 0 else None}


def cpu_rows(threads=None, budget_s=1.5):
    """the reference's own AVX2 code on the host cores for the rows of SURVEY section 8 outside the headline step (TU round trip, MCTF block
    matching grid, fractional SATD grid, MCTF apply): a bounded sample each, same units as the matching extra.* GPU entries.  Needs oracle/_ref."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from _libs import have_ref, refshim, P, PO
    if not have_ref():
        return {'unavailable': 'oracle/_ref not built'}
    R = refshim()
    threads = threads or host_cpus()[0]
    w, h = 1280, 720
    org, ref, S = synth_picture_pair(4321, w, h, MARGIN)
    base = MARGIN * S + MARGIN
    rs = np.random.RandomState(77)
    rows = {'cores': threads, 'kind': 'reference', 'picture': '%dx%d sample of the same synthetic content' % (w, h)}

    def sized(run, n0, cap):
        """calibrate on n0 units, then one run sized to the budget"""
        t = run(n0)
        n = int(min(cap, max(n0, n0 * budget_s / max(t, 1e-6))))
        t = run(n)
        reps = int(min(50, max(1, budget_s / max(t, 1e-6))))                      # sample capped by the picture: repeat it until the budget is used
        return n, sum(run(n) for _ in range(reps)) / reps

    # TU round trip (TrQuant::transformNxN + Quant::quant + dequant + invTransformNxN + reconstruct + SSE), DCT-II, QP of the step
    tu = {}
    for n in SIZES:
        cap = (64 << 20) // (4 * n * n)
        o = rs.randint(0, 1024, size=cap * n * n).astype(np.int16)
        pr = np.clip(o + rs.randint(-200, 201, size=o.size), 0, 1023).astype(np.int16)
        q = np.zeros(cap * n * n, dtype=np.int16); rc = np.zeros(cap * n * n, dtype=np.int16); o4 = np.zeros(cap * 4, dtype=np.uint64)
        def run(cnt):
            t0 = time.perf_counter()
            R.refshim_tu_roundtrip_batch(1, 0, 0, P(o), P(pr), cnt, n, n, BITDEPTH, QP, 0, P(q), P(rc), P(o4), threads)
            return time.perf_counter() - t0
        cnt, t = sized(run, 16 * threads, cap)
        tu[str(n)] = {'tus': cnt, 's': t, 'tu_per_s': cnt / t}
    rows['tu_roundtrip'] = tu

    # MCTF block matching (motionErrorLumaFrac6/Int8): every 16x16 block, the 49 quarter-step vectors of the doubleRes refinement
    B = 16
    gx, gy = np.meshgrid(np.arange(0, w - B + 1, B), np.arange(0, h - B + 1, B))
    off = np.array([(dx, dy) for dy in range(-12, 13, 4) for dx in range(-12, 13, 4)], dtype=np.int32)
    nbk = gx.size; K = len(off)
    desc = np.zeros((nbk * K, 6), dtype=np.int32)
    desc[:, 0] = np.repeat(gx.reshape(-1), K); desc[:, 1] = np.repeat(gy.reshape(-1), K)
    desc[:, 2] = np.tile(off[:, 0], nbk) + 32; desc[:, 3] = np.tile(off[:, 1], nbk) - 16; desc[:, 4] = B; desc[:, 5] = B
    err = np.zeros(nbk * K, dtype=np.int32)
    def run(cnt):
        t0 = time.perf_counter()
        R.refshim_mctf_err_list(1, 0, PO(org, base), S, PO(ref, base), S, P(desc), cnt, BITDEPTH, P(err), threads)
        return time.perf_counter() - t0
    cnt, t = sized(run, K * 4 * threads, nbk * K)
    rows['mctf_match_16x16'] = {'candidates': cnt, 's': t, 'cand_per_s': cnt / t, 'block_refs_per_s': cnt / K / t}

    # MCTF motion search of one neighbour picture (motionEstimationMCTF: pyramids + 4 levels of motionEstimationLuma), the reference's members on ONE thread
    # (the probe drives one MCTF object; inside the encoder the block lines of a level are spread over the thread pool): a 960x544 crop, scaled by area
    try:
        cw, ch = min(960, w), min(544, h)
        co = np.ascontiguousarray(org[MARGIN:MARGIN + ch, MARGIN:MARGIN + cw]); cr_ = np.ascontiguousarray(ref[MARGIN:MARGIN + ch, MARGIN:MARGIN + cw])
        expf = np.zeros(((ch + 15) // 16, (cw + 15) // 16, 4), dtype=np.int32)
        t0 = time.perf_counter()
        R.refshim_mctf_estimate_pyramid(1, P(co), P(cr_), cw, ch, BITDEPTH, 16, 0, 0, 0, P(expf))
        dt = time.perf_counter() - t0
        rows['mctf_motion_estimation'] = {'sample': '%dx%d crop, unit 16, 4 levels, AVX2 members' % (cw, ch), 'threads': 1, 's': dt, 'pels_per_s_per_thread': cw * ch / dt,
                                          'pels_per_s_if_all_threads_scaled': cw * ch / dt * threads}
    except Exception as ex:
        rows['mctf_motion_estimation'] = {'error': str(ex)}

    # fractional SATD grid (InterpolationFilter two-pass + HAD): 49 quarter-pel offsets per block
    fr = {}
    for n in (8, 16, 32):
        xs, ys = block_grid(n, w, h)
        blk = np.zeros((len(xs), 6), dtype=np.int32)
        blk[:, 0] = xs; blk[:, 1] = ys; blk[:, 2] = n; blk[:, 3] = n; blk[:, 4] = rs.randint(-8, 9, size=len(xs)); blk[:, 5] = rs.randint(-8, 9, size=len(xs))
        out = np.zeros(len(xs) * 49, dtype=np.uint32)
        def run(cnt):
            t0 = time.perf_counter()
            R.refshim_frac_cost_grid_mt(1, PO(org, base), S, PO(ref, base), S, P(blk), cnt, 2, BITDEPTH, 2, 0, P(out), threads)
            return time.perf_counter() - t0
        cnt, t = sized(run, min(len(xs), 2 * threads), len(xs))
        fr[str(n)] = {'blocks': cnt, 's': t, 'cand_per_s': cnt * 49 / t}
    rows['frac_satd_grid'] = fr

    # MCTF apply stage (xFinalizeBlkLine: applyFrac + planar correction + applyBlock), 8 neighbour pictures, unit 16
    nrefs = 8
    planes = [np.ascontiguousarray(np.roll(ref, (i + 1, 2 * i - 5), axis=(0, 1))) for i in range(nrefs)]
    ptrs = (ctypes.c_void_p * nrefs)(*[ctypes.cast(PO(p_, base), ctypes.c_void_p).value for p_ in planes])
    bxN, byN = w // B, h // B
    mv4 = np.zeros((nrefs, bxN * byN, 4), dtype=np.int32)
    mv4[:, :, 0] = rs.randint(-40, 41, size=(nrefs, bxN * byN)); mv4[:, :, 1] = rs.randint(-40, 41, size=(nrefs, bxN * byN))
    mv4[:, :, 2] = rs.randint(5, 150, size=(nrefs, bxN * byN)); mv4[:, :, 3] = rs.randint(0, 30, size=(nrefs, bxN * byN))
    stg = (ctypes.c_double * nrefs)(0.85, 0.57, 0.41, 0.33, 0.30, 0.20, 0.18, 0.15)
    dst = np.zeros((h, w), dtype=np.int16)
    R.refshim_mctf_finalize_picture.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_void_p,
                                                ctypes.c_int, ctypes.c_int]
    def run(_):
        t0 = time.perf_counter()
        R.refshim_mctf_finalize_picture(1, PO(org, base), S, ptrs, S, nrefs, P(mv4), w, h, B, BITDEPTH, 0, 1, stg, 0.4, 9 * (128.0 + 3.0 / 256.0 * 32 ** 3), P(dst), w, threads)
        return time.perf_counter() - t0
    _, t = sized(run, 1, 1)
    rows['mctf_apply'] = {'pels': w * h, 'refs': nrefs, 'unit': B, 's': t, 'pels_per_s': w * h / t, 'block_refs_per_s': bxN * byN * nrefs / t}
    return rows



# ---------------------------------------------------------------------------------------------------------------
class Job:
    """device-resident state of one band of a picture geometry: per-size block lists (quad-tree order) and every output buffer of a step"""

    def __init__(self, env, width, lists, tag):
        torch, V = env['torch'], env['V']
        self.width = width; self.tag = tag
        self.blocks_np, self.d_blocks, self.d_best, self.d_satd, self.d_q, self.d_sum, self.d_last, self.d_nr = {}, {}, {}, {}, {}, {}, {}, {}
        KP = env['KP']
        for n, (xs, ys) in zip(SIZES, lists):
            b = np.zeros(len(xs), dtype=V.BLOCK_DT)
            b['x'] = xs; b['y'] = ys; b['left'] = -SEARCH_RANGE; b['right'] = SEARCH_RANGE; b['top'] = -SEARCH_RANGE; b['bottom'] = SEARCH_RANGE
            self.blocks_np[n] = b
            self.d_blocks[n] = env['dev'](b)
            nb = max(1, len(b))
            self.d_best[n] = torch.empty(nb * 16, dtype=torch.uint8, device='cuda')
            self.d_satd[n] = torch.empty(nb * KP, dtype=torch.int32, device='cuda')
            self.d_q[n] = torch.empty(nb * n * n, dtype=torch.int16, device='cuda')
            self.d_sum[n] = torch.empty(nb, dtype=torch.int32, device='cuda'); self.d_last[n] = torch.empty(nb, dtype=torch.int32, device='cuda')
            self.d_nr[n] = torch.empty(nb, dtype=torch.uint8, device='cuda')
        nlev = len(SIZES)
        self.counts = {n: len(self.blocks_np[n]) for n in SIZES}
        self.pyr_blocks = (ctypes.c_void_p * nlev)(*[self.d_blocks[n].data_ptr() for n in SIZES])
        self.pyr_best = (ctypes.c_void_p * nlev)(*[self.d_best[n].data_ptr() for n in SIZES])
        self.pyr_counts = (ctypes.c_int * nlev)(*[self.counts[n] for n in SIZES])
        self.units = units_of(self.counts)
        self.total_units = self.units['sad'] + self.units['satd'] + self.units['tu']
        self.best_bytes = sum(self.counts[n] * 16 for n in SIZES)

    def best_pieces(self):
        return [self.d_best[n][:self.counts[n] * 16] for n in SIZES]

    def run(self, env, po, pr, direct=False):
        """one picture: search -> SATD refinement around the best vector -> residual + DCT-II + quantise, chained on the device"""
        lib, eng, V, chk, me, nx = env['lib'], env['eng'], env['V'], env['chk'], env['me'], env['nx']
        P_ = ctypes.c_void_p
        nlev = len(SIZES)
        if not direct:       # SAD pyramid: pel work at 8x8 only, larger sizes are exact sums of their children's SADs at the same vector
            chk(lib.vvb_sad_search_pyramid_dev(eng.h, po, pr, nlev, self.pyr_blocks, self.pyr_counts, SIZES[0], ctypes.byref(me), nx, nx, self.pyr_best))
        for n in SIZES:
            nb = self.counts[n]
            if nb == 0:
                continue
            if direct:       # every size searched on its own (what InterSearch::xPatternSearch does per PU)
                chk(lib.vvb_sad_search_dev(eng.h, po, pr, P_(self.d_blocks[n].data_ptr()), nb, n, n, ctypes.byref(me), nx, nx, None, 0, P_(self.d_best[n].data_ptr())))
            chk(lib.vvb_blocks_set_start_dev(eng.h, P_(self.d_blocks[n].data_ptr()), P_(self.d_best[n].data_ptr()), nb))
            chk(lib.vvb_cost_pattern_dev(eng.h, V.DF_HAD, po, pr, P_(self.d_blocks[n].data_ptr()), nb, n, n, P_(env['d_pat'].data_ptr()), env['KP'], ctypes.byref(me),
                                         P_(self.d_satd[n].data_ptr()), None))
            chk(lib.vvb_fwd_trquant_planes_dev(eng.h, ctypes.byref(env['tu_par'][n]), po, pr, P_(self.d_blocks[n].data_ptr()), nb, None, P_(self.d_q[n].data_ptr()),
                                               P_(self.d_sum[n].data_ptr()), P_(self.d_last[n].data_ptr()), P_(self.d_nr[n].data_ptr())))

    def snapshot(self, torch):
        return {n: (self.d_best[n][:self.counts[n] * 16].clone(), self.d_satd[n].clone(), self.d_sum[n].clone(), self.d_last[n].clone(), self.d_q[n].clone()) for n in SIZES}


DUMP_Q_VALUES = 1 << 20      # levels kept per block size in --dump-outputs: a seeded sample of whole blocks


def dump_outputs(job, out_dir, V):
    """what a caller of the step receives for its last picture, per block size: best vector records, SATD ring costs, TU summaries and the
    levels of a fixed sample of blocks (all of them would be 133 MB as float32); integers stored exactly (float64 where they may pass 2^24)"""
    os.makedirs(out_dir, exist_ok=True)
    for n in SIZES:
        nb = job.counts[n]
        best = np.frombuffer(job.d_best[n][:nb * 16].cpu().numpy().tobytes(), dtype=V.BEST_DT)
        np.save(os.path.join(out_dir, 'best_%dx%d.npy' % (n, n)), np.stack([best[f].astype(np.float64) for f in ('dx', 'dy', 'sad', 'cost')], axis=1))
        np.save(os.path.join(out_dir, 'satd_%dx%d.npy' % (n, n)), job.d_satd[n][:nb * len(refine_pattern())].cpu().numpy().astype(np.float64).reshape(nb, -1))
        tu = [job.d_sum[n][:nb], job.d_last[n][:nb], job.d_nr[n][:nb]]
        np.save(os.path.join(out_dir, 'tu_sum_last_rdoq_%dx%d.npy' % (n, n)), np.stack([t.cpu().numpy().astype(np.float64) for t in tu], axis=1))
        pick = np.sort(np.random.RandomState(n).choice(nb, size=min(nb, DUMP_Q_VALUES // (n * n)), replace=False))
        q = job.d_q[n][:nb * n * n].cpu().numpy().reshape(nb, n * n)[pick]
        np.save(os.path.join(out_dir, 'q_%dx%d.npy' % (n, n)), q.astype(np.float32))
        np.save(os.path.join(out_dir, 'q_blocks_%dx%d.npy' % (n, n)), pick.astype(np.float64))


def sharded_parity(env, jobs_all_bands, gather, po, pr, own_job):
    """rank 0: every band recomputed on this GPU alone must equal what the band's owner sent through the all-gather, bit for bit"""
    torch, eng = env['torch'], env['eng']
    checked = 0; equal = True
    for b, job in enumerate(jobs_all_bands):
        job.run(env, po, pr)
        eng.synchronize(); torch.cuda.synchronize()
        mine = torch.cat(job.best_pieces())
        got = gather.table(b)
        equal = equal and bool(torch.equal(mine, got))
        checked += sum(job.counts.values())
    return {'bands': len(jobs_all_bands), 'blocks_checked': int(checked), 'gathered_equals_single_gpu': bool(equal)}


def strong_4320p(env, rank, world, pictures=6):
    """BASELINE configs[4]: ONE 7680x4320 picture, CTU rows sharded over the ranks (bands.split_ctu_rows), all-gather of the result tables, gathered table ==
    single-GPU table; strong-scaling efficiency = t(1 GPU, whole picture) / (N * t(N GPUs))"""
    torch, dist, V, eng, bands = env['torch'], env['dist'], env['V'], env['eng'], env['bands']
    w4, h4 = 2 * W, 2 * H
    sets = []
    for s in range(2):
        org, ref, S = synth_picture_pair(777 + s, w4, h4, MARGIN)
        dorg = torch.from_numpy(org).cuda(); dref = torch.from_numpy(ref).cuda()
        base = (MARGIN * S + MARGIN) * 2
        eng.bind_plane_dev(50 + 2 * s, dorg.data_ptr() + base, S, w4, h4, MARGIN, BITDEPTH)
        eng.bind_plane_dev(51 + 2 * s, dref.data_ptr() + base, S, w4, h4, MARGIN, BITDEPTH)
        sets.append((dorg, dref))
    rows = bands.split_ctu_rows(h4, CTU, world)
    jobs = [Job(env, w4, bands.band_pyramid_lists(SIZES[0], len(SIZES), w4, y0, y1), 'band%d' % b) if (b == rank or rank == 0) else None for b, (y0, y1) in enumerate(rows)]
    whole = Job(env, w4, bands.band_pyramid_lists(SIZES[0], len(SIZES), w4, 0, h4), 'whole') if rank == 0 else None
    own = jobs[rank]
    ext = env['ext']
    all_bytes = [sum(len(xs) * 16 for xs, _ in bands.band_pyramid_lists(SIZES[0], len(SIZES), w4, y0, y1)) for (y0, y1) in rows]
    gather = bands.BandGather(all_bytes, torch.device('cuda', env['local'])) if world > 1 else None

    def timed(fn, count):
        for i in range(2):
            fn(i)
        eng.synchronize(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record(ext)
            for i in range(count):
                fn(2 + i)
            if gather is not None:
                gather.wait(ext)
            e1.record(ext)
        eng.synchronize(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / count], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def band_step(i):
        s = i % 2
        own.run(env, 50 + 2 * s, 51 + 2 * s)
        if gather is not None:
            gather.launch(own.best_pieces(), ext)
    ms_n = timed(band_step, pictures)
    out = {'picture': '%dx%d 10-bit, 1 reference' % (w4, h4), 'n_gpus': world, 'ctu_rows_per_rank': [(y1 - y0 + CTU - 1) // CTU for y0, y1 in rows],
           'ms_per_picture_sharded': ms_n, 'pictures_timed': pictures}
    u_total = sum(units_of({n: len(xs) for n, (xs, _) in zip(SIZES, bands.band_pyramid_lists(SIZES[0], len(SIZES), w4, 0, h4))}).values())
    out['value_sharded'] = u_total / (ms_n * 1e-3)
    if world > 1:
        # parity on the last picture issued (set index known), then the single-GPU time of the whole picture on rank 0
        last = (2 + pictures - 1) % 2
        band_step(2 + pictures - 1)
        with torch.cuda.stream(ext):
            gather.wait(ext)
        eng.synchronize(); torch.cuda.synchronize(); dist.barrier()
        if rank == 0:
            out['parity'] = sharded_parity(env, jobs, gather, 50 + 2 * last, 51 + 2 * last, own)
            whole.run(env, 50 + 2 * last, 51 + 2 * last)
            eng.synchronize(); torch.cuda.synchronize()
            # the whole-picture job lists the same blocks in another order (its own quad-tree walk): compare as sets keyed by (size, x, y)
            def keyed(job_list):
                d = {}
                for j in job_list:
                    for n in SIZES:
                        bl = j.blocks_np[n]; be = np.frombuffer(j.d_best[n][:j.counts[n] * 16].cpu().numpy().tobytes(), dtype=V.BEST_DT)
                        for k in range(0, len(bl), max(1, len(bl) // 4000)):            # sampled: 4000 blocks per size and band
                            d[(n, int(bl['x'][k]), int(bl['y'][k]))] = (int(be['dx'][k]), int(be['dy'][k]), int(be['cost'][k]))
                return d
            a = keyed(jobs); bfull = keyed([whole])
            common = [k for k in a if k in bfull]
            out['parity']['whole_picture_vs_bands_sampled'] = {'blocks': len(common), 'equal': all(a[k] == bfull[k] for k in common)}
        t1 = torch.tensor([0.0], dtype=torch.float64, device='cuda')
        if rank == 0:
            def whole_step(i):
                s = i % 2
                whole.run(env, 50 + 2 * s, 51 + 2 * s)
            for i in range(2):
                whole_step(i)
            eng.synchronize(); torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(ext):
                e0.record(ext)
                for i in range(pictures):
                    whole_step(2 + i)
                e1.record(ext)
            eng.synchronize(); torch.cuda.synchronize()
            t1[0] = e0.elapsed_time(e1) / pictures
        dist.broadcast(t1, 0)
        out['ms_per_picture_1gpu'] = float(t1.item())
        out['strong_efficiency'] = float(t1.item()) / (world * ms_n)
    for s in range(2):
        eng.free_plane(50 + 2 * s); eng.free_plane(51 + 2 * s)
    del sets
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed steps of the headline measurement (the e2e leg times min(max(steps, 2), 5) steps)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-budget', type=float, default=12.0)
    ap.add_argument('--pictures-per-step', type=int, default=PICTURES_PER_STEP)
    ap.add_argument('--skip-e2e', action='store_true')
    ap.add_argument('--skip-cpu', action='store_true', help='profiling runs: no CPU baseline leg')
    ap.add_argument('--skip-extras', action='store_true', help='profiling runs: no per-kernel rows')
    ap.add_argument('--strong', action='store_true', help='also run the 4320p strong-scaling case at N = 1 (always run for N > 1)')
    ap.add_argument('--dump-outputs', metavar='DIR', help="write the last timed picture's results (rank 0's band) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the GPU path\'s results; --impl reference has none')
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1')); local = int(os.environ.get('LOCAL_RANK', '0'))
    PPS = max(1, args.pictures_per_step)
    u = units_per_picture()
    config = {'workload': '2160p10_fullsearch_me_rdo', 'step': 'a batch of %d pictures (each: full search + SATD refinement + TU for every 8/16/32/64 block)' % PPS,
              'pictures_per_step': PPS, 'search': 'SAD pyramid (exact): pels visited at 8x8, 16/32/64 = sums of children; extra.direct_search has the per-size search',
              'picture': '%dx%d 10-bit luma, 1 reference picture' % (W, H), 'block_sizes': list(SIZES),
              'search_range': SEARCH_RANGE, 'satd_points': len(refine_pattern()), 'tu': 'DCT-II + quant, one per block', 'qp': QP,
              'units_per_picture': u, 'l2': 'inputs rotated over %d picture sets (> L2)' % N_PICTURE_SETS,
              'parallelism': 'ctu-row bands x%d of one %dx%d picture' % (max(1, args.gpus), W, H * max(1, args.gpus))}

    # ------------------------------------------------------------------------------------------- reference arm
    if args.impl == 'reference':
        if rank != 0:
            return 0
        K, Wm = max(1, args.steps), max(0, args.warmup)
        budget = max(2.0, min(12.0, 100.0 / (K + Wm)))
        vals = []
        for i in range(K + Wm):
            r = cpu_arm(budget)
            if i >= Wm:
                vals.append(r)
        v = statistics.mean(x['value'] for x in vals)
        r = vals[-1]
        per_pic = u['sad'] + u['satd'] + u['tu']
        line = {'impl': 'reference', 'metric': 'candidate-blocks/s (SAD+SATD+DCT-quant) on 2160p10', 'value': v, 'unit': 'candidate-blocks/s',
                'n_gpus': args.gpus, 'steps': K, 'warmup': Wm, 'ms_per_step': 1e3 * per_pic * PPS / v, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'int16/int32', 'data': 'synthetic', 'config': config,
                'cpu_baseline': {'value': v, 'unit': 'candidate-blocks/s', 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample'],
                                 'value_per_thread': v / r['cores'], 'host': r['host'], 'thread_sweep': r['thread_sweep'],
                                 'run_to_run': {'min': min(x['value'] for x in vals), 'max': max(x['value'] for x in vals)}},
                'e2e': {'value': v, 'unit': 'candidate-blocks/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line)); return 0

    # ------------------------------------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    import vvenc_b200 as V
    from vvenc_b200 import bands
    eng = V.CostEngine(local)
    if os.environ.get('VVB_TMA', '') == '1':            # A/B switch: stage the search windows with cp.async.bulk.tensor where they are 16-byte aligned
        eng.set_tma_staging(1)
    if os.environ.get('VVB_PYRAMID', '') != '':         # A/B switch: 0 = per-quad pyramid kernel + table sums through HBM (round 1), 1 = in-CTA pyramid
        eng.set_pyramid_engine(int(os.environ['VVB_PYRAMID']))
    lib = eng.lib
    ext = torch.cuda.ExternalStream(eng.stream, device=torch.device('cuda', local))
    hbm_peak, peak_src = measured_peaks()

    pat_np = np.zeros(len(refine_pattern()), dtype=V.MV_DT)
    pat_np['dx'] = [p[0] for p in refine_pattern()]; pat_np['dy'] = [p[1] for p in refine_pattern()]
    KP = len(pat_np)
    me = eng.me_par(LAMBDA, 2, 0, 0, 1, 2)   # quad_order: the block lists below are in z-order; pattern_radius 2: the refinement ring
    nx = 2 * SEARCH_RANGE + 1

    def dev(a):
        return torch.from_numpy(np.frombuffer(a.tobytes(), dtype=np.uint8).copy()).cuda()

    def chk(rc):
        if rc != 0:
            raise RuntimeError('vvenc_b200: ' + lib.vvb_last_error(eng.h).decode())

    env = {'torch': torch, 'dist': dist, 'V': V, 'eng': eng, 'lib': lib, 'chk': chk, 'me': me, 'nx': nx, 'dev': dev, 'KP': KP, 'd_pat': dev(pat_np), 'ext': ext,
           'bands': bands, 'local': local,
           'tu_par': {n: eng.tu_par(n, n, V.DCT2, V.DCT2, BITDEPTH, QP, False, False) for n in SIZES}}

    # resident inputs: N_PICTURE_SETS pairs of ONE picture of 3840 x (2160 * world), replicated on every rank
    HT = H * world
    host_sets = []
    dev_planes = []
    for s in range(N_PICTURE_SETS):
        org, ref, S = synth_picture_pair(1234 + 17 * s)
        host_sets.append((org, ref, S))
        torg = tall_picture(org, world); tref = tall_picture(ref, world)
        dorg = torch.from_numpy(torg).cuda(); dref = torch.from_numpy(tref).cuda()
        dev_planes.append((dorg, dref))
        base = (MARGIN * S + MARGIN) * 2
        eng.bind_plane_dev(2 * s, dorg.data_ptr() + base, S, W, HT, MARGIN, BITDEPTH)
        eng.bind_plane_dev(2 * s + 1, dref.data_ptr() + base, S, W, HT, MARGIN, BITDEPTH)
    rows = bands.split_ctu_rows(HT, CTU, world)
    band_lists = [bands.band_pyramid_lists(SIZES[0], len(SIZES), W, y0, y1) for (y0, y1) in rows]
    job = Job(env, W, band_lists[rank], 'band%d' % rank)
    all_units = [sum(units_of({n: len(xs) for n, (xs, _) in zip(SIZES, bl)}).values()) for bl in band_lists]
    units_picture_all = sum(all_units)                       # candidate-blocks of the whole (tall) picture = what all ranks process per picture
    gather = bands.BandGather([sum(len(xs) * 16 for xs, _ in bl) for bl in band_lists], torch.device('cuda', local)) if world > 1 else None
    torch.cuda.synchronize()

    P_ = ctypes.c_void_p
    nlev = len(SIZES)
    blocks_np, d_blocks, d_best, d_satd, d_q, d_sum, d_last, d_nr, tu_par = job.blocks_np, job.d_blocks, job.d_best, job.d_satd, job.d_q, job.d_sum, job.d_last, job.d_nr, env['tu_par']
    pyr_blocks, pyr_best, pyr_counts = job.pyr_blocks, job.pyr_best, job.pyr_counts

    def picture_resident(idx, direct=False):
        s = idx % N_PICTURE_SETS
        job.run(env, 2 * s, 2 * s + 1, direct)
        if gather is not None:
            # per-block result tables of the band: snapshot on the compute stream, all-gather on a side stream so that the collective overlaps the next picture's search
            gather.launch(job.best_pieces(), ext)

    def step_resident(i, direct=False):
        for p in range(PPS):
            picture_resident(i * PPS + p, direct)

    def timed(fn, steps, warm):
        for i in range(warm):
            fn(i)
        eng.synchronize(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = eng.launches
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record(ext)
            for i in range(steps):
                fn(warm + i)
            if gather is not None:
                gather.wait(ext)                                         # the last all-gather is inside the timed region
            e1.record(ext)
        eng.synchronize(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.barrier()
        return float(t.item()), eng.launches - l0

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total, launches = timed(step_resident, args.steps, max(3, args.warmup))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(job, args.dump_outputs, V)
    ms_step = ms_total / args.steps
    ms_picture = ms_step / PPS
    value = units_picture_all * PPS / (ms_step * 1e-3)
    launch_t = torch.tensor([launches], dtype=torch.int64, device='cuda')
    if world > 1:
        dist.all_reduce(launch_t)
    launches_all = int(launch_t.item())

    # ------------------------------------------------------------------------------------------- sharded parity (N > 1): gathered tables == single-GPU tables
    extra = {}
    if world > 1:
        idx = (max(3, args.warmup) + args.steps) * PPS
        picture_resident(idx)
        with torch.cuda.stream(ext):
            gather.wait(ext)
        eng.synchronize(); torch.cuda.synchronize(); dist.barrier()
        if rank == 0:
            s = idx % N_PICTURE_SETS
            jobs_all = [job if b == 0 else Job(env, W, band_lists[b], 'band%d' % b) for b in range(world)]
            extra['sharded_parity'] = sharded_parity(env, jobs_all, gather, 2 * s, 2 * s + 1, job)
            if not extra['sharded_parity']['gathered_equals_single_gpu']:
                raise RuntimeError('sharded result tables differ from the single-GPU tables')
            del jobs_all
        dist.barrier()
    n_direct = 1 if world > 1 else 3
    ms_direct, _ = timed(lambda i: step_resident(i, True), n_direct, 1)
    ms_direct /= n_direct

    # ------------------------------------------------------------------------------------------- per-kernel timing + rooflines (rank 0)
    roofline = None
    if rank == 0 and not args.skip_extras:
        def time_launch(fn, reps=10):
            fn(); eng.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(ext):
                e0.record(ext)
                for _ in range(reps):
                    fn()
                e1.record(ext)
            eng.synchronize(); torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps
        kt = {}
        t_search = 0.0; pel_diffs = 0
        ctrp = [0]
        def f_pyr():
            s = ctrp[0] % N_PICTURE_SETS; ctrp[0] += 1
            chk(lib.vvb_sad_search_pyramid_dev(eng.h, 2 * s, 2 * s + 1, nlev, pyr_blocks, pyr_counts, SIZES[0], ctypes.byref(me), nx, nx, pyr_best))
        def f_base():
            s = ctrp[0] % N_PICTURE_SETS; ctrp[0] += 1
            chk(lib.vvb_sad_search_dev(eng.h, 2 * s, 2 * s + 1, P_(d_blocks[SIZES[0]].data_ptr()), len(blocks_np[SIZES[0]]), SIZES[0], SIZES[0], ctypes.byref(me), nx, nx, None, 0,
                                       P_(d_best[SIZES[0]].data_ptr())))
        t_pyr = time_launch(f_pyr, 20); t_base = time_launch(f_base)
        eng.set_pyramid_engine(0); t_pyr_r1 = time_launch(f_pyr); eng.set_pyramid_engine(int(os.environ.get('VVB_PYRAMID', '1') or 1))
        for n in SIZES:
            nb = len(blocks_np[n])
            ctr = [0]
            def f_search(n=n, nb=nb, ctr=ctr):
                s = ctr[0] % N_PICTURE_SETS; ctr[0] += 1
                chk(lib.vvb_sad_search_dev(eng.h, 2 * s, 2 * s + 1, P_(d_blocks[n].data_ptr()), nb, n, n, ctypes.byref(me), nx, nx, None, 0, P_(d_best[n].data_ptr())))
            def f_satd(n=n, nb=nb, ctr=ctr):
                s = ctr[0] % N_PICTURE_SETS; ctr[0] += 1
                chk(lib.vvb_cost_pattern_dev(eng.h, V.DF_HAD, 2 * s, 2 * s + 1, P_(d_blocks[n].data_ptr()), nb, n, n, P_(env['d_pat'].data_ptr()), KP, ctypes.byref(me),
                                             P_(d_satd[n].data_ptr()), None))
            def f_tu(n=n, nb=nb, ctr=ctr):
                s = ctr[0] % N_PICTURE_SETS; ctr[0] += 1
                chk(lib.vvb_fwd_trquant_planes_dev(eng.h, ctypes.byref(tu_par[n]), 2 * s, 2 * s + 1, P_(d_blocks[n].data_ptr()), nb, None, P_(d_q[n].data_ptr()),
                                                   P_(d_sum[n].data_ptr()), P_(d_last[n].data_ptr()), P_(d_nr[n].data_ptr())))
            kt[n] = {'sad_search_ms': time_launch(f_search, 3), 'satd_pattern_ms': time_launch(f_satd), 'trquant_ms': time_launch(f_tu)}
            t_search += kt[n]['sad_search_ms']
            pel_diffs += nb * nx * nx * n * n
        # issue ceiling of the packed-SAD instruction pair: the alu pipe (VIMNMX.S16x2) and the fma pipe (IDP.2A) each take one warp instruction every second
        # cycle per scheduler (B300_MICROARCH.md "fma vs alu split"), so one min + one dot product per pel PAIR = 1 pel difference per lane and cycle at best
        sm_mhz = (clocks or {}).get('sm_max_mhz') or 1965.0
        issue_peak = 148 * 4 * 32 * sm_mhz * 1e6
        ctas, iters = 148 * 8, 4096
        t_probe = time_launch(lambda: chk(lib.vvb_alu_probe_dev(eng.h, ctas, iters, 1)), reps=5)
        alu_probe = ctas * 256 * iters * 16 / (t_probe * 1e-3)
        n0 = SIZES[0]; nb0 = len(blocks_np[n0])
        pyr_bytes = nb0 * (2 * n0 * n0 + 2 * (n0 + 2 * SEARCH_RANGE) ** 2 + 16)            # SURVEY 8d W2: compulsory bytes per block, base level (the only pel pass)
        pyr_pel = nb0 * nx * nx * n0 * n0                                                     # pel differences actually evaluated by the pyramid
        ach_alu = pyr_pel / (t_pyr * 1e-3)
        traffic, traffic_src = ncu_dram_traffic('sad_pyramid8_kernel<4>')
        if traffic is None:
            traffic, traffic_src = ncu_dram_traffic('sad_search_kernel<1, 1, 1>')
            traffic_src = (traffic_src or '') + ' (round-1 kernel; the in-CTA pyramid has no capture in this checkout yet)'
        roofline = {'kernel': 'sad_pyramid8_kernel<4> (vvb_sad_search_pyramid_dev: one CTA per 64x64 root, all four levels on the SM)', 'bound': 'alu',
                    'achieved': ach_alu / 1e12, 'peak': issue_peak / 1e12, 'unit': 'Tpel-diff/s', 'frac': ach_alu / issue_peak,
                    'peak_source': 'issue ceiling 148 SM x 4 schedulers x 32 lanes x %.0f MHz: one VIMNMX.S16x2 (alu pipe) + one IDP.2A (fma pipe) per pel pair, each pipe '
                                   'accepting a warp instruction every 2nd cycle' % sm_mhz,
                    'probe': {'achieved_by_register_only_probe': alu_probe / 1e12, 'frac_of_probe': ach_alu / alu_probe,
                              'note': 'alu_probe_kernel: the same instruction pair on register operands, measured in this run'},
                    'ms_per_launch': t_pyr, 'share_of_step': t_pyr / ms_picture,
                    'traffic': traffic, 'traffic_source': 'dram__bytes_read.sum + dram__bytes_write.sum per launch, ' + str(traffic_src),
                    'hbm': {'achieved': pyr_bytes / (t_pyr * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': pyr_bytes / (t_pyr * 1e-3) / 1e9 / hbm_peak,
                            'peak_source': peak_src, 'bytes': 'compulsory 2N^2 + 2(N+2R)^2 + 16 per 8x8 block (SURVEY 8d W2): small by construction, every reference '
                                                              'pel is re-used up to 4225x from shared memory'},
                    'round1_engine_ms': t_pyr_r1}
        extra['kernel_ms'] = kt
        extra['pyramid_ms'] = t_pyr; extra['pyramid_round1_engine_ms'] = t_pyr_r1; extra['base_level_direct_ms'] = t_base
        extra['direct_search'] = {'ms_per_picture': ms_direct / PPS, 'value': units_picture_all * PPS / (ms_direct * 1e-3), 'search_ms': t_search,
                                  'alu_achieved_Tpel_diff_s': pel_diffs / (t_search * 1e-3) / 1e12, 'alu_frac_of_issue_ceiling': pel_diffs / (t_search * 1e-3) / issue_peak,
                                  'note': 'same step with every block size searched on its own (no SAD pyramid): 4 sad_search launches'}
        # HBM-streaming evidence (SURVEY 8d W1, the ">= 60 % of HBM on the SAD sweep" line): candidate pools >> L2, 2wh + 2wh/K + 8 bytes per candidate
        try:
            Kp = 32
            sweep = {}
            chk(lib.vvb_pool_hint(eng.h, 1))
            for n in SIZES:
                nb = len(blocks_np[n])
                pool = torch.randint(0, 1024, (nb * Kp * n * n,), dtype=torch.int16, device='cuda')
                pos = np.zeros(nb, dtype=V.POS_DT); pos['x'] = blocks_np[n]['x']; pos['y'] = blocks_np[n]['y']
                d_pos = dev(pos); d_out = torch.empty(nb * Kp, dtype=torch.int32, device='cuda')
                for fam, name in ((V.DF_SAD, 'sad'), (V.DF_SSE, 'sse'), (V.DF_HAD, 'satd')):
                    t = time_launch(lambda fam=fam: chk(lib.vvb_dist_pool_dev(eng.h, fam, 0, P_(d_pos.data_ptr()), nb, n, n, Kp, P_(pool.data_ptr()), 0, P_(d_out.data_ptr()))), reps=5)
                    byt = nb * Kp * (2 * n * n + 2 * n * n / Kp + 8)
                    sweep['%s_%dx%d' % (name, n, n)] = {'ms': t, 'GBps': byt / (t * 1e-3) / 1e9, 'frac_hbm': byt / (t * 1e-3) / 1e9 / hbm_peak, 'cand_per_s': nb * Kp / (t * 1e-3)}
                del pool, d_out
            roofline['w1_hbm_sweep'] = {'bound': 'hbm', 'peak': hbm_peak, 'unit': 'GB/s', 'peak_source': peak_src, 'K': Kp, 'pool_MB_per_size': nb0 * Kp * n0 * n0 * 2 / 1e6,
                                        'bytes': '2wh + 2wh/K + 8 per candidate (SURVEY 8d W1)', 'frac': sweep['sad_16x16']['frac_hbm'],
                                        'frac_min_sad': min(v['frac_hbm'] for k, v in sweep.items() if k.startswith('sad')), **sweep}
        except Exception as ex:     # the sweep is evidence, not part of the metric
            roofline['w1_hbm_sweep'] = {'error': str(ex)}
        # TU round trip (SURVEY 8f-1: residual -> transform -> quant -> dequant -> inverse -> reconstruct -> SSE in one kernel) over candidate pools >> L2;
        # algorithmic bytes per TU = 2wh (org) + 2wh (pred) + 2wh (levels out) + 2wh (reco out) + 32 (result record)
        try:
            rt = {}
            for n in SIZES:
                ntu = (512 << 20) // (8 * n * n)                                   # 4 x 128 MB of pel data per launch
                d_o = torch.randint(0, 1024, (ntu * n * n,), dtype=torch.int16, device='cuda')
                d_p = (d_o + torch.randint(-200, 201, (ntu * n * n,), dtype=torch.int16, device='cuda')).clamp_(0, 1023)
                d_lv = torch.empty(ntu * n * n, dtype=torch.int16, device='cuda'); d_rc = torch.empty(ntu * n * n, dtype=torch.int16, device='cuda')
                d_rs = torch.empty(ntu * 32, dtype=torch.uint8, device='cuda')
                torch.cuda.synchronize()
                t = time_launch(lambda: chk(lib.vvb_tu_roundtrip_dev(eng.h, ctypes.byref(tu_par[n]), P_(d_o.data_ptr()), P_(d_p.data_ptr()), ntu, P_(d_lv.data_ptr()),
                                                                     P_(d_rc.data_ptr()), P_(d_rs.data_ptr()), None)), reps=3)
                byt = ntu * (8 * n * n + 32)
                nz = int((torch.frombuffer(bytearray(d_rs.cpu().numpy().tobytes()), dtype=torch.int32).view(-1, 8)[:, 6] > 0).sum())
                rt[str(n)] = {'ms': t, 'tus': ntu, 'tu_per_s': ntu / (t * 1e-3), 'GBps': byt / (t * 1e-3) / 1e9, 'frac_hbm': byt / (t * 1e-3) / 1e9 / hbm_peak, 'nonzero_tus': nz}
                del d_o, d_p, d_lv, d_rc, d_rs
            extra['tu_roundtrip_pool'] = rt
        except Exception as ex:
            extra['tu_roundtrip_pool'] = {'error': str(ex)}
        # W4 at scale (SURVEY 8d): forward transform + quantiser alone and the inverse path alone over the same kind of pools
        #   fwd bytes per TU = 2wh (Pel in) + 2wh (TCoeffSig out) + 9 ; inv bytes per TU = 2wh + 2wh
        try:
            tq = {}
            for n in SIZES:
                ntu = (256 << 20) // (4 * n * n)
                d_r = torch.randint(-200, 201, (ntu * n * n,), dtype=torch.int16, device='cuda')
                d_lv = torch.empty(ntu * n * n, dtype=torch.int16, device='cuda'); d_rc = torch.empty(ntu * n * n, dtype=torch.int16, device='cuda')
                d_s = torch.empty(ntu, dtype=torch.int32, device='cuda'); d_l = torch.empty(ntu, dtype=torch.int32, device='cuda'); d_n = torch.empty(ntu, dtype=torch.uint8, device='cuda')
                torch.cuda.synchronize()
                tf = time_launch(lambda: chk(lib.vvb_fwd_trquant_dev(eng.h, ctypes.byref(tu_par[n]), P_(d_r.data_ptr()), ntu, None, P_(d_lv.data_ptr()), P_(d_s.data_ptr()),
                                                                     P_(d_l.data_ptr()), P_(d_n.data_ptr()))), reps=3)
                ti = time_launch(lambda: chk(lib.vvb_inv_trquant_dev(eng.h, ctypes.byref(tu_par[n]), P_(d_lv.data_ptr()), ntu, P_(d_rc.data_ptr()))), reps=3)
                bf = ntu * (4 * n * n + 9); bi = ntu * 4 * n * n
                tq[str(n)] = {'tus': ntu, 'fwd_ms': tf, 'fwd_GBps': bf / (tf * 1e-3) / 1e9, 'fwd_frac_hbm': bf / (tf * 1e-3) / 1e9 / hbm_peak, 'fwd_tu_per_s': ntu / (tf * 1e-3),
                              'inv_ms': ti, 'inv_GBps': bi / (ti * 1e-3) / 1e9, 'inv_frac_hbm': bi / (ti * 1e-3) / 1e9 / hbm_peak}
                del d_r, d_lv, d_rc
            extra['trquant_pool'] = tq
            roofline['w4_trquant'] = {'bound': 'hbm', 'bytes': '2wh + 2wh + 9 per TU (SURVEY 8d W4)', **{'fwd_frac_%s' % k: v['fwd_frac_hbm'] for k, v in tq.items()}}
        except Exception as ex:
            extra['trquant_pool'] = {'error': str(ex)}
        # W5 (SURVEY 8d): MCTF block matching, final-level shape -- every 16x16 block of the picture against one neighbour frame, 49 quarter-step
        # candidates (7x7 around the integer vector, 6-tap 1/16-pel filters) as MCTF::estimateLumaLn's doubleRes refinement evaluates (MCTF.cpp:1245-1287)
        try:
            B = 16
            xs = np.arange(0, W - B + 1, B); ys = np.arange(0, H - B + 1, B)
            gx, gy = np.meshgrid(xs, ys)
            off = np.array([(dx, dy) for dy in range(-12, 13, 4) for dx in range(-12, 13, 4)], dtype=np.int32)
            nbk = gx.size; K5 = len(off)
            c5 = np.zeros(nbk * K5, dtype=V.MCTF_DT)
            c5['x'] = np.repeat(gx.reshape(-1), K5); c5['y'] = np.repeat(gy.reshape(-1), K5)
            c5['mvx'] = np.tile(off[:, 0], nbk) + 16 * 2; c5['mvy'] = np.tile(off[:, 1], nbk) - 16
            c5['w'] = B; c5['h'] = B
            d_c5 = dev(c5); d_e5 = torch.empty(nbk * K5, dtype=torch.int32, device='cuda')
            chk(lib.vvb_mctf_hint(eng.h, B))
            t5 = time_launch(lambda: chk(lib.vvb_mctf_error_batch_dev(eng.h, 0, 1, P_(d_c5.data_ptr()), nbk * K5, 0, P_(d_e5.data_ptr()))), reps=5)
            byt = nbk * (2 * B * B + 2 * (B + 2 * 1 + 6) ** 2 + 16)
            # the same 49 vectors through the grid-search entry point (window staged once per block, horizontal pass shared per column of the grid)
            b5 = np.zeros(nbk, dtype=V.MCTF_DT)
            b5['x'] = gx.reshape(-1); b5['y'] = gy.reshape(-1); b5['mvx'] = 32; b5['mvy'] = -16; b5['w'] = B; b5['h'] = B
            d_b5 = dev(b5); d_g5 = torch.empty(nbk * K5, dtype=torch.int32, device='cuda')
            tg = time_launch(lambda: chk(lib.vvb_mctf_search_grid_dev(eng.h, 0, 1, P_(d_b5.data_ptr()), nbk, 4, 3, 0, P_(d_g5.data_ptr()))), reps=5)
            same = bool(torch.equal(d_g5.view(nbk, K5), d_e5.view(nbk, K5)))
            extra['mctf_grid_16x16'] = {'blocks': int(nbk), 'step': 4, 'radius': 3, 'ms': tg, 'cand_per_s': nbk * K5 / (tg * 1e-3), 'block_refs_per_s': nbk / (tg * 1e-3),
                                        'GBps_w5_formula': byt / (tg * 1e-3) / 1e9, 'frac_hbm_w5_formula': byt / (tg * 1e-3) / 1e9 / hbm_peak, 'equals_candidate_list': same}
            extra['mctf_match_16x16'] = {'blocks': int(nbk), 'candidates_per_block': K5, 'ms': t5, 'cand_per_s': nbk * K5 / (t5 * 1e-3), 'block_refs_per_s': nbk / (t5 * 1e-3),
                                         'GBps_w5_formula': byt / (t5 * 1e-3) / 1e9, 'frac_hbm_w5_formula': byt / (t5 * 1e-3) / 1e9 / hbm_peak,
                                         'note': 'fractional candidates: separable 6-tap filtering per candidate (ALU-bound by construction, SURVEY 8d W5)'}
        except Exception as ex:
            extra['mctf_match_16x16'] = {'error': str(ex)}
        # fractional-pel refinement grid (SURVEY 8f-2): every block of the picture, SATD at all 49 quarter-pel offsets around the best integer vector
        try:
            fr = {}
            for n in (8, 16, 32):
                nb = len(blocks_np[n])
                d_ft = torch.empty(nb * 49, dtype=torch.int32, device='cuda')
                tf_ = time_launch(lambda: chk(lib.vvb_frac_cost_grid_dev(eng.h, V.DF_HAD, 0, 1, P_(d_blocks[n].data_ptr()), nb, n, n, 2, 0, P_(d_ft.data_ptr()))), reps=5)
                byt = nb * (2 * n * n + 2 * (n + 8) ** 2 + 49 * 4)
                fr[str(n)] = {'blocks': nb, 'ms': tf_, 'cand_per_s': nb * 49 / (tf_ * 1e-3), 'GBps': byt / (tf_ * 1e-3) / 1e9, 'frac_hbm': byt / (tf_ * 1e-3) / 1e9 / hbm_peak}
            fr['bytes_formula'] = 'per block: 2 N^2 original + 2 (N+8)^2 window + 196 table; ALU-bound by construction (two 8-tap passes + 8x8 Hadamard per candidate)'
            extra['frac_satd_grid'] = fr
        except Exception as ex:
            extra['frac_satd_grid'] = {'error': str(ex)}
        # MCTF apply stage (SURVEY 8f-3): the whole 3840x2160 luma picture filtered against 8 neighbour pictures, unit 16 (xFinalizeBlkLine per block)
        try:
            from vvenc_b200 import _lib as VL
            B = 16; nrefs = 8
            nbk = (W // B) * (HT // B)
            rs_ = np.random.RandomState(5)
            mv = np.zeros((nrefs, nbk), dtype=V.MCTF_MV_DT)
            mv['x'] = rs_.randint(-40, 41, size=(nrefs, nbk)); mv['y'] = rs_.randint(-40, 41, size=(nrefs, nbk))
            mv['error'] = rs_.randint(5, 150, size=(nrefs, nbk)); mv['rmsme'] = rs_.randint(0, 30, size=(nrefs, nbk))
            d_mv = dev(mv)
            apar = VL.vvb_mctf_apply_par()
            apar.num_refs = nrefs; apar.block_size = B; apar.low_res_filter = 0; apar.planar_correction = 1; apar.weight_scaling = 0.4; apar.sigma_sq = 9 * (128.0 + 3.0 / 256.0 * 32 ** 3)
            for i_, (pl, st) in enumerate(zip([1, 3, 5, 7, 2, 4, 6, 1], [0.85, 0.57, 0.41, 0.33, 0.30, 0.20, 0.18, 0.15])):
                apar.ref_plane[i_] = pl; apar.ref_strength[i_] = st
            d_flt = torch.empty(W * HT, dtype=torch.int16, device='cuda')
            ta = time_launch(lambda: chk(lib.vvb_mctf_apply_dev(eng.h, 0, ctypes.byref(apar), P_(d_mv.data_ptr()), P_(d_flt.data_ptr()), W)), reps=5)
            byt = nbk * (nrefs * (2 * (B + 5) ** 2 + 16) + 4 * B * B)
            extra['mctf_apply_2160p'] = {'blocks': int(nbk), 'refs': nrefs, 'unit': B, 'ms': ta, 'pels_per_s': W * HT / (ta * 1e-3), 'block_refs_per_s': nbk * nrefs / (ta * 1e-3),
                                         'GBps': byt / (ta * 1e-3) / 1e9, 'frac_hbm': byt / (ta * 1e-3) / 1e9 / hbm_peak,
                                         'bytes_formula': 'per block: refs * (2 (B+5)^2 window + 16 vector) + 2 B^2 original + 2 B^2 filtered'}
            del d_flt
        except Exception as ex:
            extra['mctf_apply_2160p'] = {'error': str(ex)}
        # MCTF motion search (SURVEY a5, BASELINE configs[3] shape): motionEstimationMCTF of one 2160p neighbour picture with the control on the device --
        # subsampled pyramids, 5 chained levels, selection chains and the upper / left neighbour wavefront without the host seeing a number
        try:
            from vvenc_b200 import _lib as VL
            o_, r_, S_ = host_sets[0]
            pad = 128
            po = np.ascontiguousarray(np.pad(o_[MARGIN:MARGIN + H, MARGIN:MARGIN + W], pad, mode='edge')); pr_ = np.ascontiguousarray(np.pad(r_[MARGIN:MARGIN + H, MARGIN:MARGIN + W], pad, mode='edge'))
            eng.upload_plane(60, po, W, H, pad); eng.upload_plane(61, pr_, W, H, pad)
            fh_, fw_ = (H + 15) // 16, (W + 15) // 16
            d_field = torch.zeros(fh_ * fw_ * 4, dtype=torch.int32, device='cuda')
            ppar = VL.vvb_mctf_pyr_par(16, 1, 0, 0)
            l0 = eng.launches
            tm = time_launch(lambda: chk(lib.vvb_mctf_estimate_pyramid_dev(eng.h, 60, 61, ctypes.byref(ppar), P_(d_field.data_ptr()))), reps=4)
            nl = (eng.launches - l0) // 5
            fld = d_field.cpu().numpy().reshape(fh_, fw_, 4)
            extra['mctf_motion_estimation_2160p'] = {'unit': 16, 'levels': 5, 'ms_per_neighbour_picture': tm, 'launches_per_neighbour_picture': int(nl), 'blocks': int(fh_ * fw_),
                                                     'block_refs_per_s': fh_ * fw_ / (tm * 1e-3), 'pels_per_s': W * H / (tm * 1e-3),
                                                     'nonzero_vectors': int(((fld[..., 0] != 0) | (fld[..., 1] != 0)).sum()), 'fractional_vectors': int((((fld[..., 0] | fld[..., 1]) & 15) != 0).sum())}
            eng.free_plane(60); eng.free_plane(61); del d_field
        except Exception as ex:
            extra['mctf_motion_estimation_2160p'] = {'error': str(ex)}
        # fixed diamond-search candidate set (SURVEY 8d W3 -> W1 byte formula): TZ point pattern, range 64, around the zero vector
        try:
            from vvenc_b200 import candidates as cand
            tz = cand.tz_diamond_pattern(64)
            d_tz = dev(tz); Kt = len(tz); dia = {}
            for n in (8, 16, 32, 64):
                nb = len(blocks_np[n])
                bb = blocks_np[n].copy(); bb['left'] = -64; bb['right'] = 64; bb['top'] = -64; bb['bottom'] = 64
                d_bb = dev(bb); d_s = torch.empty(nb * Kt, dtype=torch.int32, device='cuda'); d_b = torch.empty(nb * 16, dtype=torch.uint8, device='cuda')
                t = time_launch(lambda: chk(lib.vvb_sad_pattern_dev(eng.h, 0, 1, P_(d_bb.data_ptr()), nb, n, n, P_(d_tz.data_ptr()), Kt, ctypes.byref(me),
                                                                    P_(d_s.data_ptr()), P_(d_b.data_ptr()))), reps=5)
                byt = nb * Kt * (2 * n * n + 2 * n * n / Kt + 8)
                dia[str(n)] = {'ms': t, 'cand_per_s': nb * Kt / (t * 1e-3), 'GBps_w1_formula': byt / (t * 1e-3) / 1e9, 'frac_hbm_w1_formula': byt / (t * 1e-3) / 1e9 / hbm_peak}
            extra['diamond_set_sad'] = {'points': Kt, 'range': 64, 'note': 'candidates overlap in the L2-resident reference plane: the W1 byte formula counts every candidate block '
                                        'as fresh bytes, so fractions above 1.0 mean L2 hits, not missing work (DRAM traffic in profiles/)', **dia}
        except Exception as ex:
            extra['diamond_set_sad'] = {'error': str(ex)}
        # fast RDOQ (SURVEY 8f-4, QuantRDOQ2::xRateDistOptQuantFast, what Quant::m_RDOQ == 2 of the presets faster / fast runs): one TU per thread, bound by the serial
        # chain of a TU, so the row holds one picture's worth of TUs per launch and sixteen; the CPU row is the same text compiled by g++ on ONE host thread
        try:
            from vvenc_b200 import _lib as VL
            sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'tests'))
            from _libs import dq_oracle, P as P_np
            g6 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'tests', 'golden', 'golden_v6_rdoq.npz'))
            rates_flat = np.ascontiguousarray(g6['rates'][[i for i, r in enumerate(g6['cases']) if int(r[7]) == 0][3]])
            rates = eng.rdoq_rates(rates_flat)
            rsq = np.random.RandomState(1); rq_rows = {}
            for n in (8, 16, 32, 64):
                cnt = (W // n) * (H // n)
                scale = rsq.choice([3, 10, 40, 150, 600], size=(cnt, 1, 1))
                coef = rsq.laplace(0, 1.0, size=(cnt, n, n)) * scale * (1.0 / (1 + np.add.outer(np.arange(n), np.arange(n))) ** 0.7)
                coef = np.clip(coef, -32768, 32767).astype(np.int32); coef[:, :, 32:] = 0; coef[:, 32:, :] = 0
                par = eng.tu_par(n, n, 0, 0, BITDEPTH, QP, sign_hiding=True); rqp = VL.vvb_rdoq_par(57.3, 8, 0)
                row = {'tus': int(cnt)}
                for mult in (1, 16):
                    d_c = torch.from_numpy(coef).cuda().repeat(mult, 1, 1); d_rq = torch.zeros((cnt * mult, n, n), dtype=torch.int16, device='cuda')
                    d_s = torch.zeros(cnt * mult, dtype=torch.int32, device='cuda'); d_l = torch.zeros(cnt * mult, dtype=torch.int32, device='cuda')
                    t = time_launch(lambda: chk(lib.vvb_rdoq_dev(eng.h, ctypes.byref(par), ctypes.byref(rqp), ctypes.byref(rates), P_(d_c.data_ptr()), None, cnt * mult,
                                                                 P_(d_rq.data_ptr()), P_(d_s.data_ptr()), P_(d_l.data_ptr()))), reps=3)
                    row['ms_per_picture' if mult == 1 else 'ms_per_picture_at_16_pictures'] = t / mult
                    if mult == 1:
                        q_dev = d_rq.cpu().numpy(); l_dev = d_l.cpu().numpy()
                    del d_c, d_rq, d_s, d_l
                qq = np.zeros((cnt, n, n), dtype=np.int16); ss = np.zeros(cnt, dtype=np.int32); ll = np.zeros(cnt, dtype=np.int32)
                t0 = time.perf_counter()
                dq_oracle().orc_rdoq(n, n, BITDEPTH, QP, 0, 0, 0, 1, 57.3, 8, P_np(rates_flat), P_np(coef), cnt, P_np(qq), P_np(ss), P_np(ll))
                row['cpu_port_ms_per_picture_1thread'] = (time.perf_counter() - t0) * 1e3
                # ... and on all usable host CPUs (the C call releases the GIL; the TU list is cut into one chunk per thread)
                from concurrent.futures import ThreadPoolExecutor
                nthr, _ = host_cpus()
                cuts = [cnt * k // nthr for k in range(nthr + 1)]
                def port_chunk(k):
                    a, b = cuts[k], cuts[k + 1]
                    if b > a:
                        dq_oracle().orc_rdoq(n, n, BITDEPTH, QP, 0, 0, 0, 1, 57.3, 8, P_np(rates_flat), P_np(coef[a:b]), b - a, P_np(qq[a:b]), P_np(ss[a:b]), P_np(ll[a:b]))
                with ThreadPoolExecutor(nthr) as ex:
                    t0 = time.perf_counter()
                    list(ex.map(port_chunk, range(nthr)))
                    row['cpu_port_ms_per_picture_all_threads'] = (time.perf_counter() - t0) * 1e3
                row['cpu_threads'] = int(nthr)
                row['device_equals_port'] = bool(np.array_equal(q_dev, qq) and np.array_equal(l_dev, ll))
                row['coded_tus'] = int((ll >= 0).sum())
                rq_rows[str(n)] = row
            extra['rdoq_2160p'] = rq_rows
        except Exception as ex:
            extra['rdoq_2160p'] = {'error': str(ex)}

    # ------------------------------------------------------------------------------------------- BASELINE configs[4]: 4320p, strong scaling + parity
    if (world > 1 or args.strong) and not args.skip_extras:
        try:
            r = strong_4320p(env, rank, world)
            if rank == 0:
                extra['strong_4320p'] = r
        except Exception as ex:
            if rank == 0:
                extra['strong_4320p'] = {'error': repr(ex)}
            raise

    # ------------------------------------------------------------------------------------------- end-to-end through the host-buffer C ABI
    e2e = None
    if not args.skip_e2e:
        # NCTX contexts, each driven by its own host thread (as encoder workers would, EncSlice.cpp:142-147), take the pictures in turn; the GPU overlaps
        # one worker's uploads / downloads with the other workers' kernels.  Every picture still uploads its own planes and downloads all of its results
        # inside the timed region.  (N > 1: every rank uploads the 3840x2160 window of its band -- band rows plus the search margin.)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
        y0b = rows[rank][0]
        h_planes = []
        for (org, ref, S) in host_sets:
            # the band's rows of the tall picture, with margins: for world == 1 this is the picture itself
            torg = tall_picture(org, world); tref = tall_picture(ref, world)
            hb_rows = rows[rank][1] - rows[rank][0]
            po = pin((hb_rows + 2 * MARGIN, S), torch.int16); pr = pin((hb_rows + 2 * MARGIN, S), torch.int16)
            po[:] = torg[y0b:y0b + hb_rows + 2 * MARGIN]; pr[:] = tref[y0b:y0b + hb_rows + 2 * MARGIN]
            h_planes.append((po, pr, S, hb_rows))
            del torg, tref
        NCTX = int(os.environ.get('VVB_E2E_CTX', '4'))
        engs = [eng] + [V.CostEngine(local) for _ in range(NCTX - 1)]
        for e in engs:
            e.set_async(True)
            if os.environ.get('VVB_PYRAMID', '') != '':
                e.set_pyramid_engine(int(os.environ['VVB_PYRAMID']))
        PA = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        hb = []
        for c in range(NCTX):
            d = dict(blocks={n: pin((len(blocks_np[n]) * 24,), torch.uint8) for n in SIZES}, best={n: pin((len(blocks_np[n]) * 16,), torch.uint8) for n in SIZES},
                     satd={n: pin((len(blocks_np[n]) * KP,), torch.int32) for n in SIZES}, q={n: pin((len(blocks_np[n]) * n * n,), torch.int16) for n in SIZES},
                     sum={n: pin((len(blocks_np[n]),), torch.int32) for n in SIZES}, last={n: pin((len(blocks_np[n]),), torch.int32) for n in SIZES},
                     nr={n: pin((len(blocks_np[n]),), torch.uint8) for n in SIZES}, off={n: pin((len(blocks_np[n]) + 1,), torch.int32) for n in SIZES})
            for n in SIZES:
                bl = blocks_np[n].copy(); bl['y'] -= y0b                              # the uploaded plane starts at the band's first row
                d['blocks'][n][:] = np.frombuffer(bl.tobytes(), dtype=np.uint8)
            d['pyr_blocks'] = (ctypes.c_void_p * nlev)(*[d['blocks'][n].ctypes.data for n in SIZES])
            d['pyr_best'] = (ctypes.c_void_p * nlev)(*[d['best'][n].ctypes.data for n in SIZES])
            hb.append(d)
        h_pat = pin((KP * 4,), torch.uint8); h_pat[:] = np.frombuffer(pat_np.tobytes(), dtype=np.uint8)
        E0, E1 = 40, 41        # plane ids of the uploaded pictures
        PACKED = os.environ.get('VVB_E2E_PACKED', '1') == '1'    # levels come back trimmed to lastPos, written by the device straight into the pinned buffer
        h2d = 0; d2h = 0
        for n in SIZES:
            nb = len(blocks_np[n])
            h2d += nb * 24 + KP * 4
            d2h += nb * 16 + nb * KP * 4 + nb * 9 + ((nb + 1) * 4 if PACKED else nb * n * n * 2)      # + the packed levels themselves, counted after the run
        S0 = host_sets[0][2]
        h2d += 2 * (h_planes[0][3] + 2 * MARGIN) * S0 * 2

        def e2e_upload(i):
            c = i % NCTX
            e = engs[c]
            po, pr, S, hbr = h_planes[i % N_PICTURE_SETS]
            base = MARGIN * S + MARGIN
            chk(lib.vvb_plane_upload(e.h, E0, ctypes.c_void_p(po.ctypes.data + base * 2), S, W, hbr, MARGIN, BITDEPTH))
            chk(lib.vvb_plane_upload(e.h, E1, ctypes.c_void_p(pr.ctypes.data + base * 2), S, W, hbr, MARGIN, BITDEPTH))

        import vvenc_b200._lib as VL
        ios = []
        for c in range(NCTX):
            arr = (VL.vvb_level_io * nlev)()
            for l, n in enumerate(SIZES):
                d = hb[c]
                arr[l].blocks = d['blocks'][n].ctypes.data; arr[l].count = len(blocks_np[n]); arr[l].best = d['best'][n].ctypes.data
                arr[l].refine_cost = d['satd'][n].ctypes.data
                if PACKED:
                    arr[l].packed_q = d['q'][n].ctypes.data; arr[l].packed_offsets = d['off'][n].ctypes.data
                else:
                    arr[l].q = d['q'][n].ctypes.data
                arr[l].abs_sum = d['sum'][n].ctypes.data; arr[l].last_pos = d['last'][n].ctypes.data; arr[l].need_rdoq = d['nr'][n].ctypes.data
                arr[l].tu = tu_par[n]
            ios.append(arr)

        def e2e_chain(i):
            # one call: block lists up, search -> start = best (on the device) -> SATD ring -> TU, every result down; nothing returns to the host in between
            c = i % NCTX
            chk(lib.vvb_search_refine_tu(engs[c].h, E0, E1, nlev, ios[c], SIZES[0], ctypes.byref(me), nx, nx, V.DF_HAD, PA(h_pat), KP))

        def run_e2e(first, count):
            # one host thread per context, as one encoder worker per context would run (EncSlice.cpp:142-147; ctypes releases the GIL inside the library):
            # worker c takes the pictures first+c, first+c+NCTX, ... and runs each of them upload -> chained search / refinement / TU call -> wait for the
            # downloads; the GPU overlaps one worker's copies with the other workers' kernels
            errs = []
            def worker(c):
                try:
                    pc = time.perf_counter
                    for i in range(first + c, first + count, NCTX):
                        t = pc(); e2e_upload(i); e2e_chain(i); host_ms['upload_and_enqueue'] += pc() - t
                        t = pc(); chk(lib.vvb_synchronize(engs[i % NCTX].h)); host_ms['wait_results'] += pc() - t
                except Exception as ex:
                    errs.append(ex)
            th = [threading.Thread(target=worker, args=(c,)) for c in range(NCTX)]
            for t_ in th: t_.start()
            for t_ in th: t_.join()
            if errs:
                raise errs[0]

        host_ms = {k: 0.0 for k in ('upload_and_enqueue', 'wait_results')}
        ke_steps = max(2, min(args.steps, 5))
        ke = ke_steps * PPS // NCTX * NCTX                   # pictures inside the timed region
        run_e2e(0, 2 * NCTX)
        host_ms = {k: 0.0 for k in host_ms}
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        run_e2e(2 * NCTX, ke)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / ke                 # seconds per picture
        t = torch.tensor([dt], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        e2e = {'value': units_picture_all / dt, 'unit': 'candidate-blocks/s', 'h2d_bytes_per_step': int(h2d) * PPS, 'd2h_bytes_per_step': int(d2h) * PPS,
               'h2d_bytes_per_picture': int(h2d), 'd2h_bytes_per_picture': int(d2h), 'ms_per_step': dt * 1e3 * PPS, 'ms_per_picture': dt * 1e3,
               'steps': ke / PPS, 'pictures': ke, 'contexts': NCTX, 'worker_ms_per_picture': {k: v * 1e3 / ke for k, v in host_ms.items()},
               'timing': 'host wall clock over %d pictures (%.1f steps) issued through the host-buffer C ABI (vvb_plane_upload x2 + vvb_search_refine_tu per picture) from pinned memory '
                         'by %d worker threads, one asynchronous context each; every upload and download is inside the timed region; max over ranks' % (ke, ke / PPS, NCTX)}
        last = 2 * NCTX + ke - 1                               # index of the last picture issued
        if PACKED:
            packed_bytes = sum(int(hb[last % NCTX]['off'][n][len(blocks_np[n])]) * 2 for n in SIZES)
            d2h += packed_bytes
            e2e['d2h_bytes_per_picture'] = int(d2h); e2e['d2h_bytes_per_step'] = int(d2h) * PPS
            e2e['levels'] = {'form': 'trimmed to lastPos, scan order, written by the device into the pinned buffer (vvb_level_io.packed_q)', 'bytes_per_picture': packed_bytes,
                             'untrimmed_bytes_per_picture': sum(len(blocks_np[n]) * n * n * 2 for n in SIZES)}
        for e in engs:
            e.set_async(False)
        for e in engs[1:]:
            e.close()
        # raw PCIe copy rates of this box (pinned, 64 MB, each direction alone and both together): the floor under any host-buffer path
        try:
            hp = torch.empty(64 << 20, dtype=torch.uint8).pin_memory(); hp2 = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
            dp = torch.empty(64 << 20, dtype=torch.uint8, device='cuda'); dp2 = torch.empty(64 << 20, dtype=torch.uint8, device='cuda')
            s1 = torch.cuda.Stream(); s2 = torch.cuda.Stream()
            def rate(fn, nbytes):
                fn(); torch.cuda.synchronize()
                t_ = time.perf_counter()
                for _ in range(4): fn()
                torch.cuda.synchronize()
                return nbytes * 4 / (time.perf_counter() - t_) / 1e9
            def f_h2d():
                with torch.cuda.stream(s1): dp.copy_(hp, non_blocking=True)
            def f_d2h():
                with torch.cuda.stream(s2): hp2.copy_(dp2, non_blocking=True)
            def f_both():
                f_h2d(); f_d2h()
            extra['pcie_GBps'] = {'h2d': rate(f_h2d, 64 << 20), 'd2h': rate(f_d2h, 64 << 20), 'both_directions_sum': rate(f_both, 128 << 20)}
            extra['pcie_GBps']['e2e_floor_ms_per_picture'] = max(h2d, d2h) / 1e6 / min(extra['pcie_GBps']['h2d'], extra['pcie_GBps']['d2h'])
            del hp, hp2, dp, dp2
        except Exception as ex:
            extra['pcie_GBps'] = {'error': str(ex)}
        # parity check of what came back: replay the last e2e picture (same picture set) on the device-resident path and compare every best vector / cost
        # and every TU's level sum bit for bit
        job.run(env, 2 * (last % N_PICTURE_SETS), 2 * (last % N_PICTURE_SETS) + 1)
        eng.synchronize(); torch.cuda.synchronize()
        hl = hb[last % NCTX]
        ok = True
        for n in SIZES:
            nb = len(blocks_np[n])
            ok = ok and np.array_equal(np.frombuffer(d_best[n][:nb * 16].cpu().numpy().tobytes(), dtype=np.uint8), hl['best'][n])
            ok = ok and np.array_equal(d_sum[n][:nb].cpu().numpy(), hl['sum'][n])
            if PACKED:
                so = np.zeros(min(n, 32) ** 2, dtype=np.int32)
                chk(lib.vvb_scan_order(n, n, so.ctypes.data_as(ctypes.c_void_p)))
                off = hl['off'][n].astype(np.int64); lens = np.maximum(hl['last'][n].astype(np.int64) + 1, 0)
                ok = ok and np.array_equal(np.diff(off), lens)
                tot = int(off[nb])
                full = np.zeros((nb, n * n), dtype=np.int16)
                tu_idx = np.repeat(np.arange(nb), lens); pos = np.arange(tot) - np.repeat(off[:nb], lens)
                full[tu_idx, so[pos]] = hl['q'][n][:tot]
                ok = ok and np.array_equal(d_q[n][:nb * n * n].cpu().numpy().reshape(nb, n * n), full)
            else:
                ok = ok and np.array_equal(d_q[n][:nb * n * n].cpu().numpy().reshape(-1), hl['q'][n])
        extra['e2e_matches_resident'] = bool(ok)

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cpu = cpu_arm(args.cpu_budget)
        try:
            extra['cpu_rows'] = cpu_rows(threads=cpu['cores'])
            cr = extra['cpu_rows']; sp = {}
            # GPU (resident) rate over the reference's all-threads rate, same unit per row; informational -- the headline ratio is e2e over the --impl reference arm
            for n in SIZES:
                g = extra.get('tu_roundtrip_pool', {}).get(str(n), {}).get('tu_per_s'); c = cr.get('tu_roundtrip', {}).get(str(n), {}).get('tu_per_s')
                if g and c:
                    sp['tu_roundtrip_%d' % n] = g / c
            g = extra.get('mctf_grid_16x16', {}).get('cand_per_s'); c = cr.get('mctf_match_16x16', {}).get('cand_per_s')
            if g and c:
                sp['mctf_grid_16x16'] = g / c
            for n in (8, 16, 32):
                g = extra.get('frac_satd_grid', {}).get(str(n), {}).get('cand_per_s'); c = cr.get('frac_satd_grid', {}).get(str(n), {}).get('cand_per_s')
                if g and c:
                    sp['frac_satd_grid_%d' % n] = g / c
            g = extra.get('mctf_apply_2160p', {}).get('pels_per_s'); c = cr.get('mctf_apply', {}).get('pels_per_s')
            if g and c:
                sp['mctf_apply'] = g / c
            g = extra.get('mctf_motion_estimation_2160p', {}).get('pels_per_s'); c = cr.get('mctf_motion_estimation', {}).get('pels_per_s_if_all_threads_scaled')
            if g and c:
                sp['mctf_motion_estimation_vs_all_threads_scaled'] = g / c
            extra['row_speedup_vs_cpu'] = sp
        except Exception as ex:
            extra['cpu_rows'] = {'error': str(ex)}

    if rank == 0:
        line = {'metric': 'candidate-blocks/s (SAD+SATD+DCT-quant) on 2160p10', 'value': value, 'unit': 'candidate-blocks/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'int16 pels / int32 accumulation (exact)', 'data': 'synthetic', 'config': config, 'roofline': roofline,
                'cpu_baseline': None if cpu is None else {k: cpu[k] for k in ('value', 'unit', 'cores', 'kind', 'sample', 'value_per_thread', 'host', 'thread_sweep')},
                'e2e': e2e, 'clocks': clocks, 'gpu_launches': launches_all, 'ms_per_picture': ms_picture, 'timed_region_s': ms_total * 1e-3, 'extra': extra}
        if cpu is not None:
            line['extra']['cpu_s_per_picture'] = cpu['cpu_s_per_picture']; line['extra']['cpu_legs'] = cpu['legs']
            line['extra']['cpu_search_cpu_seconds_per_wall_second'] = cpu['search_cpu_seconds_per_wall_second']
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    eng.close()
    return 0


if __name__ == '__main__':
    sys.exit(main())
