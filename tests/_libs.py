"""ctypes loaders shared by the tests: the CPU oracle (oracle/_build/liboracle.so), the optional reference
probe (oracle/_ref/libvvenc_refshim.so, only where the reference sources were available to build it) and the product
C-ABI library (vvenc_b200/csrc/libvvenc_b200.so).

Where the probe is absent, refshim() answers from tests/golden/refshim/<module>.npz: the probe calls a test module made,
recorded on a machine that had the probe (VVB_RECORD_REFSHIM=1 python -m pytest tests/<module>.py; a partial run updates
only the tests it ran).  Every recorded call carries a digest of its inputs, its return value and the small outputs it
wrote (by-reference scalars, arrays up to SMALL_OUTPUT bytes); larger output arrays are kept for a fixed, seeded sample
of the calls: the first calls in an order seeded by the test id, as many as TEST_BUDGET compressed bytes allow, at least two.  Replay checks each digest, then writes what was recorded
into the caller's buffers; answered(a, ...) tells a test whether the reference's values of those arrays were written,
so it compares large outputs on the sampled calls and everything else on every call."""
import atexit, ctypes, hashlib, json, os, subprocess, weakref, zlib
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
c_i16p = ctypes.c_void_p
RECORDINGS = os.path.join(ROOT, 'tests', 'golden', 'refshim')
SMALL_OUTPUT = 16
TEST_BUDGET = 1500


class _ArrayPtr(ctypes.c_void_p):
    """a c_void_p that remembers the numpy array it points into (the refshim recorder reads and writes through it)"""


def P(a):
    p = _ArrayPtr(a.ctypes.data)
    p.arr = a
    return p


def PO(a, off):
    """pointer to element offset `off` (may be inside a margin) of a contiguous array"""
    p = _ArrayPtr(a.ctypes.data + off * a.itemsize)
    p.arr = a
    return p


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        so = os.path.join(ROOT, 'oracle', '_build', 'liboracle.so')
        if not os.path.exists(so):
            subprocess.check_call(['make', '-s', '-C', os.path.join(ROOT, 'oracle')])
        L = ctypes.CDLL(so)
        for name in ('orc_sad', 'orc_sse', 'orc_had', 'orc_had2sad', 'orc_dist', 'orc_sad_mask', 'orc_fix_wsse', 'orc_mv_cost'):
            getattr(L, name).restype = ctypes.c_uint64
        L.orc_mv_bits.restype = ctypes.c_uint32
        L.orc_mv_cost.argtypes = [ctypes.c_double] + [ctypes.c_int] * 6
        L.orc_full_search.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        _oracle = L
    return _oracle


_dqoracle = None


def dq_oracle():
    """oracle/_build/libdqoracle.so: the dependent-quantisation restatement (vvenc_b200/csrc/depquant_core.h) compiled for the CPU"""
    global _dqoracle
    if _dqoracle is None:
        so = os.path.join(ROOT, 'oracle', '_build', 'libdqoracle.so')
        if not os.path.exists(so):
            subprocess.check_call(['make', '-s', '-C', os.path.join(ROOT, 'oracle')])
        L = ctypes.CDLL(so)
        L.orc_dep_quant.argtypes = [ctypes.c_int] * 4 + [ctypes.c_double] + [ctypes.c_int] * 4 + [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.orc_dep_quant_chroma.argtypes = [ctypes.c_int] * 4 + [ctypes.c_double] + [ctypes.c_int] * 3 + [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.orc_dep_quant_constants.argtypes = [ctypes.c_int] * 4 + [ctypes.c_double, ctypes.c_int, ctypes.c_void_p]
        # oracle/rdoq_oracle.cpp (vvenc_b200/csrc/rdoq_core.h compiled for the CPU) lives in the same library
        L.orc_rdoq.argtypes = [ctypes.c_int] * 8 + [ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.orc_rdoq_constants.argtypes = [ctypes.c_int] * 8 + [ctypes.c_void_p]
        L.orc_rdoq_v2.argtypes = L.orc_rdoq.argtypes
        L.orc_rdoq_ts.argtypes = [ctypes.c_int] * 5 + [ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.orc_rdoq_ts_constants.argtypes = [ctypes.c_int] * 5 + [ctypes.c_void_p, ctypes.c_void_p]
        L.orc_rdoq_bdpcm.argtypes = [ctypes.c_int] * 6 + [ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        _dqoracle = L
    return _dqoracle


_ref = None


def refshim_path():
    return os.path.join(ROOT, 'oracle', '_ref', 'libvvenc_refshim.so')


def have_ref():
    return os.path.exists(refshim_path())


def _module():
    """test module of the running test (pytest sets PYTEST_CURRENT_TEST = 'tests/<module>.py::<name> (<phase>)')"""
    cur = os.environ.get('PYTEST_CURRENT_TEST', '')
    return os.path.splitext(os.path.basename(cur.split('::')[0]))[0] if '::' in cur else None


def _test_id():
    return os.environ.get('PYTEST_CURRENT_TEST', '').rsplit(' (', 1)[0]


def have_ref_results(module):
    """the reference's answers are available to `module`: the probe itself, or a recording of its calls"""
    return have_ref() or os.path.exists(os.path.join(RECORDINGS, module + '.npz'))


_UNANSWERED = {}          # id(array) -> weakref: arrays the last replayed call writing them could not fill (not sampled)
_STALE = {}               # id(array) -> weakref: arrays that missed a write at some point, so differ from what the reference saw


def answered(*arrays):
    """False when one of these arrays is a probe output that replay could not fill (not in the recorded sample)"""
    return not any(id(a) in _UNANSWERED and _UNANSWERED[id(a)]() is a for a in arrays)


def refshim_reset():
    """start of a test: replay restarts the test's call sequence (a test run twice in one process replays twice)"""
    _UNANSWERED.clear()
    _STALE.clear()
    if isinstance(_ref, _Replay):
        _ref.cursor.clear()


def _arg_state(args):
    """(input digest, buffers the call may write): arrays behind P / PO pointers, objects passed by reference, ctypes arrays"""
    h = hashlib.sha256()
    bufs = []
    for i, a in enumerate(args):
        if isinstance(a, _ArrayPtr):
            arr = a.arr
            h.update(b'P%d:%s:%s:%d:' % (i, arr.dtype.str.encode(), str(arr.shape).encode(), a.value - arr.ctypes.data))
            h.update(np.ascontiguousarray(arr).view(np.uint8).tobytes())
            bufs.append((i, 'arr', arr))
        elif type(a).__name__ == 'CArgObject':                       # ctypes.byref(x)
            h.update(b'R%d:%s:' % (i, type(a._obj).__name__.encode()) + bytes(a._obj))
            bufs.append((i, 'ref', a._obj))
        elif isinstance(a, ctypes.Array):
            if a._type_ in (ctypes.c_void_p, ctypes.c_char_p):     # pointer tables: addresses differ from run to run
                h.update(b'T%d:%d:' % (i, len(a)))
            else:
                h.update(b'A%d:' % i + bytes(a))
                bufs.append((i, 'carr', a))
        elif isinstance(a, ctypes._SimpleCData):
            h.update(b'S%d:%r:' % (i, a.value))
        else:
            h.update(b'V%d:%r:' % (i, a))
    return h.hexdigest()[:4], bufs


def _snapshot(kind, obj):
    return np.ascontiguousarray(obj).view(np.uint8).tobytes() if kind == 'arr' else bytes(obj)


def _seeded_order(tid, n):
    return sorted(range(n), key=lambda k: zlib.crc32(b'%s:%d' % (tid.encode(), k)))


def _load_recording(mod):
    """{test id: {'sampled': n, 'calls': [[name, digest, ret, [[arg, bytes or None], ...]], ...]}} of a module's recording, {} if none"""
    path = os.path.join(RECORDINGS, mod + '.npz')
    if not os.path.exists(path):
        return {}
    z = np.load(path)
    index = json.loads(zlib.decompress(z['index'].tobytes()))
    data = z['blobs'].tobytes()
    blobs = [data[o:o + n] for o, n in index['blobs']]
    return {t: {'sampled': r['sampled'], 'calls': [[index['names'][c[0]], c[1], c[2], [[i, None if b < 0 else blobs[b]] for i, b in c[3]]] for c in r['calls']]}
            for t, r in index['tests'].items()}


class _Recorder:
    """wraps the probe: every call runs for real and is logged per test (input digest, return value, buffers it changed)"""

    def __init__(self, lib):
        self._lib = lib
        self._calls = {}                 # module -> test id -> [[name, digest, ret, [[arg, bytes], ...]]]
        atexit.register(self._save)

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        rec = self

        class Call:
            def __setattr__(self, k, v):
                setattr(fn, k, v)

            def __getattr__(self, k):
                return getattr(fn, k)

            def __call__(self, *args):
                digest, bufs = _arg_state(args)
                before = [_snapshot(kind, obj) for _, kind, obj in bufs]
                raw = fn(*args)
                out = [[i, _snapshot(kind, obj)] for (i, kind, obj), b0 in zip(bufs, before) if _snapshot(kind, obj) != b0]
                ret = {'bytes': raw.decode('latin-1')} if isinstance(raw, bytes) else raw
                rec._calls.setdefault(_module() or '_unknown', {}).setdefault(_test_id(), []).append([name, digest, ret, out])
                return raw

        return Call()

    @staticmethod
    def _sample(tid, calls):
        """large outputs of the first m calls in the seeded order, m as large as TEST_BUDGET compressed bytes allow (at least 2)"""
        large = [k for k in _seeded_order(tid, len(calls)) if any(len(b) > SMALL_OUTPUT for _, b in calls[k][3])]
        lo, hi = min(2, len(large)), len(large)
        while lo < hi:                                                   # largest m that fits
            m = (lo + hi + 1) // 2
            kept = {b for k in large[:m] for _, b in calls[k][3] if len(b) > SMALL_OUTPUT}
            if len(zlib.compress(b''.join(sorted(kept)), 9)) <= TEST_BUDGET:
                lo = m
            else:
                hi = m - 1
        keep = set(large[:lo])
        return {'sampled': lo, 'calls': [[n, d, r, [[i, b if (len(b) <= SMALL_OUTPUT or k in keep) else None] for i, b in out]]
                                         for k, (n, d, r, out) in enumerate(calls)]}

    def _save(self):
        os.makedirs(RECORDINGS, exist_ok=True)
        for mod, new in self._calls.items():
            tests = _load_recording(mod)                                 # tests this run did not select keep their recording
            tests.update({t: self._sample(t, calls) for t, calls in new.items()})
            names, blobs, pos = {}, {}, 0
            for r in tests.values():
                for c in r['calls']:
                    names.setdefault(c[0], len(names))
                    for _, b in c[3]:
                        if b is not None:
                            blobs.setdefault(b, len(blobs))
            order = sorted(blobs, key=blobs.get)
            offsets = []
            for b in order:
                offsets.append([pos, len(b)]); pos += len(b)
            index = {'names': sorted(names, key=names.get), 'blobs': offsets,
                     'tests': {t: {'sampled': r['sampled'], 'calls': [[names[n], d, ret, [[i, -1 if b is None else blobs[b]] for i, b in out]] for n, d, ret, out in r['calls']]}
                               for t, r in sorted(tests.items())}}
            np.savez_compressed(os.path.join(RECORDINGS, mod + '.npz'), index=np.frombuffer(zlib.compress(json.dumps(index, separators=(',', ':')).encode(), 9), dtype=np.uint8),
                                blobs=np.frombuffer(b''.join(order) or b'\0', dtype=np.uint8))


class _Replay:
    """answers probe calls from a recording: same call sequence per test, same input digests, the recorded outputs written back"""

    def __init__(self):
        self._files = {}
        self.cursor = {}

    def _recording(self, mod):
        if mod not in self._files:
            if not os.path.exists(os.path.join(RECORDINGS, mod + '.npz')):
                raise RuntimeError('no reference probe (%s) and no recording of its calls for %s' % (refshim_path(), mod))
            self._files[mod] = _load_recording(mod)
        return self._files[mod]

    def __getattr__(self, name):
        rep = self

        class Call:
            def __setattr__(self, k, v):                             # argtypes / restype: the recorded values already have the right form
                pass

            def __call__(self, *args):
                mod, tid = _module(), _test_id()
                rec = rep._recording(mod).get(tid)
                assert rec is not None, 'the recording of %s has no calls of %s: record it again' % (mod, tid)
                seq = rec['calls']
                k = rep.cursor.get(tid, 0)
                assert k < len(seq), '%s: more probe calls than recorded (%d)' % (tid, len(seq))
                rep.cursor[tid] = k + 1
                rname, digest, ret, out = seq[k]
                got, bufs = _arg_state(args)
                # an input that is itself an unsampled output of an earlier call differs from what the reference saw: only the call order is checked then
                fed = any(kind == 'arr' and id(obj) in _STALE and _STALE[id(obj)]() is obj for _, kind, obj in bufs)
                assert rname == name and (got == digest or fed), '%s: probe call %d is %s with other inputs than the recorded %s' % (tid, k, name, rname)
                by_pos = {i: (kind, obj) for i, kind, obj in bufs}
                for i, b in out:
                    kind, obj = by_pos[i]
                    if kind == 'arr' and (b is None or fed):
                        _UNANSWERED[id(obj)] = _STALE[id(obj)] = weakref.ref(obj)
                    elif b is None:
                        continue
                    elif kind == 'arr':
                        _UNANSWERED.pop(id(obj), None)
                        obj.reshape(-1).view(np.uint8)[:] = np.frombuffer(b, dtype=np.uint8)
                    else:
                        ctypes.memmove(ctypes.addressof(obj), b, len(b))
                return ret['bytes'].encode('latin-1') if isinstance(ret, dict) else ret

        return Call()


def refshim():
    global _ref
    if _ref is None and not have_ref():
        _ref = _Replay()
    if _ref is None:
        L = ctypes.CDLL(refshim_path())
        for name in ('refshim_dist', 'refshim_sad_mask', 'refshim_fix_wsse', 'refshim_mv_cost'):
            getattr(L, name).restype = ctypes.c_uint64
        L.refshim_mv_bits.restype = ctypes.c_uint32
        L.refshim_mv_cost.argtypes = [ctypes.c_double] + [ctypes.c_int] * 6
        L.refshim_set_simd.restype = ctypes.c_char_p
        L.refshim_full_search.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.refshim_pattern_search_member.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                                    ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.refshim_dep_quant.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 8 + [ctypes.c_double] + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 5
        L.refshim_dep_quant_comp.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 8 + [ctypes.c_double] + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 5
        L.refshim_dep_quant_b200_comp.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 8 + [ctypes.c_double] + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3
        L.refshim_dep_quant_b200.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 8 + [ctypes.c_double] + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3
        L.refshim_rdoq.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 9 + [ctypes.c_double] + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 5
        L.refshim_rdoq_b200.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 9 + [ctypes.c_double] + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3
        L.refshim_rdoq_ts.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5
        L.refshim_rdoq_ts_b200.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 2
        L.refshim_rdoq_bdpcm.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 7 + [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
        L.refshim_rdoq_bdpcm_b200.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 4
        L.refshim_set_simd(b'AVX2')
        _ref = _Recorder(L) if os.environ.get('VVB_RECORD_REFSHIM') == '1' else L
    return _ref
