"""ctypes bindings of the CPU oracle (oracle/libgyoracle.so) and of the compiled reference (oracle/_ref/libgyref.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs. Nothing under gyeeta_b200/ may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

EVENT_DTYPE = np.dtype([("svc_id", "<u8"), ("flow_key", "<u8"), ("value", "<u4"), ("host_idx", "<u4"),
                        ("tsec", "<u4"), ("type", "<u2"), ("flags", "<u2")], align=True)
assert EVENT_DTYPE.itemsize == 32

SERIAL_DTYPE = np.dtype([("count", "<u8"), ("sum", "<i8")])
CENTROID_DTYPE = np.dtype([("mean", "<f8"), ("weight", "<u8")])
TD_CAP = 256

CLS = dict(RESP_TIME=0, SEMI_LOG=1, SEMI_LOG_LO=2, DURATION=3, HASH_10_5000=4, HASH_5_250=5, HASH_1_3000=6,
           PERCENT=7, FD_I8_9_26_5=8, FD_INT_M15_M3_4=9)
T_INT64, T_INT, T_INT8 = 0, 1, 2


class TDigest(C.Structure):
    _fields_ = [("c", C.c_byte * (16 * TD_CAP)), ("n", C.c_uint32), ("total", C.c_uint64),
                ("minv", C.c_double), ("maxv", C.c_double)]

    def centroids(self):
        a = np.frombuffer(bytes(self.c), dtype=CENTROID_DTYPE)[: self.n]
        return a["mean"].copy(), a["weight"].copy()


def build(ref=True):
    """make the oracle (and, when /root/reference is present, oracle/_ref)."""
    subprocess.run(["make", "-s", "-C", HERE] + ([] if ref else [os.path.join(HERE, "libgyoracle.so")]), check=True)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "libgyoracle.so")
        if not os.path.exists(path):
            build(ref=False)
        L = C.CDLL(path)
        L.gyo_jhash_2words.restype = C.c_uint32
        L.gyo_jhash_2words.argtypes = [C.c_uint32] * 3
        L.gyo_jhash2.restype = C.c_uint32
        L.gyo_jhash2.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.gyo_jhash.restype = C.c_uint32
        L.gyo_jhash.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.gyo_uint64_hash.restype = C.c_uint32
        L.gyo_uint64_hash.argtypes = [C.c_uint64]
        L.gyo_nbuckets.argtypes = [C.c_int]
        L.gyo_bucket.argtypes = [C.c_int, C.c_int64]
        L.gyo_bucket_max_threshold.restype = C.c_int64
        L.gyo_bucket_max_threshold.argtypes = [C.c_int, C.c_int, C.c_size_t]
        L.gyo_hist_run.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gyo_cms_index.restype = C.c_uint32
        L.gyo_cms_index.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32]
        L.gyo_cms_increment.restype = C.c_uint64
        L.gyo_cms_increment.argtypes = [C.c_uint32]
        L.gyo_td_code.restype = C.c_uint32
        L.gyo_td_code.argtypes = [C.c_uint32]
        L.gyo_flow_hashes.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p]
        L.gyo_hll_hash.restype = C.c_uint64
        L.gyo_hll_hash.argtypes = [C.c_uint64]
        L.gyo_hll_idx_rank.argtypes = [C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
        L.gyo_hll_estimate.restype = C.c_double
        L.gyo_hll_estimate.argtypes = [C.c_void_p, C.c_uint32]
        L.gyo_td_init.argtypes = [C.c_void_p]
        L.gyo_td_add_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_double]
        L.gyo_td_add_classic.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_double]
        L.gyo_td_compress.restype = C.c_uint32
        L.gyo_td_compress.argtypes = [C.c_void_p, C.c_uint32, C.c_double, C.c_void_p, C.c_uint32]
        L.gyo_td_quantile.restype = C.c_double
        L.gyo_td_quantile.argtypes = [C.c_void_p, C.c_uint32, C.c_double, C.c_double, C.c_double]
        L.gyo_td_quantile_f.restype = C.c_double
        L.gyo_td_quantile_f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_double]
        L.gyo_create.restype = C.c_void_p
        L.gyo_create.argtypes = [C.c_uint32] * 9
        L.gyo_destroy.argtypes = [C.c_void_p]
        L.gyo_register_ids.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int]
        L.gyo_ingest.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.gyo_flush.argtypes = [C.c_void_p, C.c_uint32]
        L.gyo_task_last.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.gyo_set_idle_evict.argtypes = [C.c_void_p, C.c_uint32]
        L.gyo_evicted.restype = C.c_uint32
        L.gyo_evicted.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.gyo_nsvcs.restype = C.c_uint32
        L.gyo_nsvcs.argtypes = [C.c_void_p]
        L.gyo_export_hist.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gyo_export_hll.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.gyo_export_tdigest.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.gyo_export_conn.argtypes = [C.c_void_p, C.c_uint64] + [C.c_void_p] * 4
        L.gyo_export_conn_bitmap.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
        L.gyo_export_aux.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.gyo_export_state.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        L.gyo_listener_state.restype = None
        L.gyo_listener_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gyo_cms_table.restype = C.c_void_p
        L.gyo_cms_table.argtypes = [C.c_void_p, C.c_int]
        L.gyo_counters.argtypes = [C.c_void_p, C.c_void_p]
        L.gyo_merge_from.argtypes = [C.c_void_p, C.c_void_p]
        L.gyo_bench_ingest.restype = C.c_double
        L.gyo_bench_ingest.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64]
        _lib = L
    return _lib


def ref():
    """the reference's own code compiled into oracle/_ref/libgyref.so; None when it is not available."""
    global _ref
    if _ref is None:
        path = os.path.join(HERE, "_ref", "libgyref.so")
        if not os.path.exists(path):
            if os.path.exists("/root/reference/common/gy_statistics.h"):
                build(ref=True)
            if not os.path.exists(path):
                return None
        R = C.CDLL(path)
        R.gyref_hist_run.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        R.gyref_hist_pct_from_serial.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p,
                                                 C.c_size_t, C.c_void_p, C.c_void_p]
        R.gyref_uint64_hash.restype = C.c_uint32
        R.gyref_uint64_hash.argtypes = [C.c_uint64]
        R.gyref_jhash_2words.restype = C.c_uint32
        R.gyref_jhash_2words.argtypes = [C.c_uint32] * 3
        R.gyref_jhash2.restype = C.c_uint32
        R.gyref_jhash2.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        R.gyref_jhash.restype = C.c_uint32
        R.gyref_jhash.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        R.gyref_sizeof_hist_resp.restype = C.c_size_t
        R.gyref_bench_resp_hist.restype = C.c_double
        R.gyref_bench_resp_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
        _ref = R
    return _ref


def hist_run(L, fn, cls, tkind, vals, pcts=()):
    """run a fresh histogram over vals with either library; returns dict(stats, total, max, pct, buckets, avg, nb)."""
    vals = np.ascontiguousarray(vals, dtype=np.int64)
    pcts = np.ascontiguousarray(pcts, dtype=np.float32)
    stats = np.zeros(16, dtype=SERIAL_DTYPE)
    total, mx, avg = C.c_uint64(), C.c_int64(), C.c_float()
    out_pct = np.zeros(max(len(pcts), 1), dtype=np.int64)
    ids = np.zeros(max(len(vals), 1), dtype=np.int64)
    nb = getattr(L, fn)(cls, tkind, _p(vals), len(vals), _p(pcts), len(pcts), _p(stats), C.byref(total), C.byref(mx),
                        _p(out_pct), _p(ids), C.byref(avg))
    return dict(nb=nb, stats=stats[:nb].copy(), total=total.value, max=mx.value, pct=out_pct[: len(pcts)].copy(),
                buckets=ids[: len(vals)].copy(), avg=avg.value)


class OracleEngine:
    def __init__(self, max_svcs=1024, max_tasks=1024, cms_depth=4, cms_log2_width=20, hll_p=12, td_compression=200,
                 flags=1, rank=0, world=1):
        self.L = lib()
        self.cfg = dict(max_svcs=max_svcs, max_tasks=max_tasks, cms_depth=cms_depth, cms_log2_width=cms_log2_width,
                        hll_p=hll_p, td_compression=td_compression, flags=flags, rank=rank, world=world)
        self.h = self.L.gyo_create(max_svcs, max_tasks, cms_depth, cms_log2_width, hll_p, td_compression, flags, rank, world)

    def close(self):
        if self.h:
            self.L.gyo_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def register_ids(self, ids, is_task=False):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        return self.L.gyo_register_ids(self.h, _p(ids), len(ids), int(is_task))

    def ingest(self, ev):
        assert ev.dtype == EVENT_DTYPE
        ev = np.ascontiguousarray(ev)
        return self.L.gyo_ingest(self.h, _p(ev), len(ev))

    def flush(self, tsec=0):
        self.L.gyo_flush(self.h, tsec)

    def task_last(self, id_):
        out = np.zeros(6, dtype=np.uint64)
        rc = self.L.gyo_task_last(self.h, int(id_), _p(out))
        return None if rc else out

    def set_idle_evict(self, secs):
        self.L.gyo_set_idle_evict(self.h, secs)

    def evicted_ids(self, cap=1 << 20):
        out = np.zeros(cap, dtype=np.uint64)
        tot = C.c_uint64()
        n = self.L.gyo_evicted(self.h, _p(out), cap, C.byref(tot))
        return out[:n].copy(), tot.value

    def nsvcs(self):
        return self.L.gyo_nsvcs(self.h)

    def export_hist(self, id_, which):
        out = np.zeros(15, dtype=SERIAL_DTYPE)
        total, mx = C.c_uint64(), C.c_int64()
        rc = self.L.gyo_export_hist(self.h, int(id_), which, _p(out), C.byref(total), C.byref(mx))
        if rc:
            return None
        return out, total.value, mx.value

    def export_hll(self, id_):
        regs = np.zeros(1 << self.cfg["hll_p"], dtype=np.uint8)
        rc = self.L.gyo_export_hll(self.h, int(id_), _p(regs))
        return None if rc else regs

    def export_tdigest(self, id_):
        td = TDigest()
        rc = self.L.gyo_export_tdigest(self.h, int(id_), C.byref(td))
        return None if rc else td

    def export_conn(self, id_):
        v = [C.c_uint64() for _ in range(4)]
        rc = self.L.gyo_export_conn(self.h, int(id_), *[C.byref(x) for x in v])
        return None if rc else tuple(x.value for x in v)

    def export_state(self, id_):
        """{state, issue, issue_bit_hist, high_resp_bit_hist, nconn_active} the last flush derived, None if the id is unknown"""
        out = np.zeros(5, dtype=np.uint32)
        if self.L.gyo_export_state(self.h, int(id_), _p(out)):
            return None
        return tuple(int(x) for x in out)

    def export_aux(self, id_):
        """dict(act_cur, act_last, err_cur, err_last: packed {lo32, hi32}; rtt_cur, rtt_last: float)"""
        out = np.zeros(6, dtype=np.uint64)
        if self.L.gyo_export_aux(self.h, int(id_), _p(out)):
            return None
        f = lambda b: float(np.array([b], dtype=np.uint32).view(np.float32)[0])
        return dict(act_cur=int(out[0]), act_last=int(out[1]), err_cur=int(out[2]), err_last=int(out[3]), rtt_cur=f(int(out[4])), rtt_last=f(int(out[5])))

    def export_conn_bitmap(self, id_, last_window=False):
        masks = np.zeros(15, dtype=np.uint32)
        cnt = np.zeros(15, dtype=np.uint8)
        rc = self.L.gyo_export_conn_bitmap(self.h, int(id_), int(last_window), _p(masks), _p(cnt))
        return None if rc else (masks, cnt)

    def cms(self, last_window=False):
        n = self.cfg["cms_depth"] << self.cfg["cms_log2_width"]
        ptr = self.L.gyo_cms_table(self.h, int(last_window))
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint64)), shape=(n,)).copy()

    def counters(self):
        out = np.zeros(8, dtype=np.uint64)
        self.L.gyo_counters(self.h, _p(out))
        return dict(zip(["in", "dropped", "resp", "tcp", "task", "nsvcs", "ntasks", "foreign"], out.tolist()))

    def merge_from(self, other):
        self.L.gyo_merge_from(self.h, other.h)


def td_quantile(td, q):
    return lib().gyo_td_quantile(C.byref(td), td.n, td.minv, td.maxv, q)


def td_compress(means, weights, delta):
    """gyo_td_compress of one mean-sorted centroid list -> (means, weights) of at most TD_CAP clusters"""
    src = np.zeros(len(means), dtype=CENTROID_DTYPE)
    src["mean"], src["weight"] = means, weights
    out = np.zeros(TD_CAP, dtype=CENTROID_DTYPE)
    n = lib().gyo_td_compress(_p(src), len(src), float(delta), _p(out), TD_CAP)
    assert n <= TD_CAP, n
    return out["mean"][:n].copy(), out["weight"][:n].copy()


def merge_compress(a, b, delta):
    """what the merge kernels do with two digests a, b = (means, weights): a stable merge by mean, `a` first on equal means, then
    the fixed-grid compress. Both lists are sorted by mean, so a stable sort of a + b is that merge."""
    means = np.concatenate([np.asarray(a[0], dtype=np.float64), np.asarray(b[0], dtype=np.float64)])
    weights = np.concatenate([np.asarray(a[1], dtype=np.uint64), np.asarray(b[1], dtype=np.uint64)])
    if not len(means):
        return means, weights
    order = np.argsort(means, kind="stable")
    return td_compress(means[order], weights[order], delta)


def td_new():
    td = TDigest()
    lib().gyo_td_init(C.byref(td))
    return td


def td_add(td, vals, delta=200.0, classic=False):
    vals = np.ascontiguousarray(vals, dtype=np.uint32)
    fn = lib().gyo_td_add_classic if classic else lib().gyo_td_add_batch
    fn(C.byref(td), _p(vals), len(vals), delta)
    return td


def ref_hist_rate(slots, vals_ms, nthreads):
    """samples/s of the REFERENCE's own GY_HISTOGRAM::add_data (oracle/_ref), samples pre-sharded by slot % nthreads"""
    R = ref()
    if R is None:
        return None
    slots = np.ascontiguousarray(slots, dtype=np.uint32)
    owner = (slots % nthreads).astype(np.int32)
    order = np.argsort(owner, kind="stable")
    s2 = np.ascontiguousarray(slots[order]); v2 = np.ascontiguousarray(np.asarray(vals_ms, dtype=np.int64)[order])
    offs = np.concatenate([[0], np.cumsum(np.bincount(owner, minlength=nthreads))]).astype(np.uint64)
    tot = C.c_uint64()
    sec = R.gyref_bench_resp_hist(_p(s2), _p(v2), _p(offs), int(slots.max()) + 1, nthreads, C.byref(tot))
    assert tot.value == len(slots)
    return len(slots) / sec


def listener_state(inp, high_resp_bit_hist=0):
    """gyo_listener_state on a struct with gysk_listener_state_in's layout -> (state, issue, new high_resp_bit_hist)"""
    hb, st, iss = C.c_uint8(high_resp_bit_hist), C.c_uint8(), C.c_uint8()
    lib().gyo_listener_state(C.byref(inp), C.byref(hb), C.byref(st), C.byref(iss))
    return st.value, iss.value, hb.value


def task_groupby(samples, rec_dtype):
    """gyo_task_groupby: the CPU statement of row a15b -> records of rec_dtype (72 bytes), groups in order of first appearance"""
    samples = np.ascontiguousarray(samples)
    out = np.zeros(max(len(samples), 1), dtype=rec_dtype)
    L = lib()
    L.gyo_task_groupby.restype = C.c_uint32
    L.gyo_task_groupby.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32]
    ng = L.gyo_task_groupby(_p(samples), len(samples), _p(out), len(out))
    return out[:ng].copy()
