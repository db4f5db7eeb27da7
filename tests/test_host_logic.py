"""CPU-side tests (no GPU): the C-ABI library loads and exports every symbol include/gysketch.h declares; the pure host
helpers of the library (percentile rule, bucket ids, estimators) agree with the oracle; the t-digest oracle variants agree
within epsilon and obey the sketch's rank-error bound; creating an engine without a GPU fails loudly."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from gyeeta_b200 import engine as ge
from gyeeta_b200 import synth
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "gysketch.h")).read()
    names = set(re.findall(r"\b(gysk_[a-z0-9_]+)\s*\(", hdr))
    names -= {"gysk_svc_summary", "gysk_flow_est"}
    assert len(names) >= 35
    L = C.CDLL(ge.LIB_PATH)
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing
    assert ge.load_library().gysk_abi_version() == 2


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(ge.GyskError) as ei:
        ge.Engine()
    assert ei.value.code == -19 and "no CPU fallback" in str(ei.value)


def test_product_never_touches_the_oracle():
    """the product tree may not import / link / dlopen anything under oracle/"""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "gyeeta_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc")):
                src = open(os.path.join(dirpath, f)).read()
                assert "pyoracle" not in src and "libgyoracle" not in src and "gyo_" not in src and "gyref" not in src, f
    out = os.popen(f"ldd {ge.LIB_PATH}").read()
    assert "gyoracle" not in out and "gyref" not in out


def test_host_helpers_match_oracle():
    L, O = ge.load_library(), po.lib()
    rng = np.random.default_rng(2)
    assert L.gysk_uint64_hash(42) == 4033382092
    vals = np.concatenate([rng.integers(-100, 200000, 3000), rng.integers(-2 ** 40, 2 ** 40, 500), [2 ** 31, 2 ** 32 + 5, -1, 0]])
    for cls in range(8):
        assert L.gysk_hist_nbuckets(cls) == O.gyo_nbuckets(cls)
        for v in vals:
            assert L.gysk_hist_bucket(cls, int(v)) == O.gyo_bucket(cls, int(v)), (cls, v)
    pcts = np.array([25, 50, 95, 99, 99.999, 0.001, 100], dtype=np.float32)
    for cls in range(8):
        for tk in (0, 1):
            for scale in (10, 2 ** 25, 2 ** 40):
                r = po.hist_run(O, "gyo_hist_run", cls, tk, rng.integers(-5, 70000, 2000), pcts)
                stats = np.zeros(15, dtype=ge.SERIAL_DTYPE)
                stats[: r["nb"]] = r["stats"]
                stats["count"] *= scale          # exercise the float cut-off far beyond 2^24
                total = int(stats["count"].sum())
                h = np.zeros(1, dtype=np.dtype([("stats", po.SERIAL_DTYPE, 16), ("total", "<u8"), ("max", "<i8"), ("cls", "<i4"), ("tk", "<i4")]))
                h["stats"][0][:15] = stats
                h["total"], h["cls"], h["tk"] = total, cls, tk
                want = np.zeros(len(pcts), dtype=np.int64)
                O.gyo_hist_percentiles(po._p(h), po._p(pcts), C.c_size_t(len(pcts)), po._p(want), None)
                got = np.zeros(len(pcts), dtype=np.int64)
                assert L.gysk_hist_percentiles(cls, tk, ge._p(stats), total, ge._p(pcts), len(pcts), ge._p(got)) == 0
                assert np.array_equal(got, want), (cls, tk, scale)
    for p in (4, 8, 12, 16):
        regs = rng.integers(0, 40, 1 << p).astype(np.uint8) * (rng.random(1 << p) < 0.6)
        regs = regs.astype(np.uint8)
        assert L.gysk_hll_estimate(ge._p(regs), p) == O.gyo_hll_estimate(po._p(regs), p)
    td = po.td_add(po.td_new(), rng.integers(0, 10 ** 8, 50000).astype(np.uint32))
    means, weights = td.centroids()
    for q in (0.0, 0.001, 0.5, 0.95, 0.99, 0.9999, 1.0):
        assert L.gysk_tdigest_quantile(ge._p(means), ge._p(weights), len(means), td.minv, td.maxv, q) == po.td_quantile(td, q)


def test_tdigest_oracle_properties():
    from tests.util import td_p99_tolerance
    rng = np.random.default_rng(4)
    for sigma, n in ((1.2, 200_000), (1.5, 50_000), (0.5, 10_000)):
        x = np.minimum(np.exp(rng.normal(np.log(2000.0), sigma, n)), 9e8).astype(np.uint32)
        tb = po.td_new()
        for ch in np.array_split(x, 5):
            po.td_add(tb, ch, delta=200.0)
        tc = po.td_add(po.td_new(), x, delta=200.0, classic=True)
        mb, wb = tb.centroids()
        assert int(wb.sum()) == n == tb.total and tb.n <= po.TD_CAP and tc.n <= po.TD_CAP
        assert np.all(np.diff(mb) >= 0) and tb.minv == x.min() and tb.maxv == x.max()
        xs = np.sort(x)
        for q in (0.5, 0.95, 0.99):
            ex = float(xs[int(np.ceil(q * n)) - 1])
            for td in (tb, tc):
                g = po.td_quantile(td, q)
                assert abs(np.searchsorted(xs, g) / n - q) < 0.002, (sigma, n, q)          # rank error: what a t-digest bounds
                assert abs(g - ex) / ex < (0.01 if q < 0.99 else td_p99_tolerance(n)), (sigma, n, q, g, ex)
    # tiny inputs
    t = po.td_add(po.td_new(), np.array([7], dtype=np.uint32))
    assert t.n == 1 and po.td_quantile(t, 0.5) == 7.0
    t = po.td_add(po.td_new(), np.array([5, 5, 5, 5], dtype=np.uint32))
    assert po.td_quantile(t, 0.99) == 5.0


def test_oracle_engine_sharded_merge_equals_single():
    """world_size-2 statement of the merge step on the CPU oracle: shards merged with gyo_merge_from == one engine"""
    rng = np.random.default_rng(8)
    ev = synth.gen_mixed(rng, 60_000, 200, ntask=16, nhosts=32, nclients=3000)
    one = po.OracleEngine(max_svcs=512, max_tasks=64, cms_log2_width=12)
    one.ingest(ev)
    sh = [po.OracleEngine(max_svcs=512, max_tasks=64, cms_log2_width=12, rank=r, world=2) for r in range(2)]
    for s in sh:
        s.ingest(ev)
    assert sh[0].counters()["in"] + sh[1].counters()["in"] == len(ev)
    merged = po.OracleEngine(max_svcs=512, max_tasks=64, cms_log2_width=12)
    merged.merge_from(sh[0]); merged.merge_from(sh[1])
    assert np.array_equal(merged.cms(), one.cms())
    for id_ in np.unique(ev["svc_id"][ev["type"] == 5])[:40]:
        a, b = merged.export_hist(int(id_), 0), one.export_hist(int(id_), 0)
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]
        assert np.array_equal(merged.export_hll(int(id_)), one.export_hll(int(id_)))


@pytest.mark.parametrize("delta", [10, 37, 200, 256])
def test_merge_compress_equals_the_oracle_merge(delta):
    """pyoracle.merge_compress (the CPU replay of the merge kernels' digest fold) gives the same centroids, bit for bit, as the
    digest merge of gyo_merge_from, which walks the merged list in C"""
    rng = np.random.default_rng(12)
    ev = synth.gen_mixed(rng, 40_000, 60, ntask=8, nhosts=16, nclients=2000)
    ev["host_idx"] = rng.integers(0, 16, len(ev))           # every service on both shards
    sh = [po.OracleEngine(max_svcs=128, max_tasks=16, cms_log2_width=8, td_compression=delta, rank=r, world=2) for r in range(2)]
    for s in sh:
        for off in range(0, len(ev), 4096):
            s.ingest(ev[off: off + 4096])
    merged = po.OracleEngine(max_svcs=128, max_tasks=16, cms_log2_width=8, td_compression=delta)
    merged.merge_from(sh[0]); merged.merge_from(sh[1])
    nboth = 0
    for id_ in np.unique(ev["svc_id"][ev["type"] == 5]):
        parts = [s.export_tdigest(int(id_)) for s in sh]
        acc = (np.zeros(0), np.zeros(0, dtype=np.uint64))
        for td in parts:
            if td is not None:
                acc = po.merge_compress(acc, td.centroids(), delta)
        nboth += all(td is not None and td.n for td in parts)
        m, w = merged.export_tdigest(int(id_)).centroids()
        assert np.array_equal(acc[0], m) and np.array_equal(acc[1], w), hex(int(id_))
        assert len(m) <= delta
    assert nboth >= 10
    assert po.merge_compress(([], []), ([], []), delta)[0].size == 0


def test_oracle_idle_eviction_rule():
    """the checker's own statement of the listener deletion rule (common/gy_socket_stat.cc:3968-3982): never-active services
    stay (tclock == 0), an idle one goes only when last activity + 300 s < now AND first seen + 600 s < now, its slot is
    recycled and a returning id starts empty"""
    from gyeeta_b200 import engine as ge
    from oracle import pyoracle as po
    orc = po.OracleEngine(max_svcs=4, max_tasks=4, cms_log2_width=8)
    orc.set_idle_evict(300)

    def resp(ids, t):
        ev = np.zeros(len(ids), dtype=po.EVENT_DTYPE)
        ev["svc_id"] = ids; ev["type"] = 5; ev["value"] = 5000; ev["tsec"] = t; ev["flow_key"] = 7
        orc.ingest(ev)

    orc.register_ids(np.array([11, 22, 33], dtype=np.uint64))
    resp([11, 22], 100); orc.flush(100)                     # 33 never active
    resp([11], 350); orc.flush(350)
    assert len(orc.evicted_ids()[0]) == 0                   # 22: 100 + 300 < 350 fails the age test (100 + 600 < 350 is false)
    resp([11], 650); orc.flush(650)
    assert len(orc.evicted_ids()[0]) == 0                   # 100 + 600 < 650 false
    resp([11], 701); orc.flush(701)
    ids, tot = orc.evicted_ids()
    assert list(ids) == [22] and tot == 1 and orc.nsvcs() == 2
    assert orc.export_hist(22, 2) is None and orc.export_hist(33, 2) is not None
    resp([22, 44, 55], 705)                                  # 22 returns, 44 takes a fresh slot, 55 finds the table full
    assert orc.nsvcs() == 4 and orc.export_hist(55, 0) is None
    assert orc.export_hist(22, 0)[1] == 1 and orc.export_hist(44, 0)[1] == 1


def test_tdigest_pgtext_form():
    """the Postgres `tdigest` text form (tdigest_out / tdigest_in of the extension the reference queries through,
    common/gy_query_common.cc:1805-1858,3385): header fields, one "(mean, count)" pair per centroid, lossless means"""
    import ctypes as C
    import re
    from gyeeta_b200 import engine as ge
    L = ge.load_library()
    means = np.array([1.5, 2.25, 1000.000001, 123456789.123456789], dtype=np.float64)
    weights = np.array([1, 7, 3, 2], dtype=np.uint64)
    buf = C.create_string_buffer(512)
    n = L.gysk_tdigest_to_pgtext(means.ctypes.data_as(C.c_void_p), weights.ctypes.data_as(C.c_void_p), 4, 100, buf, len(buf))
    txt = buf.value.decode()
    assert n == len(txt)
    m = re.fullmatch(r"flags 1 count (\d+) compression (\d+) centroids (\d+)((?: \([^)]*\))*)", txt)
    assert m and int(m.group(1)) == 13 and int(m.group(2)) == 100 and int(m.group(3)) == 4
    pairs = re.findall(r"\(([^,]+), (\d+)\)", m.group(4))
    assert [float(a) for a, _ in pairs] == list(means) and [int(b) for _, b in pairs] == list(weights)
    small = C.create_string_buffer(40)
    assert L.gysk_tdigest_to_pgtext(means.ctypes.data_as(C.c_void_p), weights.ctypes.data_as(C.c_void_p), 4, 100, small, len(small)) == -28


def np_td_code(v):
    """numpy statement of the log-linear value code (oracle gyo_td_code): 32 bins per octave, exact below 32"""
    v = np.asarray(v, dtype=np.uint64)
    e = np.zeros(len(v), dtype=np.uint64)
    big = v >= 32
    e[big] = np.floor(np.log2(v[big].astype(np.float64))).astype(np.uint64)
    e[big] = np.where((np.uint64(1) << e[big]) > v[big], e[big] - np.uint64(1), e[big])        # guard float rounding at powers of two
    e[big] = np.where((np.uint64(2) << e[big]) <= v[big], e[big] + np.uint64(1), e[big])
    sh = np.where(big, e - np.uint64(5), np.uint64(0))
    return np.where(big, ((sh + np.uint64(1)) << np.uint64(5)) | ((v >> sh) & np.uint64(31)), v)


def test_td_code_is_monotone_and_matches_the_oracle():
    from oracle import pyoracle as po
    L = po.lib()
    rng = np.random.default_rng(2)
    v = np.unique(np.concatenate([np.arange(0, 5000), rng.integers(0, 1 << 30, 200_000), (1 << np.arange(5, 30)) - 1, 1 << np.arange(5, 30),
                                  [(1 << 30) - 1, 1_000_000_999]]).astype(np.uint64))
    code = np_td_code(v)
    assert np.array_equal(code, np.array([L.gyo_td_code(int(x)) for x in v], dtype=np.uint64))
    assert np.all(np.diff(code.astype(np.int64)) >= 0) and code.max() <= 831            # monotone; 832 codes + 15 buckets < NBINS = 848
    # bin index = code + RESP_TIME_HASH bucket of the msec value: monotone too, and one bucket per bin
    idx = code + np.array([L.gyo_bucket(0, int(x) // 1000) for x in v], dtype=np.uint64)
    assert np.all(np.diff(idx.astype(np.int64)) >= 0) and idx.max() < 848
    for i in np.unique(idx)[::5]:
        assert len({L.gyo_bucket(0, int(x) // 1000) for x in v[idx == i]}) == 1
    # a bin is at most 1/32 of its lower edge wide: 32 bins per octave
    for c in np.unique(code)[::7]:
        inb = v[code == c]
        assert inb.max() - inb.min() <= max(1, inb.min() // 32)


def test_listener_state_encoder_fields_and_limits():
    """gysk_encode_listener_state is pure host code: field mapping into LISTENER_STATE_NOTIFY (88-byte records, 8-byte aligned, no
    issue string), unknown ids skipped, 32-bit clamps, the 512-records-per-message cap (gy_comm_proto.h:2222) and ENOSPC"""
    import ctypes as C
    from gyeeta_b200 import engine as ge
    L = ge.load_library()
    LSN = np.dtype([("glob_id", "<u8"), ("nqrys_5s", "<u4"), ("total_resp_5sec", "<u4"), ("nconns", "<u4"), ("nconns_active", "<u4"),
                    ("ntasks", "<u4"), ("p95_5s", "<u4"), ("p95_5min", "<u4"), ("kb_in", "<u4"), ("kb_out", "<u4"), ("ser_errors", "<u4"),
                    ("cli_errors", "<u4"), ("t", "<u4", 6), ("ntasks_issue", "<u2"), ("is_http", "u1"), ("curr_state", "u1"),
                    ("curr_issue", "u1"), ("issue_bit_hist", "u1"), ("high_resp_bit_hist", "u1"), ("last_issue_subsrc", "u1"),
                    ("query_flags", "u1"), ("issue_string_len", "u1"), ("padding_len", "u1"), ("pad", "u1")])
    assert LSN.itemsize == 88
    n = 600
    sums = (ge.SvcSummary * n)()
    for i in range(n):
        sums[i].glob_id = 1000 + i
        sums[i].found = 0 if i % 7 == 3 else 1
        sums[i].nqrys_5s = 0 if i % 5 == 0 else 10 * i
        sums[i].total_resp_5sec = (1 << 40) if i == 1 else 3 * i
        sums[i].p95_5s_resp_ms = -1 if i == 2 else 30
        sums[i].p95_5min_resp_ms = 60
        sums[i].nconns_5s = i
        sums[i].kbytes_5s = 2 * i
        sums[i].curr_state, sums[i].curr_issue, sums[i].issue_bit_hist, sums[i].high_resp_bit_hist = i % 5, i % 9, i & 0xFF, (3 * i) & 0xFF
    buf = C.create_string_buffer(88 * 512)
    nrecs, nbytes = C.c_uint32(), C.c_uint32()
    assert L.gysk_encode_listener_state(sums, n, buf, len(buf), C.byref(nrecs), C.byref(nbytes)) == 0
    assert nrecs.value == 512 and nbytes.value == 88 * 512                       # one message holds 512 records
    recs = np.frombuffer(buf.raw[: nbytes.value], dtype=LSN)
    found_ids = [1000 + i for i in range(n) if i % 7 != 3][:512]
    assert list(recs["glob_id"]) == found_ids
    by = {int(r["glob_id"]): r for r in recs}
    assert by[1001]["total_resp_5sec"] == 0xFFFFFFFF and by[1002]["p95_5s"] == 0     # clamps
    r = by[1011]
    assert (r["nqrys_5s"], r["total_resp_5sec"], r["p95_5s"], r["p95_5min"], r["nconns"], r["kb_in"]) == (110, 33, 30, 60, 11, 22)
    assert (r["curr_state"], r["curr_issue"], r["issue_bit_hist"], r["high_resp_bit_hist"]) == (11 % 5, 11 % 9, 11, 33)   # the classifier's outputs
    assert r["issue_string_len"] == 0 and r["padding_len"] == 0
    small = C.create_string_buffer(88 * 3)
    assert L.gysk_encode_listener_state(sums, n, small, len(small), C.byref(nrecs), C.byref(nbytes)) == -28




def _state_in(**kw):
    from gyeeta_b200 import engine as ge
    x = ge.ListenerStateIn()
    for k, v in kw.items():
        setattr(x, k, v)
    return x


def test_listener_state_classifier_hand_cases():
    """TCP_LISTENER::get_curr_state (common/gy_socket_stat.cc:2020-2875), outcomes read off the reference for inputs that single out one
    rule each; product (gysk_classify_listener, host build of gysk_state.cuh) and oracle (gyo_listener_state) must both give them"""
    from gyeeta_b200 import engine as ge
    from oracle import pyoracle as po
    base = dict(r5p95=30, r5p99=60, r300p95=30, r300p99=60, r5dp95=30, r5dp99=60, r5dp25=10, rallp95=30, rallp99=60, nqrys_5s=500,
                total_resp_msec=10_000, tcount_5d=1_000_000, mean5=20.0, mean300=20.0, mean5d=20.0, meanall=20.0, qps_p95=200, qps_p25=50,
                act_p95=100, act_p25=10, secs_5d=10_000, last_qps_count=100, nconn=20, curr_active_conn=20)
    cases = [
        # :2122 no queries at all -> idle
        (dict(nqrys_5s=0, last_qps_count=0), 0, (ge.STATE_IDLE, ge.ISSUE_NONE, 0)),
        # :2139/:2143/:2145 response below the 5-day p95, QPS at or below its p25, nothing wrong -> idle
        (dict(r5p95=10, last_qps_count=40, nqrys_5s=200), 0, (ge.STATE_IDLE, ge.ISSUE_NONE, 0)),
        # :2139/:2229 fast responses but more than half of the queries are server errors -> severe
        (dict(r5p95=10, ser_errors=300), 0, (ge.STATE_SEVERE, ge.ISSUE_SERVER_ERRORS, 0)),
        # :2275-2277 faster than usual, QPS below its p95 -> good
        (dict(r5p95=10), 0b1, (ge.STATE_GOOD, ge.ISSUE_NONE, 0b10)),
        # :2287 faster than usual but QPS above its p95 (and less than two buckets faster) -> ok, QPS high
        (dict(r5p95=10, last_qps_count=300, nqrys_5s=1500), 0, (ge.STATE_OK, ge.ISSUE_QPS_HIGH, 0)),
        # :2307/:2419 same bucket as the 5-day p95, mean within 20 % -> ok
        (dict(), 0, (ge.STATE_OK, ge.ISSUE_NONE, 0)),
        # :2307/:2340/:2386 same bucket, mean 20 % below the 5-day mean -> good
        (dict(mean5=10.0), 0, (ge.STATE_GOOD, ge.ISSUE_NONE, 0)),
        # :2430/:2464 p95 three buckets above the 5-day and the 300-s p95, QPS 50 % above its p95 -> severe, QPS high; the high bit is set
        (dict(r5p95=150, r5p99=300, last_qps_count=300, nqrys_5s=1500, mean5=90.0), 0, (ge.STATE_SEVERE, ge.ISSUE_QPS_HIGH, 1)),
        # :2525 one bucket up, active connections above their p95 -> bad, active conns high
        (dict(r5p95=60, mean5=40.0, curr_active_conn=150, nconn=150), 0, (ge.STATE_BAD, ge.ISSUE_ACTIVE_CONN_HIGH, 1)),
        # :2748 one bucket up, nothing else unusual, high in only 3 of the last 8 windows -> ok
        (dict(r5p95=60, mean5=40.0, r300p95=60, curr_active_conn=10, nconn=10), 0b0101, (ge.STATE_OK, ge.ISSUE_NONE, 0b1011)),
        # :2771-2860 the same with the response high in 5 of the last 8 windows -> bad, source unknown
        (dict(r5p95=60, mean5=40.0, r300p95=60, curr_active_conn=10, nconn=10), 0b1111, (ge.STATE_BAD, ge.ISSUE_UNKNOWN, 0b11111)),
        # :2825 ... and the listener depends on other listeners -> their issue
        (dict(r5p95=60, mean5=40.0, r300p95=60, nserdepends=2, curr_active_conn=10, nconn=10), 0b1111, (ge.STATE_BAD, ge.ISSUE_DEPENDENT, 0b11111)),
        # :2710 ... or the slow buckets hold at most 3 connections each of 20 active ones -> a local effect, ok
        (dict(r5p95=60, mean5=40.0, r300p95=60), 0b1111, (ge.STATE_OK, ge.ISSUE_NONE, 0b11111)),
        # :2494 a process issue with a slow response -> listener tasks
        (dict(r5p95=60, mean5=40.0, task_issue=1, ntasks_issue=2), 0, (ge.STATE_BAD, ge.ISSUE_LISTENER_TASKS, 1)),
        # :2402-2415 the reference's fall-through: same bucket, lower mean, server errors without a process issue end as {ok, tasks}
        (dict(mean5=10.0, ser_errors=5), 0, (ge.STATE_OK, ge.ISSUE_LISTENER_TASKS, 0)),
    ]
    for i, (delta, hb, want) in enumerate(cases):
        x = _state_in(**{**base, **delta})
        assert ge.classify_listener(x, hb) == want, (i, delta)
        assert po.listener_state(x, hb) == want, (i, delta)


def test_listener_state_classifier_random_inputs_agree():
    """product and oracle restatements of the decision tree agree on 60 000 random inputs that reach every rule (operand types matter:
    uint32 products of ser_errors, float / double constants)"""
    from gyeeta_b200 import engine as ge
    from oracle import pyoracle as po
    rng = np.random.default_rng(21)
    vals = [0, 1, 10, 30, 60, 100, 150, 200, 300, 450, 700, 1000, 3000, 15000, 32767]
    qv = [-1, 1, 10, 50, 200, 500, 1000, 3000, 6000, 2147483647]
    av = [-1, 1, 5, 10, 25, 50, 75, 100, 32767]
    seen = set()
    for _ in range(60_000):
        x = ge.ListenerStateIn()
        base = int(rng.integers(1, 13))
        for f in ("r5p95", "r5p99", "r300p95", "r300p99", "r5dp95", "r5dp99", "r5dp25", "rallp95", "rallp99"):
            setattr(x, f, vals[int(np.clip(base + rng.integers(-2, 3), 0, 14))])
        x.nqrys_5s = int(rng.choice([0, 3, 40, 500, 20_000]))
        x.total_resp_msec = int(x.nqrys_5s * rng.integers(1, 200))
        x.tcount_5d = int(rng.integers(0, 10_000_000))
        m = float(rng.integers(1, 300))
        x.mean5, x.mean300, x.mean5d, x.meanall = m, m * float(rng.choice([0.7, 0.95, 1.0, 1.3])), m * float(rng.choice([0.7, 1.0, 1.15, 1.5])), m * float(rng.choice([0.8, 1.0, 1.2]))
        q = sorted(int(v) for v in rng.choice(qv, 2)); a = sorted(int(v) for v in rng.choice(av, 2))
        x.qps_p25, x.qps_p95, x.act_p25, x.act_p95 = q[0], q[1], a[0], a[1]
        x.secs_5d = int(rng.choice([1, 300, 432000]))
        x.last_qps_count = int(rng.choice([0, 2, 45, 210, 5000]))
        x.nconn, x.curr_active_conn = int(rng.integers(0, 200)), int(rng.integers(0, 200))
        x.ser_errors = int(rng.choice([0, 0, 0, 1, 30, 400, 0x90000000]))
        for b in range(15):
            x.nactive_conn_arr[b] = int(rng.integers(0, 6))
        if rng.random() < 0.4:
            x.task_issue, x.task_severe, x.task_delay = int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 2))
            x.cpu_issue, x.mem_issue = int(rng.integers(0, 2)), int(rng.integers(0, 2))
            x.ntasks_issue, x.ntasks_noissue = int(rng.integers(0, 4)), int(rng.integers(0, 4))
            x.tasks_delay_msec = int(rng.choice([0, 500, 5000, 10 ** 7]))
            x.nserdepends = int(rng.integers(0, 2))
        hb = int(rng.integers(0, 256))
        g, o = ge.classify_listener(x, hb), po.listener_state(x, hb)
        assert g == o, (g, o)
        seen.add(g[:2])
    assert len(seen) == 18, sorted(seen)            # every (state, issue) pair the tree can produce


def test_task_groupby_oracle_hand_case():
    """the CPU statement of row a15b on a hand-made walk (common/gy_task_handler.cc:763-872): pid slots, issue fields, float order"""
    from gyeeta_b200 import engine as ge, wire
    from oracle import pyoracle as po
    s = np.zeros(5, dtype=ge.PROC_SAMPLE_DTYPE)
    s["aggr_task_id"] = [7, 9, 7, 7, 9]
    s["pid"] = [100, 200, 101, 102, 201]
    s["cpu_pct"] = np.array([1e8, 3.0, 1.0, -1e8, 0.5], dtype=np.float32)      # (1e8 + 1) - 1e8 = 0 in float, 1 in any other order
    s["is_issue"] = [0, 1, 1, 1, 0]
    s["issue"] = [0, 4, 5, 6, 0]
    s["state"] = [2, 3, 4, 1, 2]
    s["issue_bit_hist"] = [1, 2, 4, 8, 16]; s["severe_issue_bit_hist"] = [1, 2, 4, 8, 16]
    s["rss_mb"] = [10, 20, 30, 40, 50]; s["cpu_delay_msec"] = [1, 2, 3, 4, 5]; s["tcp_kbytes"] = [0, 7, 0, 9, 0]
    s["comm"] = [b"a", b"b", b"c", b"d", b"e"]
    out = po.task_groupby(s, wire.TASK)
    assert list(out["aggr_task_id"]) == [7, 9]                                 # order of first appearance
    g7, g9 = out[0], out[1]
    assert g7["total_cpu_pct"] == np.float32(0.0) and g9["total_cpu_pct"] == np.float32(3.5)
    assert g7["ntasks_total"] == 3 and g7["ntasks_issue"] == 2 and g7["curr_state"] == 4 and g7["curr_issue"] == 6
    # pid slots: first process -> [0]; first issue process overwrites [0] (:764-766), second issue process -> [1]; the second
    # process of the group also lands in [1] (:864) before that
    assert list(g7["pid_arr"]) == [101, 102] and list(g9["pid_arr"]) == [200, 201]
    assert g7["issue_bit_hist"] == 12 and g7["severe_issue_bit_hist"] == 12 and g9["issue_bit_hist"] == 2
    assert g7["rss_mb"] == 80 and g7["cpu_delay_msec"] == 8 and g7["tcp_kbytes"] == 9 and g9["tcp_kbytes"] == 7
    assert g7["onecomm"] == b"a" and g9["onecomm"] == b"b"


def test_every_profile_named_in_the_docs_exists():
    """README.md / DESIGN.md / profiles/README.md quote measured numbers by file: a quoted file that is not in profiles/ is a number
    without evidence (gpurun_out/ is scratch and does not survive a session)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = set()
    for f in ("README.md", "DESIGN.md", os.path.join("profiles", "README.md"), "INTEGRATION.md"):
        t = open(os.path.join(root, f)).read()
        names |= set(m.group(1) for m in re.finditer(r"`(?:profiles/)?((?:r0\d|ncu)_[A-Za-z0-9_.]+\.(?:json|csv|md|log|txt))`", t))
    assert len(names) > 20
    missing = sorted(n for n in names if not os.path.exists(os.path.join(root, "profiles", n)))
    assert not missing, missing


def test_hot_row_layout_keeps_neighbouring_bins_on_different_lines():
    """DESIGN.md §3: L2 applies same-line atomics one after the other, and neighbouring value bins fill up together — the row layout
    must be a bijection of the 848 bins into the 1024 words of a half row with neighbours at least two 128-byte lines (32 words) apart"""
    L = C.CDLL(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gyeeta_b200", "libgysketch.so"))
    L.gysk_hot_row_word.restype = C.c_uint32
    L.gysk_hot_row_word.argtypes = [C.c_uint32]
    words = [L.gysk_hot_row_word(b) for b in range(848)]
    assert len(set(words)) == 848 and max(words) < 1024
    assert L.gysk_hot_row_word(848) == 0xFFFFFFFF
    for d in range(1, 9):                                  # the bins around a mode: none of them shares a line with another
        assert all(abs(words[b + d] - words[b]) // 16 >= 1 for b in range(848 - d)), d
    assert all(abs(words[b + 1] - words[b]) >= 32 for b in range(847) if (b & 31) != 31)
    lines = [w // 16 for w in words]
    for b in range(0, 848 - 16):
        assert len(set(lines[b: b + 16])) == 16, b         # any 16 consecutive bins: 16 different lines


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the product arm): one JSON line with the product arm's metric,
    unit, direction and config, its own cpu_baseline and an e2e that repeats the value with no host-device bytes"""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "60000"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "events/sec aggregated" and d["unit"] == "events/s" and d["higher_is_better"] is True
    assert d["config"]["workload"].startswith("configs[2]") and d["config"]["events_per_step_per_gpu"] == 100_000_000
    assert d["sample_events_per_step"] == 60000 and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 leave without work
    r2 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=120, cwd=root, env={**os.environ, "RANK": "1", "WORLD_SIZE": "2"})
    assert r2.returncode == 0 and not r2.stdout.strip()
