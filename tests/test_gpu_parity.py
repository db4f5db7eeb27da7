"""GPU parity tests proper: the CUDA path (through the C ABI of libgysketch.so) against the CPU oracle on the same seeded
inputs. Integer state is compared bit for bit; t-digest quantiles within the stated epsilon."""
import ctypes as C
import os

import numpy as np
import pytest

from gyeeta_b200 import engine as ge
from gyeeta_b200 import synth
from oracle import pyoracle as po
from tests.util import assert_hist_equal, exact_quantile, feed_both, make_pair, td_p99_tolerance

pytestmark = pytest.mark.gpu

TD_BATCHED_REL_EPS = 0.0   # GPU vs the CPU t-digest path: same IEEE operation sequence (no libm in the loop) => identical bits
TD_REL_EPS = 0.01          # north-star epsilon: p50 / p95 within 1 % of the classic buffered CPU t-digest AND of the exact quantile
TD_P99_EXACT_EPS = 0.01    # SURVEY §8c-4: p99 within 1 % of the exact quantile too (the engine keeps delta = 200); below 150 K samples per
                           # service the sample's own order-statistic noise exceeds that: tests.util.td_p99_tolerance(n)
TD_RANK_EPS = 0.001        # |F(estimate) - q| on the exact empirical CDF


def test_counters_and_edge_cases():
    eng, orc = make_pair(max_svcs=64, max_tasks=16, max_batch=4096)
    ev = np.zeros(12, dtype=ge.EVENT_DTYPE)
    ev["svc_id"] = [0, 5, 5, 5, 6, 7, 7, 8, 9, 9, 5, 5]
    ev["type"] = [5, 5, 9, 0, 5, 2, 4, 6, 6, 5, 1, 3]
    ev["value"] = [10, 1_000_001_000, 1, 1, 999, 4096, 1 << 31, 3001, 0xFFFFFFFF, 1_000_000_999, 1023, 1024]
    ev["flow_key"] = [1, 2, 3, 4, 5, 6, 6, (70000 << 32) | 65001, 0xFFFFFFFF_80000000, 7, 8, 9]
    feed_both(eng, orc, ev, 4096)
    s, o = eng.stats(), orc.counters()
    assert s["events_in"] == o["in"] == 12
    assert s["events_dropped"] == o["dropped"] == 4            # svc 0, value beyond 1e6 msec, type 9, type 0
    assert (s["events_resp"], s["events_tcp"], s["events_task"]) == (o["resp"], o["tcp"], o["task"]) == (2, 4, 2)
    assert s["nsvcs"] == o["nsvcs"] and s["ntasks"] == o["ntasks"]
    for id_ in (5, 6, 7, 9):
        assert_hist_equal(eng, orc, id_, ge.HIST_RESP_CUR)
    for id_ in (8, 9):
        for which in (ge.HIST_TASK_CPU_PCT, ge.HIST_TASK_CPU_DELAY, ge.HIST_TASK_BLKIO_DELAY):
            assert_hist_equal(eng, orc, id_, which)
    assert eng.export_hist(12345, ge.HIST_RESP_CUR) is None
    assert np.array_equal(eng.export_cms(), orc.cms())
    # empty ingest is a no-op
    eng.ingest_events(ev[:0])
    eng.sync()
    assert eng.stats()["events_in"] == 12


def test_table_full_and_no_auto_register():
    eng, orc = make_pair(max_svcs=8, max_tasks=4, max_batch=2048, auto_register=False)
    ids = synth.service_ids(8)
    eng.register_ids(ids[:4]); orc.register_ids(ids[:4])
    rng = np.random.default_rng(3)
    ev = np.zeros(2000, dtype=ge.EVENT_DTYPE)
    ev["svc_id"] = ids[rng.integers(0, 8, len(ev))]
    ev["type"] = ge.EV_RESP
    ev["value"] = rng.integers(0, 50_000_000, len(ev))
    feed_both(eng, orc, ev, 2048)
    s, o = eng.stats(), orc.counters()
    assert s["events_dropped"] == o["dropped"] > 0 and s["nsvcs"] == o["nsvcs"] == 4
    for id_ in ids:
        assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_CUR)

    # auto-register with more distinct ids than capacity: exactly max_svcs services survive, the rest is dropped.
    eng2 = ge.Engine(max_svcs=8, max_tasks=4, max_batch=2048)
    ev["svc_id"] = synth.service_ids(64)[rng.integers(0, 64, len(ev))]
    eng2.ingest_events(ev); eng2.sync()
    s2 = eng2.stats()
    assert s2["nsvcs"] == 8 and s2["events_resp"] + s2["events_dropped"] == len(ev) and s2["events_dropped"] > 0
    kept = [i for i in synth.service_ids(64) if eng2.export_hist(int(i), ge.HIST_RESP_CUR) is not None]
    assert len(kept) == 8
    tot = sum(eng2.export_hist(int(i), ge.HIST_RESP_CUR)[1] for i in kept)
    assert tot == s2["events_resp"]


@pytest.mark.parametrize("nsvc,n,batch", [(50, 20_000, 8192), (3000, 300_000, 1 << 17)])
def test_mixed_stream_bit_exact(nsvc, n, batch):
    rng = np.random.default_rng(11)
    ev = synth.gen_mixed(rng, n, nsvc, ntask=max(nsvc // 4, 4), nhosts=64, nclients=20_000)
    eng, orc = make_pair(max_svcs=4096, max_tasks=1024, max_batch=batch, cms_log2_width=16)
    feed_both(eng, orc, ev, batch)
    s, o = eng.stats(), orc.counters()
    for k, ko in (("events_in", "in"), ("events_dropped", "dropped"), ("events_resp", "resp"), ("events_tcp", "tcp"),
                  ("events_task", "task"), ("nsvcs", "nsvcs"), ("ntasks", "ntasks")):
        assert s[k] == o[ko], k
    assert s["kernel_launches"] > 0
    # count-min: whole table, bit for bit
    assert np.array_equal(eng.export_cms(), orc.cms())
    svc = np.unique(ev["svc_id"][ev["type"] != ge.EV_TASK])
    tasks = np.unique(ev["svc_id"][ev["type"] == ge.EV_TASK])
    pick = svc if len(svc) <= 200 else np.concatenate([svc[:100], rng.choice(svc, 100, replace=False)])
    nresp = 0
    for id_ in pick:
        nresp += assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_CUR)
        a, b = eng.export_hll(int(id_)), orc.export_hll(int(id_))
        assert np.array_equal(a, b), hex(int(id_))
        # CONN_BITMAP (gy_socket_stat.h:390-455): masks and get_conn_breakup() counts
        bm_g, bm_o = eng.export_conn_bitmap(int(id_)), orc.export_conn_bitmap(int(id_))
        assert np.array_equal(bm_g[0], bm_o[0]) and np.array_equal(bm_g[1], bm_o[1]), hex(int(id_))
        assert eng.L.gysk_hll_estimate(a.ctypes.data_as(C.c_void_p), 12) == po.lib().gyo_hll_estimate(po._p(b), 12)
    assert nresp > 0
    for id_ in tasks[:100]:
        for which in (ge.HIST_TASK_CPU_PCT, ge.HIST_TASK_CPU_DELAY, ge.HIST_TASK_BLKIO_DELAY):
            assert_hist_equal(eng, orc, int(id_), which)
    # point queries = min over rows of both halves
    keys = np.unique(ev["flow_key"][(ev["type"] >= 1) & (ev["type"] <= 4)])[:500]
    est = eng.query_flows(keys)
    tbl = orc.cms().reshape(4, -1)
    for k, e_ in zip(keys[:50], est[:50]):
        cells = [tbl[r, po.lib().gyo_cms_index(int(k), r, 16)] for r in range(4)]
        assert e_["count"] == min(int(c) & 0xFFFFFFFF for c in cells)
        assert e_["kbytes"] == min(int(c) >> 32 for c in cells)


def test_flush_window_roll_and_summary(golden_dir):
    rng = np.random.default_rng(5)
    eng, orc = make_pair(max_svcs=512, max_tasks=64, max_batch=1 << 15, cms_log2_width=14)
    ids = None
    for w in range(3):
        ev = synth.gen_mixed(rng, 40_000, 100, ntask=16, nhosts=8, nclients=5000)
        ids = np.unique(ev["svc_id"][ev["type"] != ge.EV_TASK]) if ids is None else ids
        feed_both(eng, orc, ev, 1 << 15)
        cms_before = orc.cms()
        eng.flush(5 * (w + 1)); orc.flush(5 * (w + 1))
        assert np.array_equal(eng.export_cms(last_window=True), cms_before)
        assert not eng.export_cms().any()
        for id_ in ids[:40]:
            for which in (ge.HIST_RESP_CUR, ge.HIST_RESP_LAST, ge.HIST_RESP_ALL):
                assert_hist_equal(eng, orc, int(id_), which)
            for lw in (False, True):
                g, o = eng.export_conn_bitmap(int(id_), lw), orc.export_conn_bitmap(int(id_), lw)
                assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1])
            assert not eng.export_conn_bitmap(int(id_))[0].any()          # cleared with the window
    gold = np.load(os.path.join(golden_dir, "summary_pct_golden.npz"))
    summ = eng.query_svcs(ids[:40])
    assert len(summ) == len(gold["ids"])
    for i, (sm, id_) in enumerate(zip(summ, ids[:40])):
        last, total, mx = orc.export_hist(int(id_), ge.HIST_RESP_LAST)
        cur, last_c, all_cnt, all_kb = orc.export_conn(int(id_))
        assert sm["found"] == 1 and sm["nqrys_5s"] == total and sm["total_resp_5sec"] == int(last["sum"].sum())
        assert (sm["nconns_5s"], sm["kbytes_5s"]) == (last_c & 0xFFFFFFFF, last_c >> 32)
        assert (sm["nconns_all"], sm["kbytes_all"]) == (all_cnt, all_kb)
        # percentiles must be what the REFERENCE's own get_percentiles returned for this serial form (tests/golden/make_golden.py)
        assert id_ == gold["ids"][i] and total == gold["total"][i] and mx == gold["max"][i]
        assert np.array_equal(last["count"], gold["count"][i]) and np.array_equal(last["sum"], gold["sum"][i])
        assert [sm["p95_5s_resp_ms"], sm["p99_5s_resp_ms"], sm["p25_5s_resp_ms"]] == gold["pct"][i].tolist()
    assert eng.query_svcs([424242])[0]["found"] == 0


def test_window_membership_is_by_arrival():
    """the tsec contract (include/gysketch.h): a sample belongs to the window that is open when it ARRIVES, whatever its own tsec says —
    the reference stamps response samples with time(nullptr) of their processing (common/gy_socket_stat.cc:1560-1579) and
    gysk_flush(tsec) closes the window. Events stamped in the past, the future and with garbage land in the window they were fed in."""
    rng = np.random.default_rng(9)
    eng, orc = make_pair(max_svcs=256, max_tasks=16, max_batch=1 << 14)
    evs = []
    for w, stamp in enumerate((lambda n: np.zeros(n), lambda n: np.full(n, 10_000), lambda n: rng.integers(0, 1 << 32, n))):
        ev = synth.gen_mixed(rng, 20_000, 50, ntask=8, nhosts=4, nclients=1000)
        ev["tsec"] = stamp(len(ev)).astype(np.uint32)
        ev["tsec"][ev["type"] == ge.EV_ACTIVE] = 0
        evs.append(ev)
        feed_both(eng, orc, ev, 1 << 14)
        eng.flush(100 + 5 * w); orc.flush(100 + 5 * w)
        resp = ev[ev["type"] == ge.EV_RESP]
        for id_ in np.unique(resp["svc_id"])[:20]:
            assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_LAST)
            _cells, total, _mx = eng.export_hist(int(id_), ge.HIST_RESP_LAST)
            assert total == int((resp["svc_id"] == id_).sum())               # exactly this window's samples, none of the others'


def test_tdigest_quantiles_config1_shape():
    """config 1 shape (scaled to 200 K samples here; the 1 M version lives in the full-size test): one service"""
    rng = np.random.default_rng(1)
    ev = synth.gen_resp_config1(rng, 200_000)
    id_ = int(ev["svc_id"][0])
    eng, orc = make_pair(max_svcs=16, max_tasks=4, max_batch=1 << 16)
    feed_both(eng, orc, ev, 1 << 16)
    means, weights, mn, mx = eng.export_tdigest(id_)
    td = orc.export_tdigest(id_)
    omeans, oweights = td.centroids()
    assert int(weights.sum()) == len(ev) == td.total
    assert mn == ev["value"].min() and mx == ev["value"].max()
    assert np.all(np.diff(means) >= 0)
    # same batched algorithm on both sides: centroid for centroid
    assert len(means) == len(omeans) and np.array_equal(weights, oweights)
    assert np.array_equal(means, omeans)
    classic = po.td_add(po.td_new(), ev["value"], classic=True)
    qs = [0.5, 0.95, 0.99]
    got = eng.quantiles(id_, qs)
    sv = np.sort(ev["value"])
    for q, g in zip(qs, got):
        ex = exact_quantile(ev["value"], q)
        eps = TD_REL_EPS if q < 0.99 else td_p99_tolerance(len(ev), TD_P99_EXACT_EPS)
        assert abs(g - ex) / ex < eps, (q, g, ex)
        assert abs(g - po.td_quantile(classic, q)) / ex < eps, (q, g)
        assert abs(g - po.td_quantile(td, q)) / ex <= TD_BATCHED_REL_EPS
        assert abs(np.searchsorted(sv, g) / len(sv) - q) < TD_RANK_EPS, (q, g)
    # consistency with the reference's bucketed answer: exact quantile lies in the bucket whose upper threshold
    # GY_HISTOGRAM::get_percentile returns (+- one bucket at the boundary, float cut-off)
    hist, total, _ = eng.export_hist(id_, ge.HIST_RESP_CUR)
    out = np.zeros(3, dtype=np.int64)
    pcts = np.array([50, 95, 99], dtype=np.float32)
    eng.L.gysk_hist_percentiles(0, 0, hist.ctypes.data_as(C.c_void_p), total, pcts.ctypes.data_as(C.c_void_p), 3,
                                out.ctypes.data_as(C.c_void_p))
    for q, thr in zip(qs, out):
        b_exact = eng.L.gysk_hist_bucket(0, int(exact_quantile(ev["value"], q) // 1000))
        b_ref = eng.L.gysk_hist_bucket(0, int(thr))
        assert abs(b_exact - b_ref) <= 1


def test_tdigest_many_services_skewed():
    rng = np.random.default_rng(21)
    ev = synth.gen_mixed(rng, 400_000, 500, ntask=8, nhosts=16, nclients=5000, zipf_s=1.05)
    eng, orc = make_pair(max_svcs=1024, max_tasks=64, max_batch=1 << 17, cms_log2_width=14)
    feed_both(eng, orc, ev, 1 << 17)
    resp = ev[ev["type"] == ge.EV_RESP]
    ids, counts = np.unique(resp["svc_id"], return_counts=True)
    order = np.argsort(-counts)
    checked = 0
    for j in list(order[:10]) + list(order[len(order) // 2: len(order) // 2 + 10]) + list(order[-10:]):
        id_ = int(ids[j])
        vals = resp["value"][resp["svc_id"] == ids[j]]
        means, weights, mn, mx = eng.export_tdigest(id_)
        td = orc.export_tdigest(id_)
        om, ow = td.centroids()
        assert int(weights.sum()) == len(vals)
        assert np.array_equal(weights, ow) and np.array_equal(means, om)
        if len(vals) >= 10_000:
            sv = np.sort(vals)
            for q, g in zip([0.5, 0.95, 0.99], eng.quantiles(id_, [0.5, 0.95, 0.99])):
                ex = exact_quantile(vals, q)
                assert abs(g - ex) / ex < (TD_REL_EPS if q < 0.99 else td_p99_tolerance(len(vals), TD_P99_EXACT_EPS)), (len(vals), q, g, ex)
                assert abs(g - po.td_quantile(td, q)) / ex <= TD_BATCHED_REL_EPS
                assert abs(np.searchsorted(sv, g) / len(sv) - q) < 2 * TD_RANK_EPS, (len(vals), q, g)
            checked += 1
    assert checked >= 3
    # services without any RESP sample have an empty digest
    only_tcp = np.setdiff1d(np.unique(ev["svc_id"][ev["type"] <= 4]), ids)
    if len(only_tcp):
        m, w, _, _ = eng.export_tdigest(int(only_tcp[0]))
        assert len(m) == 0


def test_hll_estimate_within_3_sigma():
    rng = np.random.default_rng(9)
    eng, _ = make_pair(max_svcs=16, max_tasks=4, max_batch=1 << 18)
    ev = np.zeros(300_000, dtype=ge.EVENT_DTYPE)
    ev["svc_id"] = 77
    ev["type"] = ge.EV_ACCEPT
    ev["flow_key"] = rng.integers(0, 1 << 63, len(ev), dtype=np.uint64)
    ev["flow_key"][100_000:] = ev["flow_key"][:200_000]      # duplicates
    eng.ingest_events(ev); eng.sync()
    exact = len(np.unique(ev["flow_key"]))
    est = eng.query_svcs([77])[0]["distinct_clients"]
    assert abs(est - exact) / exact < 3 * 1.04 / np.sqrt(4096)
    # CMS never underestimates, and the overshoot stays inside e/width * N
    keys, cnt = np.unique(ev["flow_key"], return_counts=True)
    est_f = eng.query_flows(keys[:2000])
    assert np.all(est_f["count"] >= cnt[:2000])
    over = est_f["count"] - cnt[:2000]
    assert np.mean(over <= np.e / (1 << 20) * len(ev) + 1) > 0.995 and over.max() <= 4       # the e/w * N bound holds with probability 1 - e^-depth


def test_sharded_engines_merge_to_single_engine_integers():
    """host-id sharding (SURVEY.md §8e): two shard engines vs one engine over the full stream — the additive integer state
    (CMS cells) of the shards sums to the single-engine table bit for bit; per-service state lives wholly on one shard."""
    rng = np.random.default_rng(33)
    ev = synth.gen_mixed(rng, 100_000, 300, ntask=32, nhosts=64, nclients=5000)
    one = ge.Engine(max_svcs=1024, max_tasks=128, max_batch=1 << 16, cms_log2_width=14)
    one.ingest_events(ev); one.sync()
    shards = [ge.Engine(max_svcs=1024, max_tasks=128, max_batch=1 << 16, cms_log2_width=14, rank=r, world=2) for r in range(2)]
    for s in shards:
        s.ingest_events(ev); s.sync()               # every engine sees the stream, keeps host_idx % 2 == rank
    assert np.array_equal(shards[0].export_cms() + shards[1].export_cms(), one.export_cms())
    assert sum(s.stats()["events_in"] for s in shards) == len(ev)
    for id_ in np.unique(ev["svc_id"][ev["type"] == ge.EV_RESP])[:50]:
        owners = [s.export_hist(int(id_), ge.HIST_RESP_CUR) for s in shards]
        full = one.export_hist(int(id_), ge.HIST_RESP_CUR)
        got = [o for o in owners if o is not None]
        assert sum(int(o[1]) for o in got) == full[1]


def test_rolling_levels_300s_and_5days():
    """multi-level windows (Level_5s_5min_5days_all, gy_statistics.h:1545-1551; 10 slots per level :1105): the 300-s and
    432000-s levels after a sequence of 5-s flushes with time jumps (the scenario of test/test_timeseries_hist.cc:29-72,
    which jumps +3600 s) — bit-exact against the oracle's slot rule, and expiry actually drops old windows."""
    rng = np.random.default_rng(77)
    eng, orc = make_pair(max_svcs=128, max_tasks=8, max_batch=1 << 14, cms_log2_width=10)
    times = [5, 10, 15, 35, 65, 300, 305, 310, 3905, 3910, 50_000, 50_005, 500_000, 500_005]
    ids = None
    for t in times:
        ev = synth.gen_mixed(rng, 8000, 40, ntask=4, nhosts=4, nclients=500)
        ev["tsec"] = t
        ids = np.unique(ev["svc_id"][ev["type"] == ge.EV_RESP])[:25] if ids is None else ids
        feed_both(eng, orc, ev, 1 << 14)
        eng.flush(t); orc.flush(t)
        for id_ in ids[:10]:
            for which in (ge.HIST_RESP_LAST, ge.HIST_RESP_5MIN, ge.HIST_RESP_5DAY, ge.HIST_RESP_ALL):
                assert_hist_equal(eng, orc, int(id_), which)
    # after the jump to t = 500 005 the 300-s level only holds the last two windows, the 5-day level (span 432 000 s) has
    # dropped everything recorded before t = 68 005 and "all" still has everything
    sm = eng.query_svcs(ids[:10])
    for s_, id_ in zip(sm, ids[:10]):
        h5m = orc.export_hist(int(id_), 6); h5d = orc.export_hist(int(id_), 7); hall = orc.export_hist(int(id_), 2)
        assert s_["nqrys_5min"] == h5m[1] and s_["nqrys_5day"] == h5d[1] and s_["nqrys_all"] == hall[1]
        assert s_["nqrys_5min"] <= s_["nqrys_5day"] < s_["nqrys_all"]
        pc = np.zeros(1, dtype=np.int64)
        p95 = np.array([95], dtype=np.float32)
        ser = np.zeros(15, dtype=ge.SERIAL_DTYPE); ser[:] = h5m[0]
        eng.L.gysk_hist_percentiles(0, 0, ser.ctypes.data_as(C.c_void_p), h5m[1], p95.ctypes.data_as(C.c_void_p), 1, pc.ctypes.data_as(C.c_void_p))
        assert s_["p95_5min_resp_ms"] == pc[0]


def test_topn_services_last_window():
    """device top-N (score + radix sort) against numpy over the oracle's last-window state; per-host filter included"""
    rng = np.random.default_rng(15)
    eng, orc = make_pair(max_svcs=2048, max_tasks=16, max_batch=1 << 16, cms_log2_width=12)
    ev = synth.gen_mixed(rng, 120_000, 700, ntask=8, nhosts=16, nclients=3000)
    feed_both(eng, orc, ev, 1 << 16)
    eng.flush(5); orc.flush(5)
    ids = np.unique(ev["svc_id"][ev["type"] != ge.EV_TASK])
    host_of = {int(i): int(ev["host_idx"][np.argmax(ev["svc_id"] == i)]) for i in ids}
    qps = {int(i): (orc.export_hist(int(i), 1) or (None, 0, 0))[1] for i in ids}
    conn = {int(i): orc.export_conn(int(i))[1] for i in ids}
    for metric, score in ((0, qps), (1, {k: v & 0xFFFFFFFF for k, v in conn.items()}), (2, {k: v >> 32 for k, v in conn.items()})):
        got = eng.topn(metric, 10)
        want = sorted(score.values(), reverse=True)[:10]
        assert [s for _, s, _ in got] == [w for w in want if w > 0]
        for gid, s, h in got:
            assert score[gid] == s and host_of[gid] == h
    h = host_of[int(ids[0])]
    got = eng.topn(0, 5, host_idx=h)
    want = sorted([v for k, v in qps.items() if host_of[k] == h], reverse=True)[:5]
    assert [s for _, s, _ in got] == [w for w in want if w > 0] and all(hh == h for _, _, hh in got)


def test_idle_service_eviction_and_slot_reuse():
    """SURVEY §8f-1: a service without events for idle_evict_secs (and older than twice that) is evicted at a flush — the
    listener deletion rule of common/gy_socket_stat.cc:3968-3982 with TIMEOUT_INET_DIAG_SECS (gy_socket_stat.h:997). Same
    evicted ids as the oracle at every flush, evicted ids answer "unknown", their slots are handed to new ids (capacity is
    tight on purpose), a returning id starts from scratch, and the survivors' state stays bit-exact."""
    rng = np.random.default_rng(91)
    nsvc = 60
    eng, orc = make_pair(max_svcs=64, max_tasks=8, max_batch=1 << 14, cms_log2_width=10, idle_evict_secs=300)
    base = synth.gen_mixed(rng, 20_000, nsvc, ntask=4, nhosts=4, nclients=500)
    all_ids = np.unique(base["svc_id"][base["type"] != ge.EV_TASK])
    assert len(all_ids) >= 50
    keep = set(int(i) for i in all_ids[::2])            # these stay busy; the others go silent after t = 10

    def window(t, ids_allowed, n=6000, extra=None):
        ev = synth.gen_mixed(rng, n, nsvc, ntask=4, nhosts=4, nclients=500)
        is_task = ev["type"] == ge.EV_TASK
        ok = is_task | np.isin(ev["svc_id"], np.fromiter(ids_allowed, dtype=np.uint64))
        ev = ev[ok]
        if extra is not None:
            ev = np.concatenate([ev, extra])
        ev["tsec"] = t
        feed_both(eng, orc, ev, 1 << 14)
        eng.flush(t); orc.flush(t)
        got = np.sort(eng.evicted_ids())
        want, _tot = orc.evicted_ids()
        assert np.array_equal(got, np.sort(want)), (t, got, want)
        return got

    evicted = set()
    window(5, set(int(i) for i in all_ids))
    window(10, set(int(i) for i in all_ids))
    for t in (100, 200, 305, 311, 400, 500, 606, 611, 700):
        ev_ids = window(t, keep)
        evicted |= set(int(i) for i in ev_ids)
    silent = set(int(i) for i in all_ids) - keep
    assert evicted == silent                              # last active at t = 10, first seen t = 5: gone once t > 610
    st = eng.stats()
    assert st["svcs_evicted"] == len(silent) and st["nsvcs"] == orc.nsvcs() == len(keep)
    sm = eng.query_svcs(np.array(sorted(silent), dtype=np.uint64))
    assert all(s_["found"] == 0 for s_ in sm)
    for id_ in sorted(keep)[:12]:
        for which in (ge.HIST_RESP_LAST, ge.HIST_RESP_5MIN, ge.HIST_RESP_ALL):
            assert_hist_equal(eng, orc, id_, which)
        assert np.array_equal(eng.export_hll(id_), orc.export_hll(id_))

    # 30 new ids + one returning id: more than the 64-slot table could hold without recycling (30 live + 31 new > 64 - 30)
    new_ids = synth.splitmix64(np.arange(1, 31, dtype=np.uint64) + np.uint64(1 << 50))
    back = sorted(silent)[0]
    extra = np.zeros(3100, dtype=ge.EVENT_DTYPE)
    extra["svc_id"] = np.concatenate([np.repeat(new_ids, 100), np.full(100, back, dtype=np.uint64)])
    extra["type"] = ge.EV_RESP
    extra["value"] = rng.integers(100, 900_000, len(extra))
    extra["flow_key"] = rng.integers(1, 1 << 60, len(extra), dtype=np.uint64)
    window(705, keep, extra=extra)
    st2 = eng.stats()
    assert st2["nsvcs"] == orc.nsvcs() == len(keep) + 31
    for id_ in [back] + [int(i) for i in new_ids[:8]] + sorted(keep)[:6]:
        for which in (ge.HIST_RESP_LAST, ge.HIST_RESP_ALL):
            assert_hist_equal(eng, orc, id_, which)
        (means, weights, mn, mx), td = eng.export_tdigest(id_), orc.export_tdigest(id_)
        om, ow = td.centroids()
        assert np.array_equal(means, om) and np.array_equal(weights, ow) and mn == td.minv and mx == td.maxv
        if id_ == back or id_ in set(int(i) for i in new_ids):
            assert int(weights.sum()) == 100
    hb = eng.export_hist(back, ge.HIST_RESP_ALL)
    assert hb[1] == 100                                   # nothing of its first life is left


def test_topn_tasks_last_window():
    """device task top-N (atask_top_cpu_ / _cpu_delay_ / _io_delay_, server/gy_mconnhdlr.cc:10020-10065) over the last closed
    window = histogram totals differenced between flushes, against the oracle's task windows; second window differs from the
    first (the score must be the window's, not the running total)"""
    rng = np.random.default_rng(23)
    eng, orc = make_pair(max_svcs=256, max_tasks=512, max_batch=1 << 16, cms_log2_width=10)
    for t in (5, 10):
        ev = synth.gen_mixed(rng, 60_000, 50, ntask=300, nhosts=4, nclients=500)
        ev["tsec"] = t
        feed_both(eng, orc, ev, 1 << 16)
        eng.flush(t); orc.flush(t)
        tids = np.unique(ev["svc_id"][ev["type"] == ge.EV_TASK])
        for metric in (0, 1, 2):
            want = {}
            for i in tids:
                w = orc.task_last(int(i))
                if w is not None and w[2 * metric + 1] > 0:
                    want[int(i)] = min(int(w[2 * metric + 1]), 0xFFFFFFFF)
            got = eng.topn_tasks(metric, 10)
            top = sorted(want.values(), reverse=True)[:10]
            assert [sc for _, sc in got] == top, (t, metric)
            assert all(want[i] == sc for i, sc in got)


def test_full_value_range_keys():
    """response times over the whole 30-bit usec range incl. the largest value the validity rule lets through (all 832 codes in
    play), 1500 services: histograms, min / max and t-digest centroids stay bit-exact vs the oracle."""
    rng = np.random.default_rng(41)
    nsvc = 1500
    eng, orc = make_pair(max_svcs=2048, max_tasks=8, max_batch=1 << 18, cms_log2_width=10)
    ids = synth.service_ids(nsvc)
    n = 200_000
    ev = np.zeros(n, dtype=ge.EVENT_DTYPE)
    ev["svc_id"] = ids[rng.integers(0, nsvc, n)]
    ev["type"] = ge.EV_RESP
    ev["value"] = np.minimum(np.exp(rng.normal(np.log(2000.0), 3.0, n)), 1.0e9).astype(np.uint32)
    ev["value"][:50] = 1_000_000_999                     # the largest value the validity rule lets through (msec 1 000 000)
    ev["flow_key"] = rng.integers(1, 1 << 60, n, dtype=np.uint64)
    assert int(ev["value"].max()).bit_length() == 30
    feed_both(eng, orc, ev, 1 << 18)
    for id_ in ids[:40]:
        assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_CUR)
        got = eng.export_tdigest(int(id_)); td = orc.export_tdigest(int(id_))
        if got is None:
            assert td is None
            continue
        om, ow = td.centroids()
        assert np.array_equal(got[0], om) and np.array_equal(got[1], ow) and got[2] == td.minv and got[3] == td.maxv


def test_listener_state_per_window_equals_oracle():
    """row a10: the state decision of the 5-s reducer (TCP_LISTENER::get_curr_state behind listener_stats_update,
    common/gy_socket_stat.cc:4111-4272) evaluated on the device at every flush: qps_hist_ / active_conn_hist_ samples, level statistics,
    connection counts from ACTIVE_CONN_STATS and CONN_BITMAP, server errors, the two bit histories. Engine == oracle for every service
    and window; the stream turns slow / error-prone / busy half way so that several rules fire."""
    rng = np.random.default_rng(31)
    nsvc = 40
    eng, orc = make_pair(max_svcs=256, max_tasks=16, max_batch=1 << 14)
    ids = synth.service_ids(nsvc)
    seen_states = set()
    for w in range(30):
        n = 6000
        ev = np.zeros(n, dtype=ge.EVENT_DTYPE)
        k = rng.integers(0, nsvc, n)
        ev["svc_id"] = ids[k]
        ev["type"] = ge.EV_RESP
        slow = (w >= 14) & (k % 4 == 0)                                   # every 4th service turns 8x slower from window 14 on
        ev["value"] = np.minimum(np.exp(rng.normal(np.log(20_000.0), 1.0, n)) * np.where(slow, 8.0, 1.0), 9e8).astype(np.uint32)
        ev["flow_key"] = rng.integers(0, 1 << 16, n)
        err = (w >= 10) & (k % 5 == 1) & (rng.random(n) < (0.7 if w % 2 else 0.15))   # some services answer with server errors
        ev["flags"] = np.where(err, ge.EVF_SER_ERROR, 0)
        if w >= 18:                                                       # services 2, 6, 10 ... get 6x the queries
            extra = ev[(k % 4 == 2)]
            ev = np.concatenate([ev] + [extra] * 5)
        act = np.zeros(nsvc, dtype=ge.EVENT_DTYPE)
        act["svc_id"] = ids; act["type"] = ge.EV_ACTIVE; act["flow_key"] = 77
        act["flags"] = np.where((np.arange(nsvc) % 8 == 3) & (w >= 20), 400, 3 + (np.arange(nsvc) % 5)) if w % 3 == 0 else 0
        act = act[act["flags"] > 0]
        feed_both(eng, orc, np.concatenate([ev, act]), 1 << 14)
        eng.flush(1000 + 5 * (w + 1)); orc.flush(1000 + 5 * (w + 1))
        summ = eng.query_svcs(ids)
        for s_, id_ in zip(summ, ids):
            want = orc.export_state(int(id_))
            got = (s_["curr_state"], s_["curr_issue"], s_["issue_bit_hist"], s_["high_resp_bit_hist"])
            assert got == want[:4], (w, int(id_), got, want)
            seen_states.add(got[:2])
        for id_ in ids[:12]:
            for which in (ge.HIST_QPS, ge.HIST_ACTIVE_CONN):
                assert_hist_equal(eng, orc, int(id_), which)
    assert len(seen_states) >= 6, seen_states                             # idle / good / ok / bad / severe outcomes of several sources
    # issue ranking of the last window (a13): listeners with curr_state > OK, worst first
    bad = {int(id_): orc.export_state(int(id_))[0] for id_ in ids if orc.export_state(int(id_))[0] > ge.STATE_OK}
    top = eng.topn(ge.TOPN_ISSUE, 64)
    assert sorted((sid, sc) for sid, sc, _h in top) == sorted(bad.items()) and [sc for _s, sc, _h in top] == sorted(bad.values(), reverse=True)
