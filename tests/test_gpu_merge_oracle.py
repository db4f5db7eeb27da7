"""The logical merge step (gysk_merge_prepare / the collectives / gysk_merge_finish / gysk_query_logical) against a roll-up computed
on the CPU from the oracle. W engines on one GPU are ranks 0 .. W-1 of a host-sharded deployment; the collectives are emulated with
torch ops (tests.test_gpu_merge). One oracle per rank sees exactly that rank's events. For every logical id the expected answer is
built from the member services' oracle state:

  histograms       sum of the members' last-window / all-time histograms, percentiles by gysk_hist_percentiles
  connections      sums of the members' counters
  distinct clients the estimate of the byte-wise maximum of the members' HLL registers
  t-digest         replayed exactly as the kernels fold it: per rank, the members in map order (merge_compress(acc, member)), then
                   the ranks' digests in ascending rank order
  count-min        the row minimum over the sum of the ranks' tables"""
import numpy as np
import pytest

from gyeeta_b200 import engine as ge
from gyeeta_b200 import synth
from oracle import pyoracle as po
from tests.test_gpu_merge import _emulate_collectives
from tests.util import exact_quantile, make_pair, td_p99_tolerance

pytestmark = pytest.mark.gpu

NSVC, NHOSTS = 200, 64
NEVER = 0xDEAD0000BEEF                                      # mapped, never seen anywhere: every rank resolves it to the null slot


def _logical_map(rng, ids, tcp_ids):
    """{logical id: member glob ids}; returned as shuffled (glob, logical) pairs, so map order is neither id nor slot order"""
    groups = {7001: [ids[0]],                               # one member (the busiest service)
              7002: list(ids[1:65]),                        # 64 busy members on every rank: a fold chain far past TD_CAP
              7011: [NEVER],                                # no member exists
              7012: list(ids[129:133]),                     # ids[129] goes silent and is evicted before the last merge
              7013: list(tcp_ids)}                          # members that only ever sent TCP events
    for g in range(8):                                      # eight members on different hosts (=> ranks), one of them never seen
        groups[7003 + g] = list(ids[65 + 8 * g: 73 + 8 * g]) + ([NEVER + 1] if g == 3 else [])
    pairs = [(int(m), lid) for lid, ms in groups.items() for m in ms]
    pairs = [pairs[i] for i in rng.permutation(len(pairs))]
    return pairs


def _members_in_map_order(pairs, lid):
    return [g for g, l in pairs if l == lid]


def _expected(pairs, lid, orcs, delta, p, samples):
    """the CPU roll-up of one logical id from the per-rank oracles"""
    L = ge.load_library()
    members = _members_in_map_order(pairs, lid)
    last = np.zeros(15, dtype=ge.SERIAL_DTYPE); allh = np.zeros(15, dtype=ge.SERIAL_DTYPE)
    tot_last = tot_all = 0
    mx = np.iinfo(np.int64).min
    conn = [0, 0, 0, 0]
    regs = np.zeros(1 << p, dtype=np.uint8)
    slabs, tmin, tmax, tcount, vals = [], np.inf, -np.inf, 0, []
    for r, orc in enumerate(orcs):
        acc = (np.zeros(0), np.zeros(0, dtype=np.uint64))
        for m in members:
            h1 = orc.export_hist(m, ge.HIST_RESP_LAST)
            if h1 is None:
                continue                                    # not on this rank (or evicted): the null slot
            h2 = orc.export_hist(m, ge.HIST_RESP_ALL)
            for a, h in ((last, h1[0]), (allh, h2[0])):
                a["count"] += h["count"]; a["sum"] += h["sum"]
            tot_last += h1[1]; tot_all += h2[1]; mx = max(mx, h2[2])
            _cur, cl, ac, ak = orc.export_conn(m)
            conn[0] += cl & 0xFFFFFFFF; conn[1] += cl >> 32; conn[2] += ac; conn[3] += ak
            regs = np.maximum(regs, orc.export_hll(m))
            td = orc.export_tdigest(m)
            if td.n:
                acc = po.merge_compress(acc, td.centroids(), delta)
                tmin, tmax, tcount = min(tmin, td.minv), max(tmax, td.maxv), tcount + td.total
                vals += samples.get(m, [])
        slabs.append(acc)
    final = (np.zeros(0), np.zeros(0, dtype=np.uint64))
    for s in slabs:                                         # rank-ascending, empty slabs skipped
        if len(s[0]):
            final = po.merge_compress(final, s, delta)

    def pct(h, total, ps):
        ps = np.array(ps, dtype=np.float32)
        out = np.zeros(len(ps), dtype=np.int64)
        assert L.gysk_hist_percentiles(po.CLS["RESP_TIME"], 0, ge._p(h), total, ge._p(ps), len(ps), ge._p(out)) == 0
        return out.tolist()

    p95, p99, p25 = pct(last, tot_last, [95, 99, 25])
    a95, a99 = pct(allh, tot_all, [95, 99])
    want = dict(found=1, nqrys_5s=tot_last & 0xFFFFFFFF, total_resp_5sec=int(last["sum"].sum()), p95_5s_resp_ms=p95, p99_5s_resp_ms=p99,
                p25_5s_resp_ms=p25, nqrys_all=tot_all, p95_all_resp_ms=a95, p99_all_resp_ms=a99, max_resp_ms=mx,
                nconns_5s=conn[0] & 0xFFFFFFFF, kbytes_5s=conn[1] & 0xFFFFFFFF, nconns_all=conn[2], kbytes_all=conn[3],
                distinct_clients=po.lib().gyo_hll_estimate(po._p(regs), p), td_count=tcount)
    fm, fw = np.ascontiguousarray(final[0]), np.ascontiguousarray(final[1], dtype=np.uint64)
    for q, f in ((0.5, "td_p50_us"), (0.95, "td_p95_us"), (0.99, "td_p99_us")):
        want[f] = L.gysk_tdigest_quantile(ge._p(fm), ge._p(fw), len(fm), tmin, tmax, q) if len(fm) else float("nan")
    return want, len(fm), vals


def _same(a, b):
    return a == b or (isinstance(a, float) and isinstance(b, float) and np.isnan(a) and np.isnan(b))


@pytest.mark.parametrize("world,depth,log2w,p,delta", [(1, 4, 12, 12, 200), (2, 4, 12, 12, 200), (3, 4, 12, 12, 200), (4, 4, 12, 12, 200),
                                                       (2, 2, 8, 5, 64), (3, 2, 8, 5, 64)])
def test_logical_merge_equals_the_cpu_rollup(world, depth, log2w, p, delta):
    import torch
    rng = np.random.default_rng(31 + world + delta)
    kw = dict(max_svcs=512, max_tasks=64, max_batch=1 << 15, cms_depth=depth, cms_log2_width=log2w, hll_p=p, td_compression=delta,
              idle_evict_secs=300)
    pairs_ = [make_pair(rank=r, world=world, **kw) for r in range(world)]
    engs, orcs = [e for e, _ in pairs_], [o for _, o in pairs_]
    ids = synth.service_ids(NSVC)
    tcp_ids = synth.splitmix64(np.arange(1, 4, dtype=np.uint64) + np.uint64(1 << 56))
    pairs = _logical_map(rng, ids, tcp_ids)
    for e in engs:
        e.set_logical_map(np.array([g for g, _ in pairs], dtype=np.uint64), np.array([l for _, l in pairs], dtype=np.uint64))
    lids = np.array(sorted({l for _, l in pairs}), dtype=np.uint64)
    silent = int(ids[129])
    samples = {}
    merged_windows = 0
    for t in (5, 10, 700):
        ev = synth.gen_mixed(rng, 60_000, NSVC, ntask=16, nhosts=NHOSTS, nclients=4000, zipf_s=0.9)
        if t == 700:
            ev = ev[ev["svc_id"] != np.uint64(silent)]
        x = np.zeros(600, dtype=ge.EVENT_DTYPE)             # the TCP-only services, on three hosts
        x["svc_id"] = np.repeat(tcp_ids, 200); x["type"] = ge.EV_ACCEPT; x["host_idx"] = np.repeat([1, 2, 7], 200)
        x["value"] = rng.integers(0, 1 << 20, len(x)); x["flow_key"] = rng.integers(1, 1 << 62, len(x), dtype=np.uint64)
        ev = np.concatenate([ev, x])
        ev = ev[rng.permutation(len(ev))]
        ev["tsec"] = t
        r_ = ev[ev["type"] == ge.EV_RESP]
        for sid, v in zip(r_["svc_id"].tolist(), r_["value"].tolist()):
            samples.setdefault(sid, []).append(v)
        for off in range(0, len(ev), 1 << 15):
            ch = ev[off: off + (1 << 15)]
            for e, o in zip(engs, orcs):
                e.ingest_events(ch); e.sync(); o.ingest(ch)
        for e, o in zip(engs, orcs):
            e.flush(t); o.flush(t)
        if t == 5:
            continue
        if t == 700:
            assert all(o.export_hist(silent, ge.HIST_RESP_LAST) is None for o in orcs)      # evicted before this merge
            samples.pop(silent, None)
        _emulate_collectives(torch, engs)
        got = [e.query_logical(lids) for e in engs]
        for lid, *answers in zip(lids, *got):
            want, nfinal, vals = _expected(pairs, int(lid), orcs, delta, p, samples)
            for k, v in want.items():
                for r, a in enumerate(answers):
                    assert _same(a[k], v), (t, int(lid), r, k, a[k], v)
            assert nfinal <= delta
            if int(lid) == 7013:
                assert want["nconns_all"] > 0 and want["nqrys_all"] == 0 and np.isnan(answers[0]["td_p50_us"])
            if int(lid) == 7011:
                assert want["nqrys_all"] == 0 and want["nconns_all"] == 0
            # against the exact quantiles of the union of the member samples. A merged digest is clustered twice (the members', then
            # the fold's compress), so p99 gets twice the single-digest tolerance, as in test_gpu_merge
            if delta == 200 and len(vals) >= 2000:
                for q, f, k in ((0.5, "td_p50_us", 1), (0.95, "td_p95_us", 1), (0.99, "td_p99_us", 2)):
                    ex = exact_quantile(vals, q)
                    assert abs(answers[0][f] - ex) / ex < k * td_p99_tolerance(len(vals)), (t, int(lid), f, answers[0][f], ex)
        assert [a["found"] for a in got[0]] == [1] * len(lids)
        assert engs[0].query_logical([424242])[0]["found"] == 0
        # global count-min on the all-reduced tables: row minimum over the sum of the ranks' last-window tables
        tbl = sum(o.cms(last_window=True) for o in orcs).reshape(depth, -1)
        keys = np.unique(ev["flow_key"][(ev["type"] >= ge.EV_CONNECT) & (ev["type"] <= ge.EV_CLOSE_SER)])
        keys = keys[rng.choice(len(keys), 300, replace=False)]
        est = engs[-1].query_flows_global(keys, last_window=True)
        for k, e_ in zip(keys, est):
            cells = [int(tbl[r, po.lib().gyo_cms_index(int(k), r, log2w)]) for r in range(depth)]
            assert e_["count"] == min(c & 0xFFFFFFFF for c in cells) and e_["kbytes"] == min(c >> 32 for c in cells)
        merged_windows += 1
    assert merged_windows == 2
