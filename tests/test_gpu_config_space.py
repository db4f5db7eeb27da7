"""The engine away from its default configuration. gysk_create accepts count-min depth 1-8 and width 2^4-2^28, HyperLogLog
precision p = 4-16 and t-digest compression delta = 10-256; the kernels read all four at run time (row loops, register rows of 2^p
bytes, the per-lane split of the K_1 cells, the merge arena). Part A runs a mixed stream at points that together reach every end
of those ranges and compares everything with the CPU oracle bit for bit.

Part B runs every pass plan of the RESP key sort (key_sort_plan: TD_CODE_BITS + slot bits cut into 2-5 digits) with the test
services in the HIGHEST slots of the table, so the upper digits of their keys are not zero, and the batch geometries around the
sort's tile sizes."""
import numpy as np
import pytest

from gyeeta_b200 import engine as ge
from gyeeta_b200 import synth
from oracle import pyoracle as po
from tests.util import assert_hist_equal, feed_both, make_pair

pytestmark = pytest.mark.gpu

# (cms_depth, cms_log2_width, hll_p, td_compression): depth 1 and 8, width 2^4 (16 cells: collisions everywhere) and 2^20, p 4 / 5 / 6
# (the register counts with their own alpha) and 16, delta 10 and 256 (= TD_CAP) and the uneven per-lane cell splits of 37 and 255
CONFIGS = [(1, 4, 4, 10), (2, 6, 5, 37), (3, 11, 6, 100), (8, 16, 7, 255), (5, 20, 16, 256), (4, 20, 12, 200)]
HOT = {"hot_off": ("GYSK_HOT_ROWS", "0"), "hot_min8": ("GYSK_HOT_MIN", "8")}


def _hot(monkeypatch, mode):
    monkeypatch.setenv(*HOT[mode])                 # read by gysk_create: set before the engine exists


def _with_active(rng, ev, frac=0.05):
    """turn a share of the TCP events into ACTIVE_CONN_STATS records: value = kbytes, flags = active conns, tsec = float bits of rtt"""
    tcp = np.flatnonzero((ev["type"] >= ge.EV_CONNECT) & (ev["type"] <= ge.EV_CLOSE_SER))
    pick = tcp[rng.random(len(tcp)) < frac]
    ev["type"][pick] = ge.EV_ACTIVE
    ev["value"][pick] = rng.integers(0, 5000, len(pick))
    ev["flags"][pick] = rng.integers(1, 60, len(pick))
    ev["tsec"][pick] = rng.uniform(0.1, 900.0, len(pick)).astype(np.float32).view(np.uint32)
    return ev


def _assert_td_equal(eng, orc, id_):
    got, td = eng.export_tdigest(int(id_)), orc.export_tdigest(int(id_))
    assert (got is None) == (td is None), hex(int(id_))
    if got is None:
        return None
    om, ow = td.centroids()
    assert np.array_equal(got[0], om) and np.array_equal(got[1], ow), hex(int(id_))
    assert got[2] == td.minv and got[3] == td.maxv, hex(int(id_))
    return got


def _qtab(delta):
    """the K_1 grid q_j = (sin(pi (j / delta - 1/2)) + 1) / 2, j = 0 .. delta (the cell starts of the compress step)"""
    j = np.arange(delta + 1, dtype=np.float64)
    q = 0.5 * (np.sin(np.pi * (j / delta - 0.5)) + 1.0)
    q[0], q[-1] = 0.0, 1.0
    return q


def rank_error_bound(q, delta, max_item_frac):
    """Bound on |F(quantile(q)) - q|, F the exact empirical CDF of the samples the digest holds.

    1. Every cluster is the set of merged items whose start falls into one cell [q_j, q_j+1) of the K_1 grid, so its rank span is
       at most the cell width c_j = q_j+1 - q_j plus the weight of its last item, max_item_frac at most. Near q the cells have width
       c(q) ~ pi sqrt(q (1 - q)) / delta; we take the widest of the five cells around q, since the clusters used lie next to it.
    2. quantile(q) interpolates between the centres of the two clusters i, i+1 whose centres bracket rank qW, so the answer lies
       between their means. A mean lies within the value range of its own samples, so if the clusters held value-disjoint samples,
       F(answer) would lie in the rank span of i or i+1 and |F - q| <= span_i + span_i+1 <= 2 (c(q) + max_item_frac).
    3. The clusters of a digest fed in batches are not value-disjoint: a cluster made in an earlier batch is merged with the next
       batch's items by its mean alone, so samples of neighbouring clusters interleave in value. An old cluster ends up next to
       items that were placed on either side of it, which shifts F at its mean by at most the span of one neighbouring cluster on
       each side: two more cell widths.
    Hence |F(quantile(q)) - q| <= 4 c(q) + 2 max_item_frac. (On these streams the oracle's digests, which the kernels' equal bit
    for bit, stay within 0.12 of this bound at every delta of CONFIGS; it is a bound, not an estimate.)"""
    qt = _qtab(delta)
    j = int(np.clip(np.searchsorted(qt, q, side="right") - 1, 0, delta - 1))
    widths = np.diff(qt)[max(0, j - 2): j + 3]
    return 4.0 * float(widths.max()) + 2.0 * max_item_frac


def rank_error(sorted_vals, x, q):
    """distance of q from [F(x-), F(x)]: zero when x is a q-quantile of the sample (ties make F a step)"""
    n = len(sorted_vals)
    lo = np.searchsorted(sorted_vals, x, side="left") / n
    hi = np.searchsorted(sorted_vals, x, side="right") / n
    return max(0.0, lo - q, q - hi)


def _max_item_frac(vals, batches):
    """largest share of a service's samples that one batch put into one t-digest value bin (one item of the merge)"""
    L = po.lib()
    bins = np.array([L.gyo_td_code(int(v)) + L.gyo_bucket(po.CLS["RESP_TIME"], int(v) // 1000) for v in vals], dtype=np.int64)
    best = 0
    for b in np.unique(batches):
        _, cnt = np.unique(bins[batches == b], return_counts=True)
        best = max(best, int(cnt.max()))
    return best / len(vals)


def _flows_min(orc_tbl, keys, depth, log2w):
    tbl = orc_tbl.reshape(depth, -1)
    cnt, kb = [], []
    for k in keys:
        cells = [int(tbl[r, po.lib().gyo_cms_index(int(k), r, log2w)]) for r in range(depth)]
        cnt.append(min(c & 0xFFFFFFFF for c in cells)); kb.append(min(c >> 32 for c in cells))
    return np.array(cnt), np.array(kb)


# ---------------------------------------------------------------------------------------------------------------------------------
# A. sketch parameters
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hot", list(HOT))
@pytest.mark.parametrize("depth,log2w,p,delta", CONFIGS)
def test_sketch_parameters_bit_exact(monkeypatch, hot, depth, log2w, p, delta):
    _hot(monkeypatch, hot)
    rng = np.random.default_rng(1000 * depth + log2w + 17 * p + delta)
    nsvc, batch = 300, 1 << 14
    eng, orc = make_pair(max_svcs=512, max_tasks=64, max_batch=batch, cms_depth=depth, cms_log2_width=log2w, hll_p=p,
                         td_compression=delta, idle_evict_secs=300)
    samples = {}                                          # svc -> [(value, batch index)] of every RESP sample
    nb = 0
    for w, t in enumerate((5, 10)):
        ev = _with_active(rng, synth.gen_mixed(rng, 90_000, nsvc, ntask=16, nhosts=64, nclients=5000, zipf_s=1.1))
        assert (ev["type"] == ge.EV_ACTIVE).sum() > 100
        for off in range(0, len(ev), batch):
            ch = ev[off: off + batch]
            feed_both(eng, orc, ch, batch)
            r = ch[ch["type"] == ge.EV_RESP]
            for sid, v in zip(r["svc_id"].tolist(), r["value"].tolist()):
                samples.setdefault(sid, []).append((v, nb))
            nb += 1
        # the whole count-min table, both halves, before and after the roll
        assert np.array_equal(eng.export_cms(), orc.cms())
        eng.flush(t); orc.flush(t)
        assert np.array_equal(eng.export_cms(last_window=True), orc.cms(last_window=True))
        assert np.array_equal(eng.export_cms(), orc.cms())
        keys = np.unique(ev["flow_key"][(ev["type"] >= ge.EV_CONNECT) & (ev["type"] <= ge.EV_CLOSE_SER) | (ev["type"] == ge.EV_ACTIVE)])
        keys = keys[rng.choice(len(keys), 300, replace=False)]
        est = eng.query_flows(keys, last_window=True)
        cnt, kb = _flows_min(orc.cms(last_window=True), keys, depth, log2w)   # min over ALL cms_depth rows
        assert np.array_equal(est["count"], cnt) and np.array_equal(est["kbytes"], kb)
        assert cnt.min() > 0

    s, o = eng.stats(), orc.counters()
    assert (s["events_resp"], s["events_tcp"], s["events_task"], s["events_dropped"]) == (o["resp"], o["tcp"], o["task"], o["dropped"])
    ids = np.array(sorted(samples, key=lambda k: -len(samples[k])), dtype=np.uint64)
    pick = np.concatenate([ids[:20], ids[-20:], rng.choice(ids, 20, replace=False)])
    summ = eng.query_svcs(pick)
    for id_, sm in zip(pick, summ):
        id_ = int(id_)
        for which in (ge.HIST_RESP_CUR, ge.HIST_RESP_LAST, ge.HIST_RESP_ALL):
            assert_hist_equal(eng, orc, id_, which)
        regs = orc.export_hll(id_)
        assert len(regs) == 1 << p and np.array_equal(eng.export_hll(id_), regs), hex(id_)
        assert sm["distinct_clients"] == po.lib().gyo_hll_estimate(po._p(regs), p), hex(id_)
        means, weights, mn, mx = _assert_td_equal(eng, orc, id_)
        assert len(means) <= delta and int(weights.sum()) == len(samples[id_])
    # rank error of the digest's quantiles against the exact empirical CDF, for the services with enough samples
    nchecked = 0
    for id_ in ids[:30]:
        vb = np.array(samples[int(id_)], dtype=np.int64)
        if len(vb) < 2000:
            continue
        vals = np.sort(vb[:, 0])
        frac = _max_item_frac(vb[:, 0], vb[:, 1])
        qs = eng.quantiles(int(id_), [0.5, 0.95, 0.99])
        for q, x in zip((0.5, 0.95, 0.99), qs):
            err, bound = rank_error(vals, x, q), rank_error_bound(q, delta, frac)
            assert err <= bound, (hex(int(id_)), q, err, bound)
        nchecked += 1
    assert nchecked >= 3

    # eviction at every p: half of the services go silent, are evicted, and new ids take their slots with cleared registers
    keep = set(int(i) for i in ids[::2])
    for t in (700, 705):
        ev = synth.gen_mixed(rng, 20_000, nsvc, ntask=16, nhosts=64, nclients=5000, zipf_s=1.1)
        ev = ev[(ev["type"] == ge.EV_TASK) | np.isin(ev["svc_id"], np.fromiter(keep, dtype=np.uint64))]
        if t == 705:
            new = synth.splitmix64(np.arange(1, 201, dtype=np.uint64) + np.uint64(1 << 50))
            x = np.zeros(4000, dtype=ge.EVENT_DTYPE)
            x["svc_id"] = np.repeat(new, 20)
            x["type"] = np.where(np.arange(len(x)) % 2, ge.EV_RESP, ge.EV_ACCEPT)
            x["value"] = rng.integers(100, 900_000, len(x))
            x["flow_key"] = rng.integers(1, 1 << 62, len(x), dtype=np.uint64)
            ev = np.concatenate([ev, x])
        ev["tsec"] = t
        feed_both(eng, orc, ev, batch)
        eng.flush(t); orc.flush(t)
        got, (want, _) = np.sort(eng.evicted_ids()), orc.evicted_ids()
        assert np.array_equal(got, np.sort(want))
        if t == 700:
            assert len(got) >= len(ids) - len(keep) and not keep & set(got.tolist())
    assert eng.stats()["nsvcs"] == orc.nsvcs()
    summ = eng.query_svcs(new)
    for id_, sm in zip(new, summ):
        regs = orc.export_hll(int(id_))
        assert np.array_equal(eng.export_hll(int(id_)), regs), hex(int(id_))
        assert sm["distinct_clients"] == po.lib().gyo_hll_estimate(po._p(regs), p)
        assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_ALL)
        _assert_td_equal(eng, orc, id_)


# ---------------------------------------------------------------------------------------------------------------------------------
# B. every pass plan of the key sort, with the test services in the highest slots
# ---------------------------------------------------------------------------------------------------------------------------------
TD_CODE_BITS = 10


def sort_plan(max_svcs):
    """key_sort_plan's digits: TD_CODE_BITS + slot bits in the fewest digits of <= 8 bits, widths as even as possible"""
    sb = 1
    while sb < 24 and (1 << sb) < max_svcs:
        sb += 1
    T = TD_CODE_BITS + sb
    npass = -(-T // 8)
    return sb, [T // npass + (i < T % npass) for i in range(npass)]


# slot bits 1, 2, 5, 13, 15, 16 and 18 are the plans the rest of the suite never runs; 1 is also max_svcs = 1
PLAN_CASES = [1, 2, 4, 32, 1 << 13, 1 << 15, 1 << 16, 1 << 18]
BIG_CASES = [1 << 22, (1 << 22) + 64]       # 8 8 8 8 and the only 5-pass plan (7 7 7 7 6): tens of GB of device memory
BIG_KW = dict(max_tasks=16, hll_p=4, cms_log2_width=10, max_batch=1 << 14)     # small registers and batch: the footprint is the slots'
_slot_bytes = []


def _bytes_per_slot(torch):
    """device memory per service slot of an engine configured as BIG_KW: measured once on an engine of 2^18 slots"""
    if not _slot_bytes:
        torch.cuda.init()
        free0, _ = torch.cuda.mem_get_info()
        e = ge.Engine(max_svcs=1 << 18, **BIG_KW)
        free1, _ = torch.cuda.mem_get_info()
        e.close()
        _slot_bytes.append(max(free0 - free1, 1) / float(1 << 18))
        print(f"device memory per service slot ({BIG_KW}): {_slot_bytes[0]:.0f} bytes")
    return _slot_bytes[0]


def _feed_sizes(eng, orc, ev, sizes):
    off = 0
    for n in sizes:
        ch = ev[off: off + n]
        off += n
        eng.ingest_events(ch); eng.sync()
        orc.ingest(ch)
    assert off == len(ev)


def _resp_stream(rng, ids, n):
    ev = np.zeros(n, dtype=ge.EVENT_DTYPE)
    ev["svc_id"] = ids[rng.integers(0, len(ids), n)]
    ev["type"] = ge.EV_RESP
    ev["value"] = np.minimum(np.exp(rng.normal(np.log(3000.0), 2.5, n)), 9.9e8).astype(np.uint32)
    ev["flow_key"] = rng.integers(1, 1 << 62, n, dtype=np.uint64)
    return ev


def _check_services(eng, orc, ids):
    for id_ in ids:
        assert_hist_equal(eng, orc, int(id_), ge.HIST_RESP_CUR)
        _assert_td_equal(eng, orc, id_)


def _run_high_slots(max_svcs, k=24):
    rng = np.random.default_rng(max_svcs)
    k = min(k, max_svcs)
    eng = ge.Engine(max_svcs=max_svcs, **BIG_KW)
    orc = po.OracleEngine(max_svcs=64, max_tasks=16, hll_p=4, cms_log2_width=10)
    fill = synth.splitmix64(np.arange(1, max_svcs - k + 1, dtype=np.uint64) + np.uint64(1 << 52))
    if len(fill):
        eng.register_ids(fill)                          # one call: the fillers take slots 0 .. max_svcs - k - 1 in order
    ids = synth.service_ids(k)
    eng.register_ids(ids); orc.register_ids(ids)        # the test services: slots max_svcs - k .. max_svcs - 1
    assert eng.stats()["nsvcs"] == max_svcs
    for b in range(4):
        ev = _resp_stream(rng, ids, 12_000)
        ev["value"][:k] = 1_000_000_999                 # the largest valid value: every code bit in play
        ev["svc_id"][:k] = ids
        feed_both(eng, orc, ev, 1 << 14)
        _check_services(eng, orc, ids)
        if b == 1:
            eng.flush(5); orc.flush(5)
    s, o = eng.stats(), orc.counters()
    assert s["events_resp"] == o["resp"] and s["events_dropped"] == o["dropped"] == 0
    eng.close()


@pytest.mark.parametrize("hot", list(HOT))
@pytest.mark.parametrize("max_svcs", PLAN_CASES)
def test_key_sort_plan_with_services_in_the_top_slots(monkeypatch, hot, max_svcs):
    _hot(monkeypatch, hot)
    _run_high_slots(max_svcs)


@pytest.mark.parametrize("hot", list(HOT))
@pytest.mark.parametrize("max_svcs", BIG_CASES)
def test_key_sort_plan_big_tables(monkeypatch, hot, max_svcs):
    import torch
    _hot(monkeypatch, hot)
    need = _bytes_per_slot(torch) * max_svcs
    free, _ = torch.cuda.mem_get_info()
    if free < 2 * need:
        pytest.skip(f"max_svcs {max_svcs} needs ~{need / 2**30:.1f} GiB of device memory; {free / 2**30:.1f} GiB free, twice that required")
    _run_high_slots(max_svcs)


def test_sort_plans_cover_every_shape():
    """the cases above are the slot widths the rest of the suite leaves out, and together reach every digit count"""
    assert [sort_plan(m)[0] for m in PLAN_CASES + BIG_CASES] == [1, 1, 2, 5, 13, 15, 16, 18, 22, 23]
    assert {len(sort_plan(m)[1]) for m in PLAN_CASES + BIG_CASES} == {2, 3, 4, 5}
    assert sort_plan(1)[1] == [6, 5] and sort_plan(1 << 13)[1] == [8, 8, 7] and sort_plan(1 << 16)[1] == [7, 7, 6, 6]
    assert sort_plan(1 << 22)[1] == [8, 8, 8, 8] and sort_plan((1 << 22) + 64)[1] == [7, 7, 7, 6, 6]


# ---------------------------------------------------------------------------------------------------------------------------------
# batch geometry around the sort's tiles (SORT_TILE = 4096 keys, the run-mark tile = 2048 keys, 128-key chunks)
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hot", list(HOT))
def test_batch_sizes_around_the_warp_and_block(monkeypatch, hot):
    _hot(monkeypatch, hot)
    rng = np.random.default_rng(3)
    eng, orc = make_pair(max_svcs=256, max_tasks=16, max_batch=1024, cms_log2_width=10)
    sizes = [1, 31, 33, 63, 65, 1023, 1024, 1, 1024]
    ev = synth.gen_mixed(rng, sum(sizes), 40, ntask=4, nhosts=8, nclients=500)
    _feed_sizes(eng, orc, ev, sizes)
    assert np.array_equal(eng.export_cms(), orc.cms())
    _check_services(eng, orc, np.unique(ev["svc_id"][ev["type"] != ge.EV_TASK]))


@pytest.mark.parametrize("hot", list(HOT))
@pytest.mark.parametrize("nkeys", [2047, 2048, 2049, 4095, 4096, 4097])
def test_resp_key_counts_around_the_tiles(monkeypatch, hot, nkeys):
    _hot(monkeypatch, hot)
    rng = np.random.default_rng(nkeys)
    eng, orc = make_pair(max_svcs=1024, max_tasks=16, max_batch=1 << 13, cms_log2_width=10)
    ids = synth.service_ids(300)
    for _ in range(3):
        feed_both(eng, orc, _resp_stream(rng, ids, nkeys), 1 << 13)
        assert eng.last_batch_keys() == nkeys if hot == "hot_off" else eng.last_batch_keys() <= nkeys
    _check_services(eng, orc, ids)


@pytest.mark.parametrize("hot", list(HOT))
def test_one_value_run_across_tiles(monkeypatch, hot):
    """one service whose batch is a single value: one run of keys spans several sort tiles and 128-key chunks"""
    _hot(monkeypatch, hot)
    rng = np.random.default_rng(8)
    eng, orc = make_pair(max_svcs=64, max_tasks=16, max_batch=1 << 14, cms_log2_width=10)
    ids = synth.service_ids(3)
    for v in (777_777, 5, 777_777):
        ev = _resp_stream(rng, ids[:1], 10_000)
        ev["value"] = v
        other = _resp_stream(rng, ids[1:], 300)
        feed_both(eng, orc, np.concatenate([other[:150], ev, other[150:]]), 1 << 14)
        _check_services(eng, orc, ids)


@pytest.mark.parametrize("hot", list(HOT))
def test_every_key_in_its_own_bin(monkeypatch, hot):
    """every sample of a batch is the only one of its (service, value bin): as many runs as keys"""
    _hot(monkeypatch, hot)
    rng = np.random.default_rng(9)
    eng, orc = make_pair(max_svcs=1024, max_tasks=16, max_batch=1 << 13, cms_log2_width=10)
    ids = synth.service_ids(1000)
    for b in range(3):
        ev = np.zeros(8000, dtype=ge.EVENT_DTYPE)
        ev["svc_id"] = np.repeat(ids, 8)
        ev["type"] = ge.EV_RESP
        ev["value"] = np.tile(np.array([3, 40, 900, 17_000, 260_000, 3_100_000, 47_000_000, 700_000_000], dtype=np.uint32), 1000) + b
        ev = ev[rng.permutation(len(ev))]
        codes = [(int(s), po.lib().gyo_td_code(int(v))) for s, v in zip(ev["svc_id"], ev["value"])]
        assert len(set(codes)) == len(ev)
        feed_both(eng, orc, ev, 1 << 13)
        assert eng.last_batch_keys() <= len(ev)
    _check_services(eng, orc, ids[::7])
