"""Generates tests/golden/hist_golden.npz, jhash_golden.npz, ref_random_golden.npz and summary_pct_golden.npz by RUNNING
THE REFERENCE's own code (oracle/_ref/libgyref.so, compiled from the reference tree by oracle/Makefile). Run only where the
reference tree exists:  python tests/golden/make_golden.py
The fixtures pin oracle/gysk_oracle.c and the engine's percentiles on machines that have no reference tree."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from gyeeta_b200 import engine as ge, synth  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
PCTS = np.array([25, 50, 75, 90, 95, 99, 99.999, 0.001, 100], dtype=np.float32)


def inputs_for(cls_name, rng):
    edge = np.array([-(2 ** 40), -(2 ** 31) - 1, -(2 ** 31), -1000, -16, -15, -3, -2, -1, 0, 1, 2, 5, 8, 9, 10, 13, 14, 26, 27,
                     99, 100, 101, 250, 251, 3000, 3001, 5000, 5001, 15000, 15001, 65000, 65001, 150000, 150001,
                     5000000, 5000001, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 7, 2 ** 40], dtype=np.int64)
    ln = np.round(np.exp(rng.normal(np.log(20), 1.2, 4000))).astype(np.int64)
    uni = rng.integers(-50, 200000, 2000, dtype=np.int64)
    big = rng.integers(0, 2 ** 33, 500, dtype=np.int64)
    return np.concatenate([edge, ln, uni, big])


def main():
    R = po.ref()
    assert R is not None, "reference library not built"
    rng = np.random.default_rng(20260922)
    out = {}
    for name, cls in po.CLS.items():
        tkinds = {"FD_I8_9_26_5": [po.T_INT8], "FD_INT_M15_M3_4": [po.T_INT]}.get(name, [po.T_INT64, po.T_INT])
        for tk in tkinds:
            vals = inputs_for(name, rng)
            if tk == po.T_INT8:
                vals = rng.integers(-128, 128, 3000, dtype=np.int64)
            r = po.hist_run(R, "gyref_hist_run", cls, tk, vals, PCTS)
            key = f"{name}__{tk}"
            out[key + "__vals"] = vals
            out[key + "__buckets"] = r["buckets"].astype(np.int16)
            out[key + "__count"] = r["stats"]["count"]
            out[key + "__sum"] = r["stats"]["sum"]
            out[key + "__total_max"] = np.array([r["total"], r["max"]], dtype=np.int64)
            out[key + "__pct"] = r["pct"]
            out[key + "__avg"] = np.array([r["avg"]], dtype=np.float32)
    # percentile cut-off uses a float multiplier on size_t (gy_statistics.h:753): exercise large counts
    for total_pow in (24, 25, 31, 40):
        stats = np.zeros(16, dtype=po.SERIAL_DTYPE)
        base = (1 << total_pow) // 15
        stats["count"][:15] = base + np.arange(15) * 3 + 1
        stats["sum"][:15] = stats["count"][:15] * 7
        total = int(stats["count"].sum())
        pct = np.zeros(len(PCTS), dtype=np.int64)
        avg = po.C.c_float()
        R.gyref_hist_pct_from_serial(0, 0, po._p(stats), total, 12345, po._p(PCTS), len(PCTS), po._p(pct), po.C.byref(avg))
        out[f"bigcount_{total_pow}__count"] = stats["count"].copy()
        out[f"bigcount_{total_pow}__sum"] = stats["sum"].copy()
        out[f"bigcount_{total_pow}__pct"] = pct
        out[f"bigcount_{total_pow}__avg"] = np.array([avg.value], dtype=np.float32)
    out["pcts"] = PCTS
    np.savez_compressed(os.path.join(HERE, "hist_golden.npz"), **out)

    keys = np.concatenate([np.array([0, 1, 42, 2 ** 32 - 1, 2 ** 32, 2 ** 63, 2 ** 64 - 1], dtype=np.uint64),
                           rng.integers(0, 2 ** 64, 4096, dtype=np.uint64)])
    h64 = np.array([R.gyref_uint64_hash(int(k)) for k in keys], dtype=np.uint32)
    seeds = rng.integers(0, 2 ** 32, len(keys), dtype=np.uint32)
    h2w = np.array([R.gyref_jhash_2words(int(k & np.uint64(0xFFFFFFFF)), int(k >> np.uint64(32)), int(s))
                    for k, s in zip(keys, seeds)], dtype=np.uint32)
    blob = rng.integers(0, 256, 64, dtype=np.uint8)
    hbytes = np.array([R.gyref_jhash(po._p(blob), n, 0xceedfead) for n in range(0, 41)], dtype=np.uint32)
    words = rng.integers(0, 2 ** 32, 16, dtype=np.uint32)
    hwords = np.array([R.gyref_jhash2(po._p(words), n, 0xceedfead) for n in range(0, 13)], dtype=np.uint32)
    np.savez_compressed(os.path.join(HERE, "jhash_golden.npz"), keys=keys, h64=h64, seeds=seeds, h2w=h2w, blob=blob,
                        hbytes=hbytes, words=words, hwords=hwords)
    print("golden fixtures written:", len(out), "hist arrays")
    random_streams(R)
    summary_percentiles(R)


def random_streams(R):
    """ref_random_golden.npz: the reference's histograms over the random streams of
    test_oracle_pinning.py::test_oracle_vs_compiled_reference_random. The test draws the same streams from seed 7; the inputs
    themselves (2.5 MB) are not stored, only their SHA-256, so a generator that draws differently fails the test."""
    rng = np.random.default_rng(7)
    pcts = [25, 50, 95, 99, 99.9]
    g = {k: [] for k in ("case", "vals_sha256", "nb", "total", "max", "buckets", "count", "sum", "pct", "avg")}
    for name, cls in po.CLS.items():
        if name.startswith("FD_"):
            continue
        for tk in (po.T_INT64, po.T_INT):
            for scale in (50, 5000, 2 ** 20, 2 ** 34):
                vals = rng.integers(-scale // 10, scale, 5000, dtype=np.int64)
                b = po.hist_run(R, "gyref_hist_run", cls, tk, vals, pcts)
                stats = np.zeros(16, dtype=po.SERIAL_DTYPE)
                stats[: b["nb"]] = b["stats"]
                g["case"].append([cls, tk, scale])
                g["vals_sha256"].append(np.frombuffer(hashlib.sha256(vals.tobytes()).digest(), dtype=np.uint8))
                for k in ("nb", "total", "max", "buckets", "pct", "avg"):
                    g[k].append(b[k])
                g["count"].append(stats["count"]); g["sum"].append(stats["sum"])
    keys = rng.integers(0, 2 ** 64, 2000, dtype=np.uint64)
    dt = dict(case=np.int64, vals_sha256=np.uint8, nb=np.int64, total=np.uint64, max=np.int64, buckets=np.int8, count=np.uint64,
              sum=np.int64, pct=np.int64, avg=np.float32)
    out = {k: np.array(v, dtype=dt[k]) for k, v in g.items()}
    np.savez_compressed(os.path.join(HERE, "ref_random_golden.npz"), pcts=np.array(pcts, dtype=np.float32), keys=keys,
                        h64=np.array([R.gyref_uint64_hash(int(k)) for k in keys], dtype=np.uint32),
                        sizeof_hist_resp=np.array([R.gyref_sizeof_hist_resp()], dtype=np.int64), **out)


def summary_percentiles(R):
    """summary_pct_golden.npz: the reference's get_percentiles (p95, p99, p25) over the last-window response histograms that
    test_gpu_parity.py::test_flush_window_roll_and_summary queries, with the serial form they were computed from. The CPU oracle
    replays the test's seeded stream (it equals the engine bit for bit there)."""
    rng = np.random.default_rng(5)
    orc = po.OracleEngine(max_svcs=512, max_tasks=64, cms_log2_width=14)
    ids = None
    for w in range(3):
        ev = synth.gen_mixed(rng, 40_000, 100, ntask=16, nhosts=8, nclients=5000)
        ids = np.unique(ev["svc_id"][ev["type"] != ge.EV_TASK]) if ids is None else ids
        for off in range(0, len(ev), 1 << 15):
            orc.ingest(ev[off: off + (1 << 15)])
        orc.flush(5 * (w + 1))
    pcts = np.array([95, 99, 25], dtype=np.float32)
    rows = {k: [] for k in ("ids", "count", "sum", "total", "max", "pct")}
    for id_ in ids[:40]:
        last, total, mx = orc.export_hist(int(id_), ge.HIST_RESP_LAST)
        ser = np.zeros(16, dtype=po.SERIAL_DTYPE); ser[:15] = last
        out = np.zeros(3, dtype=np.int64)
        R.gyref_hist_pct_from_serial(0, 0, po._p(ser), total, mx, po._p(pcts), 3, po._p(out), None)
        for k, v in zip(rows, (id_, last["count"], last["sum"], total, mx, out)):
            rows[k].append(v)
    dt = dict(ids=np.uint64, count=np.uint64, sum=np.int64, total=np.uint64, max=np.int64, pct=np.int64)
    np.savez_compressed(os.path.join(HERE, "summary_pct_golden.npz"), pcts=pcts, **{k: np.array(v, dtype=dt[k]) for k, v in rows.items()})


if __name__ == "__main__":
    main()
