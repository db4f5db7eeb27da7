"""Pins the CPU oracle (oracle/gysk_oracle.c) before anything trusts it:
  1. the reference's own asserted fixture, test/test_histogram.cc:29-147 (bucket ids + 4 percentiles);
  2. golden vectors produced by RUNNING the reference here (tests/golden/*.npz, made by make_golden.py);
  3. outputs of the compiled reference (oracle/_ref/libgyref.so) on random streams, recorded in tests/golden/ref_random_golden.npz.
"""
import hashlib
import os

import numpy as np

from oracle import pyoracle as po

L = po.lib()


def run(cls, tk, vals, pcts=()):
    return po.hist_run(L, "gyo_hist_run", cls, tk, vals, pcts)


# ---- 1. test/test_histogram.cc ----------------------------------------------------------------------
def test_reference_fixture_fixed_diff_int8():
    # test/test_histogram.cc:17-86   Hist_9_26 = GY_HISTOGRAM<int8_t, FIXED_DIFF_HASH<int8_t, 9, 26, 5>>
    cls, tk = po.CLS["FD_I8_9_26_5"], po.T_INT8
    assert L.gyo_nbuckets(cls) == 6                                            # :29
    seq = [(0, 0), (8, 0), (9, 1), (10, 1), (13, 1), (14, 2), (15, 2), (18, 2), (19, 3), (20, 3), (23, 3), (24, 4)]
    vals = [v for v, _ in seq]
    r = run(cls, tk, vals, [75.0])
    assert r["buckets"].tolist() == [b for _, b in seq]                        # :31-65
    assert r["pct"][0] == 23                                                   # :67-68
    seq2 = seq + [(25, 4), (26, 4), (27, 5), (40, 5)]
    r = run(cls, tk, [v for v, _ in seq2], [90.0])
    assert r["buckets"].tolist() == [b for _, b in seq2]                       # :70-80
    assert r["pct"][0] == 26                                                   # :82-83


def test_reference_fixture_fixed_diff_negative():
    # test/test_histogram.cc:92-147  Hist_n4 = GY_HISTOGRAM<int, FIXED_DIFF_HASH<int, -15, -3, 4>>
    cls, tk = po.CLS["FD_INT_M15_M3_4"], po.T_INT
    assert L.gyo_nbuckets(cls) == 6                                            # :99
    seq = [(0, 5), (-16, 0), (-15, 1), (-13, 1), (-12, 1), (-11, 2), (-10, 2), (-8, 2)]
    r = run(cls, tk, [v for v, _ in seq], [75.0])
    assert r["buckets"].tolist() == [b for _, b in seq]                        # :104-123
    assert r["pct"][0] == -8                                                   # :125-126
    seq2 = seq + [(-7, 3), (-5, 3), (-4, 3), (-3, 4), (-2, 5)]
    r = run(cls, tk, [v for v, _ in seq2], [75.0])
    assert r["buckets"].tolist() == [b for _, b in seq2]                       # :128-141
    assert r["pct"][0] == -4                                                   # :143-144


def test_survey_probe_values():
    # SURVEY.md §8c probe of the compiled reference: 0..999 into RESP_TIME_HASH
    r = run(po.CLS["RESP_TIME"], po.T_INT64, np.arange(1000), [50, 95, 99])
    assert r["pct"].tolist() == [700, 1000, 1000] and r["total"] == 1000 and r["max"] == 999
    assert L.gyo_uint64_hash(42) == 4033382092


# ---- 2. golden vectors from the reference --------------------------------------------------------------
def test_hist_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "hist_golden.npz"))
    pcts = g["pcts"]
    nchecked = 0
    for name, cls in po.CLS.items():
        for tk in (po.T_INT64, po.T_INT, po.T_INT8):
            key = f"{name}__{tk}"
            if key + "__vals" not in g:
                continue
            r = run(cls, tk, g[key + "__vals"], pcts)
            assert np.array_equal(r["buckets"], g[key + "__buckets"]), key
            assert np.array_equal(r["stats"]["count"], g[key + "__count"]), key
            assert np.array_equal(r["stats"]["sum"], g[key + "__sum"]), key
            assert [r["total"], r["max"]] == g[key + "__total_max"].tolist(), key
            assert np.array_equal(r["pct"], g[key + "__pct"]), key
            assert np.float32(r["avg"]) == g[key + "__avg"][0], key
            nchecked += 1
    assert nchecked == 18


def test_percentile_float_cutoff_golden(golden_dir):
    # size_t * float cut-off (gy_statistics.h:753-754) at counts beyond 2^24
    import ctypes as C
    g = np.load(os.path.join(golden_dir, "hist_golden.npz"))
    pcts = g["pcts"]
    for p in (24, 25, 31, 40):
        h = np.zeros(1, dtype=np.dtype([("stats", po.SERIAL_DTYPE, 16), ("total", "<u8"), ("max", "<i8"),
                                        ("cls", "<i4"), ("tk", "<i4")]))
        h["stats"][0]["count"][:] = g[f"bigcount_{p}__count"]
        h["stats"][0]["sum"][:] = g[f"bigcount_{p}__sum"]
        h["total"] = int(g[f"bigcount_{p}__count"].astype(np.uint64).sum())
        h["max"] = 12345
        out = np.zeros(len(pcts), dtype=np.int64)
        avg = C.c_float()
        L.gyo_hist_percentiles(po._p(h), po._p(pcts), C.c_size_t(len(pcts)), po._p(out), C.byref(avg))
        assert np.array_equal(out, g[f"bigcount_{p}__pct"]), p
        assert np.float32(avg.value) == g[f"bigcount_{p}__avg"][0]


def test_jhash_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "jhash_golden.npz"))
    keys, seeds = g["keys"], g["seeds"]
    h64 = np.array([L.gyo_uint64_hash(int(k)) for k in keys], dtype=np.uint32)
    assert np.array_equal(h64, g["h64"])
    h2w = np.array([L.gyo_jhash_2words(int(k) & 0xFFFFFFFF, int(k) >> 32, int(s)) for k, s in zip(keys, seeds)],
                   dtype=np.uint32)
    assert np.array_equal(h2w, g["h2w"])
    blob = g["blob"].copy()
    assert [L.gyo_jhash(po._p(blob), n, 0xceedfead) for n in range(41)] == g["hbytes"].tolist()
    words = g["words"].copy()
    assert [L.gyo_jhash2(po._p(words), n, 0xceedfead) for n in range(13)] == g["hwords"].tolist()


# ---- 3. against the compiled reference on random streams ----------------------------------------------------
def test_oracle_vs_compiled_reference_random(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_random_golden.npz"))
    assert g["sizeof_hist_resp"][0] == 280
    rng = np.random.default_rng(7)
    pcts = g["pcts"].tolist()
    i = 0
    for name, cls in po.CLS.items():
        if name.startswith("FD_"):
            continue
        for tk in (po.T_INT64, po.T_INT):
            for scale in (50, 5000, 2 ** 20, 2 ** 34):
                vals = rng.integers(-scale // 10, scale, 5000, dtype=np.int64)
                assert g["case"][i].tolist() == [cls, tk, scale]
                assert hashlib.sha256(vals.tobytes()).digest() == g["vals_sha256"][i].tobytes(), "not the stream the reference saw"
                a = run(cls, tk, vals, pcts)
                nb = int(g["nb"][i])
                for k in ("nb", "total", "max"):
                    assert a[k] == g[k][i], (name, tk, scale, k)
                assert np.array_equal(a["buckets"], g["buckets"][i]), (name, tk, scale)
                assert np.array_equal(a["stats"]["count"], g["count"][i][:nb]), (name, tk, scale)
                assert np.array_equal(a["stats"]["sum"], g["sum"][i][:nb]), (name, tk, scale)
                assert np.array_equal(a["pct"], g["pct"][i]), (name, tk, scale)
                assert np.float32(a["avg"]) == g["avg"][i]
                i += 1
    assert i == len(g["case"]) == 64
    keys = rng.integers(0, 2 ** 64, 2000, dtype=np.uint64)
    assert np.array_equal(keys, g["keys"])
    assert [L.gyo_uint64_hash(int(k)) for k in keys] == g["h64"].tolist()
