#!/usr/bin/env python
"""bench.py — events/sec aggregated by the B200 streaming-sketch engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # product arm
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on this box's host cores
    python bench.py ... --dump-outputs DIR                   # also write what the timed steps computed (dump_outputs)

One STEP = one pass of the hot path over one batch of synthetic events: ingest_kernel (count-min / HLL / process histograms; a
response sample of a hot service updates its dense row of value bins, any other becomes a sort key), 4 one-sweep radix passes,
runs_mark / runs_sum (per-(service, bin) counts and sums of the keys), bins_merge (histogram cells + t-digest merge from rows and runs). N > 1 adds ONE sketch merge (gysk_merge_global: fold + one NCCL group + merge-compress) per timed
window, as a deployment merges once per query window. Workload = BASELINE.json configs[2] ("100 M mixed TCP/syscall events,
100 K services, t-digest p50/p95/p99 on 1xB200"), the largest single-GPU configuration: per rank EVENTS_PER_STEP
events of the 70/20/10 RESP/TCP/TASK mix over 100 K services (weak scaling: each rank ingests its own host shard).

`value`  : whole-job events/s with the batch already resident in HBM (device timed, CUDA events, max over ranks).
`e2e`    : same metric through the C-ABI call a user makes with HOST (page-locked) buffers: H2D inside the timed region,
           plus a device->host read of per-service summaries. Records = the packed per-kind structs of include/gysketch.h
           (18.4 B/event); `e2e_event32` = 32-byte canonical records; `e2e_wire` = 16 host threads calling gysk_ingest_msg /
           gysk_ingest_raw with TCP_CONN_NOTIFY / AGGR_TASK_STATE_NOTIFY messages and raw tcp_ipv4_resp_event_t arrays.
`roofline`: dominant kernel, algorithmic bytes (SURVEY.md §8d; 54.8 B/event + 32 B per event that took the hot-row way, `hot_rows`)
           / CUDA-event time, against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle port (all host cores, events pre-sharded by host) on a bounded sample of the same stream.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NSVC = 100_000
NTASK = 25_000
NHOSTS = 4096
NCLIENTS = 1_000_000
ZIPF_S = 1.05
# algorithmic bytes per event, SURVEY.md §8(d): RESP 98 = 32 + 32 + 16 + 18(t-digest), TCP 98, TASK 128.
# split per kernel group: the ingest kernel reads every record (32 B) and carries the TCP (count-min + HLL) and TASK state; the
# RESP histogram cell (32 B), per-service counter (16 B) and t-digest share (18 B) are produced from the sorted keys by the
# sort + runs + bins-merge chain (DESIGN.md §4).
# With the side-drain experiment (GYSK_SIDE_DRAIN=1, not the default) ingest_kernel only reads the records (32 B each) and queues keys /
# records; the connection state (64 + 2 B per TCP event) and the process histograms (96 B per TASK sample) are applied by
# side_drain_kernel, so their bytes count with the chain group.
SIDE_DRAIN = os.environ.get("GYSK_SIDE_DRAIN", "0") != "0"
BYTES_INGEST = 32.0 if SIDE_DRAIN else 0.7 * 32 + 0.2 * 98 + 0.1 * 128                      # 32.0 (54.8) B / event
BYTES_TDIGEST = 0.7 * (32 + 16 + 18) + (0.2 * 66 + 0.1 * 96 if SIDE_DRAIN else 0.0)        # 69.0 (46.2) B / event
BYTES_EVENT = BYTES_INGEST + BYTES_TDIGEST                                                  # 101.0 B / event


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gysketch", choices=["gysketch", "reference"])
    ap.add_argument("--events", type=int, default=100_000_000, help="events per rank per step")
    ap.add_argument("--max-batch", type=int, default=(1 << 27) - 1, help="events per device batch (value path: one batch per step)")
    ap.add_argument("--stage-batch", type=int, default=1 << 23, help="events per H2D chunk on the host-buffer path")
    ap.add_argument("--cpu-sample", type=int, default=20_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the engine's answers (a fixed sample, see dump_outputs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def rank_service_ids(rank):
    from gyeeta_b200 import synth
    ids = synth.splitmix64(np.arange(1, NSVC + 1, dtype=np.uint64) + np.uint64(rank * NSVC))
    ids[ids == 0] = 1
    return ids


def rank_task_ids(rank):
    from gyeeta_b200 import synth
    return synth.splitmix64(np.arange(1, NTASK + 1, dtype=np.uint64) + np.uint64((1 << 40) + rank * NTASK))


# ---------------------------------------------------------------------------------------------------------------
# synthetic stream on the GPU (same formulas as gyeeta_b200/synth.py::gen_mixed)
# ---------------------------------------------------------------------------------------------------------------
def gen_events_gpu(torch, n, seed, rank, world, dev):
    from gyeeta_b200 import synth
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    # a service id is unique per host (CityHash of host + netns + ip + port in the reference): every rank owns its own ids
    svc_ids = torch.from_numpy(rank_service_ids(rank).view(np.int64)).to(dev)
    task_ids = torch.from_numpy(rank_task_ids(rank).view(np.int64)).to(dev)
    cdf_s = torch.from_numpy(synth.zipf_cdf(NSVC, ZIPF_S)).to(dev)
    cdf_t = torch.from_numpy(synth.zipf_cdf(NTASK, ZIPF_S)).to(dev)
    out = torch.empty((n, 4), dtype=torch.int64, device=dev)
    chunk = 1 << 23
    for off in range(0, n, chunk):
        m = min(chunk, n - off)
        u = torch.rand(m, generator=g, device=dev, dtype=torch.float64)
        srank = torch.searchsorted(cdf_s, u).clamp_(max=NSVC - 1)
        kind = torch.rand(m, generator=g, device=dev)
        is_resp = kind < 0.70
        is_task = kind >= 0.90
        tu = torch.rand(m, generator=g, device=dev)
        ttype = torch.where(tu < 0.45, 2, torch.where(tu < 0.90, 4, 1))
        etype = torch.where(is_resp, 5, torch.where(is_task, 6, ttype)).to(torch.int64)
        trank = torch.searchsorted(cdf_t, torch.rand(m, generator=g, device=dev, dtype=torch.float64)).clamp_(max=NTASK - 1)
        w0 = torch.where(is_task, task_ids[trank], svc_ids[srank])
        # client key bound to (service rank % 8) groups; 64-bit mix done with int64 wraparound arithmetic
        cli = torch.randint(0, NCLIENTS // 8, (m,), generator=g, device=dev, dtype=torch.int64) * 8 + (srank % 8)
        z = cli + (1 << 48) + (-7046029254386353131)           # 0x9E3779B97F4A7C15 as int64
        z = (z ^ ((z >> 30) & ((1 << 34) - 1))) * (-4658895280553007687)
        z = (z ^ ((z >> 27) & ((1 << 37) - 1))) * (-7723592293110705685)
        flow = z ^ ((z >> 31) & ((1 << 33) - 1))
        resp_us = torch.exp(torch.randn(m, generator=g, device=dev) * 1.5 + float(np.log(2000.0))).clamp_(max=9.0e8)
        tcp_b = torch.exp(torch.randn(m, generator=g, device=dev) * 2.0 + float(np.log(4096.0))).clamp_(max=4.0e9)
        cpu_pct = (torch.rand(m, generator=g, device=dev) * 400.0)
        value = torch.where(is_resp, resp_us, torch.where(is_task, cpu_pct, tcp_b)).to(torch.int64)
        cpu_delay = torch.exp(torch.randn(m, generator=g, device=dev) * 2.0 + float(np.log(30.0))).clamp_(max=1.0e5).to(torch.int64)
        blkio = torch.exp(torch.randn(m, generator=g, device=dev) * 2.5 + float(np.log(5.0))).clamp_(max=1.0e5).to(torch.int64)
        w1 = torch.where(is_task, cpu_delay | (blkio << 32), flow)
        # hosts of this rank's shard: host_idx % world == rank
        host = (srank % (NHOSTS // max(world, 1))) * world + rank
        out[off: off + m, 0] = w0
        out[off: off + m, 1] = w1
        out[off: off + m, 2] = value | (host << 32)
        out[off: off + m, 3] = 1 | (etype << 32)
    return out


def pack_kinds_pinned(torch, ev):
    """the events of one batch as three page-locked arrays of packed per-kind records (gysk_resp16 / gysk_tcp24 / gysk_task24):
    -> [(raw kind, pinned int64 tensor, record count)]"""
    from gyeeta_b200 import engine as ge
    w0, w1, w2, w3 = ev[:, 0], ev[:, 1], ev[:, 2], ev[:, 3]
    etype = (w3 >> 32) & 0xFFFF
    host = (w2 >> 32) & 0xFFFF
    val = w2 & 0xFFFFFFFF
    out = []
    m = etype == 5
    r = torch.stack([w0[m], val[m] | (host[m] << 32) | ((w1[m] & 0xFF) << 48)], dim=1)             # flags byte 0
    out.append((ge.RAW_RESP16, r))
    m = (etype >= 1) & (etype <= 4)
    t = torch.stack([w0[m], w1[m], val[m] | (host[m] << 32) | (etype[m] << 48)], dim=1)
    out.append((ge.RAW_TCP24, t))
    m = etype == 6
    k = torch.stack([w0[m], val[m] | ((w1[m] & 0xFFFFFFFF) << 32), ((w1[m] >> 32) & 0xFFFFFFFF) | (host[m] << 32)], dim=1)
    out.append((ge.RAW_TASK24, k))
    res = []
    for kind, d in out:
        h = torch.empty(d.shape, dtype=torch.int64, pin_memory=True)
        h.copy_(d)
        res.append((kind, h, d.shape[0]))
    return res


def wire_leg(ge, local, nthreads=16, rounds_per_thread=8, total_events=32_000_000):
    """e2e_wire: the boundary call itself under madhava's threading model — `nthreads` host threads (the L2 handle_l2_misc threads,
    server/gy_mconnhdlr.cc:5128), each handing the engine what its partha connections deliver: whole COMM_HEADER messages of
    TCP_CONN_NOTIFY (280-byte records, 2048 per message = MAX_NUM_CONNS) and AGGR_TASK_STATE_NOTIFY (72-byte records) through
    gysk_ingest_msg, and arrays of the 24-byte tcp_ipv4_resp_event_t through gysk_ingest_raw, 70 / 20 / 10 by events. Pageable host
    memory (messages arrive in socket buffers); validation, 280 B -> 32 B compaction on the calling thread, per-thread page-locked
    staging, H2D and the device batches are all inside the wall-clock region; one query + sync closes it."""
    from gyeeta_b200 import synth, wire
    rng = np.random.default_rng(77)
    svc_ids = rank_service_ids(0)
    task_ids = synth.splitmix64(np.arange(1, NTASK + 1, dtype=np.uint64) + np.uint64(1 << 40))
    cdf_s, cdf_t = synth.zipf_cdf(NSVC, ZIPF_S), synth.zipf_cdf(NTASK, ZIPF_S)
    NT, NK, NR = 2048, 1024, 7168                       # records per round: TCP_CONN, AGGR_TASK_STATE, resp events
    per_round = NT + NK + NR
    eng = ge.Engine(device=local, max_svcs=1 << 18, max_tasks=1 << 15, max_batch=1 << 24)
    work = []
    for t in range(nthreads):
        rounds = []
        for _r in range(rounds_per_thread):
            srank = np.minimum(np.searchsorted(cdf_s, rng.random(NT)), NSVC - 1)
            c = np.zeros(NT, dtype=wire.TCP_CONN)
            c["ser_glob_id"] = svc_ids[srank]
            c["cli_task_aggr_id"] = synth.splitmix64(rng.integers(1, NCLIENTS, NT).astype(np.uint64) + np.uint64(1 << 48))
            closed = rng.random(NT) < 0.5
            c["is_accept"] = 1
            c["tusec_start"] = 1_700_000_000_000_000
            c["tusec_close"] = np.where(closed, 1_700_000_005_000_000, 0)
            c["bytes_sent"] = np.exp(rng.normal(np.log(4096.0), 2.0, NT)).astype(np.uint64)
            c["bytes_rcvd"] = np.exp(rng.normal(np.log(1024.0), 2.0, NT)).astype(np.uint64)
            k = np.zeros(NK, dtype=wire.TASK)
            k["aggr_task_id"] = task_ids[np.minimum(np.searchsorted(cdf_t, rng.random(NK)), NTASK - 1)]
            k["total_cpu_pct"] = rng.random(NK) * 400.0
            k["cpu_delay_msec"] = np.minimum(np.exp(rng.normal(np.log(30.0), 2.0, NK)), 1e5).astype(np.uint32)
            k["blkio_delay_msec"] = np.minimum(np.exp(rng.normal(np.log(5.0), 2.5, NK)), 1e5).astype(np.uint32)
            rr = np.minimum(np.searchsorted(cdf_s, rng.random(NR)), NSVC - 1)
            r = np.zeros(NR, dtype=wire.RESP4)
            r["saddr"] = 0x0A000000 + rr
            r["daddr"] = rng.integers(1, 1 << 32, NR, dtype=np.uint64).astype(np.uint32)
            r["netns"] = 4026531840
            r["sport"] = 0x901F                           # htons(8080)
            r["dport"] = rng.integers(1024, 65536, NR).astype(np.uint16)
            r["lrcvtime"] = rng.integers(0, 1 << 31, NR).astype(np.uint32)
            r["lsndtime"] = r["lrcvtime"] + np.minimum(np.exp(rng.normal(np.log(2.0), 1.5, NR)), 9.0e5).astype(np.uint32)
            rounds.append((wire.build_msg_fixed(ge.NOTIFY_TCP_CONN, c), wire.build_msg_fixed(ge.NOTIFY_AGGR_TASK_STATE, k), r))
        work.append(rounds)
    iters = max(1, total_events // (nthreads * per_round))
    # the producers are native threads (libgysynth.so's gysyn_wire_run): Python threads would time the interpreter lock, not the library

    class Round(C.Structure):
        _fields_ = [("msg1", C.c_void_p), ("msg2", C.c_void_p), ("raw", C.c_void_p), ("len1", C.c_uint32), ("len2", C.c_uint32),
                    ("nraw", C.c_uint32), ("raw_kind", C.c_uint32)]

    S = C.CDLL(os.path.join(ROOT, "gyeeta_b200", "libgysynth.so"))
    S.gysyn_wire_run.restype = C.c_double
    S.gysyn_wire_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    rounds = (Round * (nthreads * rounds_per_thread))()
    for t in range(nthreads):
        for r_, (m1, m2, r) in enumerate(work[t]):
            rounds[t * rounds_per_thread + r_] = Round(m1.ctypes.data, m2.ctypes.data, r.ctypes.data, len(m1), len(m2), len(r), ge.RAW_TCP_IPV4_RESP)
    fmsg = C.cast(eng.L.gysk_ingest_msg, C.c_void_p)
    fraw = C.cast(eng.L.gysk_ingest_raw, C.c_void_p)
    nerr = C.c_int(0)
    errs = []

    def run(count):
        t0 = time.perf_counter()
        S.gysyn_wire_run(eng.h, fmsg, fraw, C.cast(eng._host_id, C.c_void_p), C.cast(rounds, C.c_void_p), nthreads, rounds_per_thread, count, C.byref(nerr))
        if nerr.value:
            errs.append(nerr.value)
        eng.query_svcs(svc_ids[:256])
        eng.sync()
        return time.perf_counter() - t0

    run(max(1, iters // 8))                              # registers the ids, faults the stages in
    sec = run(iters)
    nev = nthreads * iters * per_round
    st = eng.stats()
    out = {"value": nev / sec, "unit": "events/s", "threads": nthreads, "events": nev, "sec": sec, "errors": len(errs),
           "wire_bytes_per_event": (len(work[0][0][0]) + len(work[0][0][1]) + work[0][0][2].nbytes) / per_round,
           "h2d_bytes_per_event": (NT * 32 + NK * 32 + NR * 24) / per_round,
           "what": "16 native threads x (TCP_CONN_NOTIFY 2048 x 280 B + AGGR_TASK_STATE_NOTIFY 1024 x 72 B via gysk_ingest_msg, 7168 x 24 B "
                   "tcp_ipv4_resp_event_t via gysk_ingest_raw), pageable memory, host wall clock incl. final query + sync",
           "wire_msgs_ok": st.get("wire_msgs_ok")}
    eng.close()
    return out


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        # samples that arrived while the timed region ran; when the region is shorter than the sampler's reaction time, the samples of
        # the whole loaded period (warm-up steps, timed region, diagnostic steps) stand in — all of them under the same load
        inside = [r for t, r in self.rows if t_begin is not None and t_begin <= t <= t_end + 0.03]
        use = inside if len(inside) >= 2 else [r for _t, r in self.rows]
        sm, smax, reasons = [], [], set()
        for r in use:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_inside_timed_region": len(inside)}


def ncu_traffic_per_event():
    """DRAM bytes per event of each kernel group from the committed `ncu --set full` captures (profiles/ncu_traffic.json)"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------------------------
def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def shard_owner(ev_np, nthreads, mode):
    """which host thread takes an event. "host": host_idx % T — how madhava pins a partha to an L2 thread
    (gy_mconnhdlr.cc:16252); "balanced": hosts dealt to threads heaviest first (longest-processing-time), still one thread per
    host; "svc": by service / task id — finer than the reference can shard, shown as the upper bound the skew allows."""
    if nthreads == 1:
        return np.zeros(len(ev_np), dtype=np.int32)
    if mode == "host":
        return (ev_np["host_idx"] % nthreads).astype(np.int32)
    if mode == "svc":
        return ((ev_np["svc_id"] * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)).astype(np.int64).__mod__(nthreads).astype(np.int32)
    cnt = np.bincount(ev_np["host_idx"])
    load = np.zeros(nthreads, dtype=np.int64)
    host_thr = np.zeros(len(cnt), dtype=np.int32)
    for h in np.argsort(-cnt, kind="stable"):
        t = int(np.argmin(load))
        host_thr[h] = t
        load[t] += cnt[h]
    return host_thr[ev_np["host_idx"]]


class CpuPort:
    """the oracle port on `nthreads` host threads: events pre-sharded (shard_owner), one engine per thread, ids registered and state
    faulted in by an untimed first pass; timed() = one pass of every thread over its shard (gyo_bench_ingest, oracle/gysk_oracle.c)"""

    def __init__(self, ev_np, nthreads, mode="host"):
        from oracle import pyoracle as po
        self.L = po.lib()
        owner = shard_owner(ev_np, nthreads, mode)
        order = np.argsort(owner, kind="stable")
        cuts = np.searchsorted(owner[order], np.arange(1, nthreads))
        self.shards = [np.ascontiguousarray(a) for a in np.split(ev_np[order], cuts)]
        self.engines = [po.OracleEngine(max_svcs=NSVC + 16, max_tasks=NTASK + 16) for _ in range(nthreads)]
        self.nthreads, self.n = nthreads, len(ev_np)
        self.eh = (C.c_void_p * nthreads)(*[e.h for e in self.engines])
        self.sp = (C.c_void_p * nthreads)(*[s.ctypes.data for s in self.shards])
        self.cn = (C.c_uint64 * nthreads)(*[len(s) for s in self.shards])
        self.largest_shard_frac = float(max(len(s) for s in self.shards)) / max(1, self.n)
        self.timed()

    def timed(self):
        return self.L.gyo_bench_ingest(self.eh, self.sp, self.cn, self.nthreads, 1 << 22)

    def close(self):
        for e in self.engines:
            e.close()


def cpu_port_rate(ev_np, nthreads, mode="host", repeat=1):
    cp = CpuPort(ev_np, nthreads, mode)
    best = min(cp.timed() for _ in range(repeat))
    frac = cp.largest_shard_frac
    cp.close()
    return len(ev_np) / best, best, frac


def cpu_arm_report(ev_np, ncores):
    """1-thread and N-thread rates of the CPU port under the three shardings, and the reference's own add_data loop"""
    from oracle import pyoracle as po
    one = ev_np[: max(1, min(len(ev_np), max(len(ev_np) // 4, 1_000_000)))]
    r1, s1, _ = cpu_port_rate(one, 1)
    out = {"threads_1": {"events_per_s": r1, "sample_events": len(one)}}
    for mode in ("host", "balanced", "svc"):
        r, sec, frac = cpu_port_rate(ev_np, ncores, mode)
        out[f"threads_{ncores}_{mode}"] = {"events_per_s": r, "speedup_vs_1": r / r1, "largest_shard_frac": frac, "sec": sec}
    resp = ev_np[ev_np["type"] == 5]
    if len(resp) and po.ref() is not None:
        _, slots = np.unique(resp["svc_id"], return_inverse=True)
        vals = (resp["value"] // 1000).astype(np.int64)
        out["ref_gy_histogram_add_data_only"] = {"threads_1": po.ref_hist_rate(slots[: len(slots) // 4], vals[: len(slots) // 4], 1),
                                                 f"threads_{ncores}": po.ref_hist_rate(slots, vals, ncores),
                                                 "unit": "RESP samples/s", "what": "the reference's own GY_HISTOGRAM<int64_t, RESP_TIME_HASH>::add_data "
                                                 "compiled from /root/reference (oracle/_ref), samples pre-sharded by slot % threads"}
    return out


def workload_config(args, world):
    """the `config` of the JSON line: the same for the product arm and for `--impl reference` (which times a bounded sample of it)"""
    return {"workload": "configs[2]: 100M mixed RESP/TCP/TASK (70/20/10) events, 100K services, count-min + HLL + "
                        "fixed-bucket histograms + t-digest(200)", "events_per_step_per_gpu": args.events, "services": NSVC,
            "zipf_s": ZIPF_S, "max_batch": args.max_batch, "stage_batch": args.stage_batch, "parallelism": f"host-shard x{world}",
            "l2": "inputs (3.2 GB/step) larger than L2, no flush needed"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port: GY_HISTOGRAM add_data + count-min +
    HLL + t-digest per event, open-addressing id tables), all host threads, events pre-sharded by host like madhava pins a partha
    to an L2 thread. `value` = the host-sharded N-thread rate; the balanced / by-service shardings and the 1-thread rate are listed
    beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gyeeta_b200 import synth
    from oracle import pyoracle as po
    po.lib()
    ncores = os.cpu_count() or 1
    n = int(min(args.cpu_sample, args.events))
    rng = np.random.default_rng(3)
    ev = synth.gen_mixed(rng, n, NSVC, ntask=NTASK, zipf_s=ZIPF_S, nhosts=NHOSTS, nclients=NCLIENTS)
    cp = CpuPort(ev, ncores)
    for _ in range(args.warmup):
        cp.timed()
    secs = [cp.timed() for _ in range(args.steps)]
    cp.close()
    rate = n * len(secs) / float(np.sum(secs))
    ms = float(np.mean(secs)) * 1e3
    detail = cpu_arm_report(ev, ncores)
    print(json.dumps({
        "impl": "reference", "metric": "events/sec aggregated", "value": rate, "unit": "events/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus)),
        "sample_events_per_step": n,
        "cpu_baseline": {"value": rate, "unit": "events/s", "cores": ncores, "kind": "port", "cpu_model": cpu_model(),
                         "sample": f"each step = {n} events of the same generator and mix (a rate per event: the bounded sample keeps the run "
                                   f"to a few minutes of CPU), pre-sharded by host over {ncores} threads", "detail": detail},
        "e2e": {"value": rate, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------
# outputs of the timed path
# ---------------------------------------------------------------------------------------------------------------
DUMP_SEED = 20261017
DUMP_SVCS = 2048            # the 64 hottest services + a seeded sample of the rest
DUMP_TASKS = 1024
DUMP_HLL_SVCS = 256
DUMP_CMS_CELLS = 1 << 20


def dump_outputs(eng, ge, rank, world, out_dir):
    """What a caller reads back after the timed steps, from a fixed seeded sample of the state (~39 MB): for DUMP_SVCS of this
    rank's services the response histogram of the open window (hist_resp: count, sum per bucket; hist_resp_total_max), every
    numeric field of the query_svcs summary (summary_<field>), the t-digest centroids (zero-padded to TD_CAP) and for the first
    DUMP_HLL_SVCS of them the HLL registers; the three process histograms of DUMP_TASKS tasks; DUMP_CMS_CELLS count-min cells
    (count and kbytes halves) and the engine's event counters. Ids are given as indices into rank_service_ids / rank_task_ids.
    Everything is float64 (integers below 2^53, exact) except the HLL registers (float32). With world > 1 each rank writes
    its own files, suffixed _rank<r>."""
    rng = np.random.default_rng(DUMP_SEED)
    svc_idx = np.union1d(np.arange(64), rng.choice(np.arange(64, NSVC), DUMP_SVCS - 64, replace=False))
    task_idx = np.sort(rng.choice(NTASK, DUMP_TASKS, replace=False))
    cells = np.sort(rng.choice(eng.cfg.cms_depth << eng.cfg.cms_log2_width, DUMP_CMS_CELLS, replace=False))
    svc_ids, task_ids = rank_service_ids(rank)[svc_idx], rank_task_ids(rank)[task_idx]
    out = {"svc_index": svc_idx, "task_index": task_idx, "cms_cell": cells}

    hist = np.zeros((len(svc_ids), 15, 2)); tot_max = np.zeros((len(svc_ids), 2))
    td_means = np.zeros((len(svc_ids), ge.TD_CAP)); td_weights = np.zeros((len(svc_ids), ge.TD_CAP)); td_min_max = np.zeros((len(svc_ids), 2))
    for i, sid in enumerate(svc_ids):
        h = eng.export_hist(int(sid), ge.HIST_RESP_CUR)
        if h is not None:
            hist[i, :, 0], hist[i, :, 1], tot_max[i] = h[0]["count"], h[0]["sum"], h[1:]
        t = eng.export_tdigest(int(sid))
        if t is not None:
            td_means[i, : len(t[0])], td_weights[i, : len(t[1])], td_min_max[i] = t[0], t[1], t[2:]
    out.update(hist_resp=hist, hist_resp_total_max=tot_max, tdigest_means=td_means, tdigest_weights=td_weights, tdigest_min_max=td_min_max)
    summ = eng.query_svcs(svc_ids)
    for f, _ in ge.SvcSummary._fields_:
        if f != "glob_id":
            out["summary_" + f] = np.array([s[f] for s in summ], dtype=np.float64)
    hll = np.zeros((DUMP_HLL_SVCS, 1 << eng.cfg.hll_p), dtype=np.float32)
    for i, sid in enumerate(svc_ids[:DUMP_HLL_SVCS]):
        r = eng.export_hll(int(sid))
        if r is not None:
            hll[i] = r
    out["hll_registers"] = hll

    th = np.zeros((len(task_ids), 3, 15, 2))
    for i, tid in enumerate(task_ids):
        for j, which in enumerate((ge.HIST_TASK_CPU_PCT, ge.HIST_TASK_CPU_DELAY, ge.HIST_TASK_BLKIO_DELAY)):
            h = eng.export_hist(int(tid), which)
            if h is not None:
                th[i, j, :, 0], th[i, j, :, 1] = h[0]["count"], h[0]["sum"]
    out["hist_task"] = th
    cms = eng.export_cms()[cells]
    out["cms_count"], out["cms_kbytes"] = cms & np.uint64(0xFFFFFFFF), cms >> np.uint64(32)
    st = eng.stats()
    out["counters"] = np.array([st[k] for k in ("events_in", "events_dropped", "events_resp", "events_tcp", "events_task", "nsvcs", "ntasks")])

    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from gyeeta_b200 import engine as ge

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n = args.events

    eng = ge.Engine(device=local, max_svcs=1 << 17, max_tasks=1 << 15, max_batch=args.max_batch, stage_batch=args.stage_batch, rank=rank, world=world)
    # two DISTINCT batches of the same stream, alternated step by step: new flows / clients keep arriving, so the HLL register
    # CAS path, the hot-cell tables and the t-digest merges do real work in the timed region (one batch repeated would saturate them)
    NB = 2
    ev_devs = [gen_events_gpu(torch, n, 1234 + rank + 7919 * b, rank, world, dev) for b in range(NB)]
    ev_dev = ev_devs[0]
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    merge_events = []

    def merge_step():
        # the multi-GPU exchange: fold + ONE grouped NCCL launch + merge-compress inside libgysketch.so (gysk_merge_global),
        # once per query window = once per timed region here, not once per batch
        if world > 1:
            with torch.cuda.stream(stream):
                a = torch.cuda.Event(enable_timing=True); a.record()
            eng.merge_global()
            with torch.cuda.stream(stream):
                b = torch.cuda.Event(enable_timing=True); b.record()
            merge_events.append((a, b))

    def setup_logical_map():
        # BASELINE configs[3]: global per-logical-service stats, 16 hosts' instances per logical service; every rank passes the
        # same (glob_id, logical_id) list so the dense logical index is identical everywhere
        ids_all = np.concatenate([rank_service_ids(r) for r in range(world)])
        logical_all = np.tile(np.arange(NSVC, dtype=np.uint64) // np.uint64(16) + np.uint64(1), world)
        eng.set_logical_map(ids_all, logical_all)

    step_no = [0]

    def step_device():
        eng.ingest_device_ptr(ev_devs[step_no[0] % NB].data_ptr(), n)
        step_no[0] += 1

    for b in range(NB):
        eng.ingest_device_ptr(ev_devs[b].data_ptr(), n)       # registers this rank's services
    eng.sync()
    if world > 1:
        from gyeeta_b200 import dist as gd
        setup_logical_map()
        gd.nccl_comm_init(eng, dist)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                # before the warm-up steps: nvidia-smi needs a few hundred ms to deliver its first sample
    for _ in range(args.warmup):
        step_device()
    merge_step()
    eng.sync()
    launches0 = eng.stats()["kernel_launches"]
    eng.profile_enable(True)
    barrier()
    wall_begin = time.perf_counter()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        t0.record()
    for _ in range(args.steps):
        step_device()
    merge_step()                       # the window's one sketch merge is inside the timed region
    with torch.cuda.stream(stream):
        t1.record()
    eng.sync()
    wall_end = time.perf_counter()
    barrier()
    dev_ms = t0.elapsed_time(t1)
    launches = eng.stats()["kernel_launches"] - launches0           # kernels of libgysketch.so launched inside the timed region
    ms_ing, ms_td, nb = eng.profile_read()
    if args.dump_outputs:
        dump_outputs(eng, ge, rank, world, args.dump_outputs)       # before the diagnostic batches below change the state
    # share of the events that took the hot-row way (two REDs into the service's dense value bins inside ingest_kernel instead of a
    # sort key): read from the engine after the timed region — response samples of the last batch minus its sort keys
    resp0 = eng.stats()["events_resp"]
    eng.ingest_device_ptr(ev_devs[step_no[0] % NB].data_ptr(), n)
    hot_share = max(0.0, (eng.stats()["events_resp"] - resp0 - eng.last_batch_keys()) / float(n))
    hot_rows = eng.hot_rows_in_use()
    eng.profile_read()                 # drop that batch's timings
    # diagnostic (outside the timed region): per-step spread of the two kernel groups
    spread = {"ingest_ms": [], "chain_ms": []}
    for i in range(min(args.steps, 8)):
        eng.ingest_device_ptr(ev_devs[i % NB].data_ptr(), n)
        a, b, _nb = eng.profile_read()
        spread["ingest_ms"].append(round(a, 3)); spread["chain_ms"].append(round(b, 3))
    eng.profile_enable(False)
    clocks = sampler.stop(wall_begin, wall_end) if rank == 0 else None
    merge_events_value = merge_events[-1:] if merge_events else []

    tms = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    max_ms = float(tms.item())
    value = world * n * args.steps / (max_ms * 1e-3)

    # ---- e2e: host buffers through the C ABI, H2D in the timed region + D2H of summaries --------------------------
    # headline `e2e`: the packed per-kind records (gysk_resp16 / gysk_tcp24 / gysk_task24, include/gysketch.h) a feeder that knows the
    # kind of a batch ships: 18.4 B/event on this mix; expanded on the device. `e2e_event32`: the same events as 32-byte canonical
    # records through gysk_ingest_pinned (round 1's path).
    e2e = e2e32 = None
    if not args.no_e2e:
        qids = ev_dev[:4096, 0].cpu().numpy().view(np.uint64)[:256].copy()

        def timed_e2e(step_fn, h2d_bytes):
            for _ in range(max(1, args.warmup // 2)):
                step_fn()
            barrier()
            w0 = time.perf_counter()
            for _ in range(args.steps):
                step_fn()
            merge_step()
            eng.sync()
            torch.cuda.synchronize()
            w1 = time.perf_counter()
            te = torch.tensor([w1 - w0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return {"value": world * n * args.steps / float(te.item()), "unit": "events/s",
                    "h2d_bytes_per_step": int(h2d_bytes + len(qids) * 8), "d2h_bytes_per_step": int(len(qids) * C.sizeof(ge.SvcSummary)),
                    "timed_with": "host wall clock around the C-ABI calls incl. final sync (max over ranks)"}

        packed = [pack_kinds_pinned(torch, e_) for e_ in ev_devs]
        torch.cuda.synchronize()

        def step_packed():
            for kind, arr, cnt in packed[step_no[0] % NB]:
                eng.ingest_raw_ptr(kind, arr.data_ptr(), cnt)
            step_no[0] += 1
            return eng.query_svcs(qids)         # syncs, copies the summaries device -> host

        e2e = timed_e2e(step_packed, sum(arr.numel() * 8 for _k, arr, _c in packed[0]))
        e2e["records"] = "gysk_resp16 / gysk_tcp24 / gysk_task24 via gysk_ingest_raw, page-locked, decoded on the device"
        e2e["bytes_per_event"] = e2e["h2d_bytes_per_step"] / n
        del packed

        hosts = [torch.empty((n, 4), dtype=torch.int64, pin_memory=True) for _ in range(NB)]
        for b in range(NB):
            hosts[b].copy_(ev_devs[b])
        torch.cuda.synchronize()

        def step_e2e32():
            eng.ingest_pinned_ptr(hosts[step_no[0] % NB].data_ptr(), n)
            step_no[0] += 1
            return eng.query_svcs(qids)

        e2e32 = timed_e2e(step_e2e32, n * 32)
        e2e32["records"] = "32-byte gysk_event via gysk_ingest_pinned"
        del hosts

    # ---- accuracy: t-digest p99 vs exact on the hottest services --------------------------------------------------
    acc = None
    if rank == 0:
        w0col = ev_dev[:, 0]
        is_resp = ((ev_dev[:, 3] >> 32) & 0xFFFF) == 5
        u, cnt = torch.unique(w0col[:2_000_000][is_resp[:2_000_000]], return_counts=True)
        order = torch.argsort(cnt, descending=True)
        hot = torch.cat([u[order[:4]], u[order[40:44]], u[order[400:404]]])
        rows = []
        for sid in hot.tolist():
            vals = torch.cat([(e_[:, 2][(e_[:, 0] == sid) & (((e_[:, 3] >> 32) & 0xFFFF) == 5)] & 0xFFFFFFFF) for e_ in ev_devs]).double()
            if vals.numel() < 10_000:
                continue
            # the steps alternate the two batches: the digest holds many copies of both, the quantiles are those of their union
            ex = torch.quantile(vals[: 16_000_000], torch.tensor([0.5, 0.95, 0.99], device=dev, dtype=torch.float64),
                                interpolation="lower").cpu().numpy()
            got = eng.quantiles(sid & 0xFFFFFFFFFFFFFFFF, [0.5, 0.95, 0.99])
            rows.append((int(vals.numel()), np.abs(got - ex) / ex))
        if rows:
            # by sample count: the exact p99 of n draws is itself an order statistic with relative 1-sigma noise
            # ~ 0.5 % x sqrt(47000 / n) on this log-normal (sigma 1.5) stream, so the small classes measure that noise, the hot one the digest
            acc = {"against": "exact sorted quantile of the same samples", "classes": {}}
            for name, lo, hi in (("n_ge_1M", 1_000_000, 1 << 62), ("n_100K_1M", 100_000, 1_000_000), ("n_10K_100K", 10_000, 100_000)):
                sel = [r for r in rows if lo <= r[0] < hi]
                if not sel:
                    continue
                e = np.max(np.array([r[1] for r in sel]), axis=0)
                nmin = min(r[0] for r in sel)
                acc["classes"][name] = {"services": len(sel), "min_samples": nmin, "max_rel_err_p50": float(e[0]), "max_rel_err_p95": float(e[1]),
                                        "max_rel_err_p99": float(e[2]), "p99_order_statistic_noise_1sigma": float(0.005 * np.sqrt(47000.0 / nmin))}
            e = np.max(np.array([r[1] for r in rows]), axis=0)
            acc.update({"services_checked": len(rows), "max_rel_err_p50": float(e[0]), "max_rel_err_p95": float(e[1]), "max_rel_err_p99": float(e[2])})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    wire = None
    if not args.no_e2e and world == 1:
        del ev_devs[1:]
        torch.cuda.empty_cache()
        wire = wire_leg(ge, local)

    peak, peak_src = measured_peak_gbs()
    nev_total = n * args.steps
    roof = []
    traffic = ncu_traffic_per_event()
    # a hot response sample's histogram-cell read-modify-write (32 of its 98 B, SURVEY.md §8d) happens in ingest_kernel — the two
    # 64-bit REDs into its value bin — not in the chain: those bytes move from one kernel group to the other, the sum stays 101 B
    moved = 32.0 * hot_share
    for name, key, ms, bpe in (("ingest_kernel", "ingest_kernel", ms_ing, BYTES_INGEST + moved),
                               ("sort + runs + bins-merge chain (os_pass x4, runs_mark, runs_sum, bins_merge)" + (" with side_drain_kernel beside it" if SIDE_DRAIN else ""), "chain", ms_td, BYTES_TDIGEST - moved)):
        if ms > 0:
            ach = nev_total * bpe / (ms * 1e-3) / 1e9
            tr = traffic.get(key, {}).get("dram_bytes_per_event")
            roof.append({"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": (tr * n if tr else None), "traffic_note": traffic.get(key, {}).get("source"),
                         "algorithmic_bytes_per_launch": bpe * n, "ms_per_launch": ms / max(nb, 1),
                         "ms_total": ms, "launch_groups": nb, "algorithmic_bytes_per_event": bpe, "peak_source": peak_src})
    # `roofline` = the dominant SINGLE kernel: ingest_kernel is one launch per device batch and holds the largest share of any
    # individual kernel (profiles/r02_launches_*.csv); the chain is 7 launches of 4 kernels
    roof.sort(key=lambda r: 0 if r["kernel"] == "ingest_kernel" else 1)
    whole = nev_total * BYTES_EVENT / (max_ms * 1e-3) / 1e9

    cpu = None
    if not args.no_cpu_baseline:
        ncores = os.cpu_count() or 1
        ns = int(min(args.cpu_sample, n))
        ev_np = ev_dev[:ns].cpu().numpy().view(np.uint8).reshape(-1).view(ge.EVENT_DTYPE)
        r, sec, frac = cpu_port_rate(ev_np, ncores)
        r1, _s1, _ = cpu_port_rate(ev_np[: max(ns // 4, min(ns, 1_000_000))], 1)
        cpu = {"value": r, "unit": "events/s", "cores": ncores, "kind": "port", "cpu_model": cpu_model(), "one_thread_events_per_s": r1,
               "largest_shard_frac": frac,
               "sample": f"first {ns} events of rank 0's stream, pre-sharded by host over {ncores} threads ({sec:.1f} s); "
                         "1-thread rate on a quarter of it; more shardings in `bench.py --impl reference`"}

    out = {
        "metric": "events/sec aggregated", "value": value, "unit": "events/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": e2e, "e2e_event32": e2e32, "e2e_wire": wire, "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roof[0] if roof else None, "roofline_other": roof[1:] or None,
        "roofline_whole_step": {"achieved": whole, "peak": peak, "unit": "GB/s", "frac": whole / peak,
                                "algorithmic_bytes_per_event": BYTES_EVENT},
        "hot_rows": {"rows_in_use": hot_rows, "share_of_events": hot_share,
                     "what": "response samples of services with >= 4096 samples in an earlier batch: two REDs into the service's dense "
                             "L2-resident value bins inside ingest_kernel instead of a sort key; their 32 B/sample of histogram-cell "
                             "traffic are counted with ingest_kernel (54.8 + 32 x share B/event), not with the chain"},
        "cpu_baseline": cpu, "accuracy": acc, "per_step_spread_ms": spread,
        "merge": ({"logical_services": NSVC // 16,
                   "what": "gysk_merge_global: fold kernels + ONE ncclGroup (3 all-reduces: u64 sum / i64 max / u8 max, 1 all-gather of t-digest slabs) + merge-compress, once per timed window", "merge_ms_of_the_window": (float(merge_events_value[0][0].elapsed_time(merge_events_value[0][1])) if merge_events_value else None)}
                  if world > 1 else None),
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
