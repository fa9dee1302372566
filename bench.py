#!/usr/bin/env python
"""bench.py — publish-topic matching throughput of the CUDA matcher (and the CPU reference arm).

One "step" = one pass of the hot path over one batch of synthetic publish topics:
    value  = topics/s with the batch resident in HBM (bfq_match_device; kernels + counter read-back)
    e2e    = topics/s through the host-buffer C-ABI call bfq_match (pinned host -> H2D -> kernels -> D2H result)
Workload = BASELINE.json config C4 by default (10M filters over 1000 tenants, Zipf-skewed fan-out, 1M-topic batch):
the metric is quoted "@10M filters" and it fits one B200. Under torchrun every rank owns its own tenants
(tenant sharding, no data-path collective; weak scaling: each rank hosts a full-size shard) unless --scaling strong.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nproc-per-node 8 ... bench.py --gpus 8
    python bench.py --impl reference        # the reference algorithm restated in C++ (oracle/), on host cores
    python bench.py --dump-outputs DIR      # also write what the last timed step computed (seeded sample) as DIR/*.npy
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the source tree may be read-only: the bench writes nothing into it

METRIC = "publish-topics matched/sec @10M filters"
UNIT = "topics/s"


def metric_name(args):
    """BASELINE.json's metric is quoted on C4 (10M filters); the other forward configs carry their own filter count"""
    return {"C1": "publish-topics matched/sec @10k filters (BASELINE config C1)", "C2": "publish-topics matched/sec @1M filters, 1 tenant (BASELINE config C2)",
            "C3": "publish-topics matched/sec @10M filters, 1000 tenants x 10k (BASELINE config C3)"}.get(args.config, METRIC)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=["C1", "C2", "C3", "C4", "C5"],
                    help="C4 is the headline (and the default); C5 = the inverse path (retained topics matched BY wildcard filters)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; invalid as a bench number)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1 only; either way ONE filter set is tenant-sharded over the ranks and the results are all-gathered inside the "
                         "timed step. weak (default): the publish batch grows with N (N x the config's batch, about one config batch per "
                         "rank); strong: the config's batch itself is split N ways")
    ap.add_argument("--no-replicate-hot", action="store_true", help="strong scaling: pure hash placement, no replicas of hot tenants")
    ap.add_argument("--retain-limit", type=int, default=10, help="C5: ids returned per filter (RetainMessageMatchLimit default 10; -1 = unlimited)")
    ap.add_argument("--exchange", default="ranges", choices=["ranges", "counts", "none"], help="N > 1: what the timed step all-gathers")
    ap.add_argument("--exchange-lag", type=int, default=1,
                    help="N > 1: matches enqueued ahead of the exchange being issued (2 was measured equal at N = 2: 0.604 vs 0.597 ms per step)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="topics in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--max-pfanout", type=int, default=2 ** 31 - 1, help="Setting.MaxPersistentFanout (reference default INT_MAX)")
    ap.add_argument("--max-gfanout", type=int, default=100, help="Setting.MaxGroupFanout (reference default 100)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (a seeded sample of the batch) as DIR/<name>.npy, "
                         "float64, under 64 MB in all: two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    return args


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (the sampler is started early so that its
    first samples exist before the region begins; rows are then filtered by timestamp)."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        """gpu_index: one index or a comma-separated list (rank 0 samples every GPU of the job from ONE nvidia-smi process:
        eight pollers at 20 ms contend for the driver and slow the ranks' launches)"""
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:   # wait for the first sample
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def begin(self):
        self.t_begin = time.time()

    def end(self):
        self.t_end = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        inside = [r for ts, r in self.rows if self.t_begin is not None and self.t_begin - 0.02 <= ts <= (self.t_end or ts) + 0.04]
        rows = inside or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_inside_timed_region": len(inside)}


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def pin_to_gpu_numa_node(dev_index):
    """Run this rank on the CPU socket its GPU hangs off (and first-touch its pinned buffers there): on a two-socket box a
    process that lands on the far socket sees a third less PCIe bandwidth, which is what the end-to-end number measures.
    Returns {"node", "cpus", "previous"} or None when the topology is not exposed; never raises."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return None
        cpus = _parse_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())
        previous = os.sched_getaffinity(0)
        target = cpus & previous
        if not target or target == previous:
            return None
        os.sched_setaffinity(0, target)
        return {"node": node, "cpus": len(target), "previous": previous}
    except Exception:
        return None


def make_roofline(sample_topic_bytes, st, ns, n_topics_per_launch, kernel_ms, gpu_ranges=None, gpu_routes=None, kernel_name=None):
    """`roofline` object of the JSON line. SURVEY.md §8(d): algorithmic bytes per topic
    B = len(topic) + 4 + 32 V + 8 P + 8 ranges (range-encoded output) + 4, with V / P / ranges counted by the oracle over the
    cpu_baseline sample (`st`, over `ns` topics: the WHOLE batch by default); achieved = B x topics per launch / the tier-0
    kernel's duration. Duplicate topics count like any other topic (the figure is per topic of the batch, whatever the
    kernel does about repeats)."""
    per_topic = (sample_topic_bytes + 4 * ns + 32 * st["V"] + 8 * st["P"] + 8 * st["ranges"] + 4 * ns) / ns
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = per_topic * n_topics_per_launch / (kernel_ms / 1000.0) / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel cannot be measured inside a bench run (ncu replays every
    # launch ~40 times); it comes from the committed `ncu --set full` capture of the same command, named here, or is null
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "latest_kernel_traffic.json")))
        if tj.get("config", "C4") == (kernel_name or {}).get("config", "C4"):
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
    except Exception:
        pass
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_source": traffic_src,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6650 GB/s",
            "frac_of_nominal_8000": achieved / 8000.0,
            "kernel": "match_topics_lane_kernel (tier 0, one lane per distinct topic)", "kernel_ms": kernel_ms, "alg_bytes_per_topic": per_topic,
            "alg_counters_per_topic": {"V": st["V"] / ns, "P": st["P"] / ns, "ranges": st["ranges"] / ns, "R": st["R"] / ns},
            "note": "algorithmic bytes per topic measured by the oracle over %d topics (%s)" % (ns, "the whole batch" if ns == n_topics_per_launch else "uniform random sample")}
    if gpu_ranges is not None and ns == n_topics_per_launch:
        # same population on both sides: the oracle's matched-filter and route counts must equal the GPU's own
        roof["counts_check"] = {"oracle_ranges": int(st["ranges"]), "gpu_ranges": int(gpu_ranges), "oracle_routes": int(st["R"]),
                                "gpu_routes": int(gpu_routes), "equal": int(st["ranges"]) == int(gpu_ranges) and int(st["R"]) == int(gpu_routes)}
    if traffic:
        # SURVEY.md §8(d) item (3): DRAM bytes the kernel actually moved (ncu capture of the same command) over the live time
        roof["dram_gbs_from_ncu_traffic"] = traffic / (kernel_ms / 1000.0) / 1e9
        roof["traffic_over_algorithmic"] = traffic / (per_topic * n_topics_per_launch)
    return roof


def make_workload(args, rank, world):
    """N = 1: the BASELINE config as written. N > 1: ONE filter set of that config, tenant-sharded over the ranks (tenant ->
    rank by fnv1a64(tenantId) mod N; hot tenants replicated, see workload.py), and a publish batch split by owner:
      weak   (default)  the batch is N times the config's (N GPUs serving N times the publish traffic of the same filter set):
                        about the config's batch per rank, whatever N
      strong            the config's batch itself, split N ways"""
    from bifromq_b200.workload import Workload
    if world > 1:
        return Workload(args.config, scale=args.scale, shard_index=rank, shard_count=world, replicate_hot=not args.no_replicate_hot,
                        topic_mult=world if args.scaling == "weak" else 1)
    return Workload(args.config, scale=args.scale)


def cpu_sample_indices(n, want):
    """UNBIASED bounded sample of a batch of n: the whole batch when it fits `want`, else a uniform random subset without
    replacement (seeded). Round 1 took "every topic of every 8th tenant", which over-weights the largest tenant (tenant index
    == Zipf rank): 1494 B/topic instead of the whole batch's 1162."""
    if n <= want:
        return np.arange(n)
    return np.sort(np.random.default_rng(0xB1F20).choice(n, want, replace=False))


# --dump-outputs: rows (topics, or filters for C5) of the seeded sample, values (route ranks / topic ids) kept of those rows, and
# throttle events kept. Every array is float64 (its integers are exact there): at most 6 x 8 B x 65536 + 8 B x 3M + 24 B x 0.5M,
# about 39 MB in all.
DUMP_ROWS, DUMP_VALUES, DUMP_EVENTS = 1 << 16, 3_000_000, 500_000


def sample_csr(offsets, values, pick, cap):
    """rows `pick` (ascending) of a CSR whose values are unordered within a row (as bfq_expand_device leaves them) -> (offsets
    over the picked rows, their values sorted within each row and cut after the first `cap`). torch tensors, any device;
    values must lie in [0, 2^32)."""
    import torch
    lens = offsets[pick + 1] - offsets[pick]
    out_off = torch.zeros(len(pick) + 1, dtype=torch.int64, device=offsets.device)
    out_off[1:] = torch.cumsum(lens, 0)
    total = int(out_off[-1])
    row = torch.repeat_interleave(torch.arange(len(pick), device=offsets.device), lens)
    pos = torch.arange(total, device=offsets.device) + (offsets[pick] - out_off[:-1])[row]
    key = torch.sort((row << 32) | values[pos].to(torch.int64)).values[:cap]
    return out_off, key & 0xFFFFFFFF


def write_dump(out_dir, arrays):
    """arrays (numpy or torch, any device) -> out_dir/<name>.npy in float64; an empty array is not written (no file says there
    is nothing, e.g. no throttle event in the sample)"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if not isinstance(a, np.ndarray):
            a = a.cpu().numpy()
        if a.size == 0:
            continue
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def dump_forward(out_dir, res, dev, stream):
    """the last timed step's bfq_match_device result, as its caller receives it, over a seeded sample of the batch's topics:
    matched routes before caps and matched filters per topic, the surviving route ranks (caps applied: bfq_expand_device's
    CSR, sorted within a topic), the number of throttle events per topic (persistent, group) and those events as
    (topic, rank, kind) rows, sorted"""
    import torch

    from bifromq_b200 import dist as D
    n = res.n_topics
    d_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    total = res.expand(d_off.data_ptr(), None, 0, stream)
    d_ranks = torch.zeros(max(total, 1), dtype=torch.int64, device=dev)
    res.expand(d_off.data_ptr(), d_ranks.data_ptr(), total, stream)
    torch.cuda.synchronize(dev)
    pick = torch.from_numpy(cpu_sample_indices(n, DUMP_ROWS)).to(dev)
    offsets, ranks = sample_csr(d_off, d_ranks, pick, DUMP_VALUES)
    route_count = D.device_view(res.d_route_count, n, "<i4", dev)[pick]
    span_count = D.device_view(res.d_span_count, n, "<i4", dev)[pick] & 0x3FFFFFFF   # the low 30 bits count the ranges
    counts = torch.zeros((len(pick), 2), dtype=torch.int64, device=dev)
    events = np.zeros((0, 3), np.int32)
    if res.n_throttled:
        ev = D.device_view(res.d_throttled, 3 * res.n_throttled, "<i4", dev).view(-1, 3)
        slot = torch.full((n,), -1, dtype=torch.int64, device=dev)   # topic -> its position in the sample
        slot[pick] = torch.arange(len(pick), device=dev)
        ev = ev[slot[ev[:, 0].long()] >= 0]
        counts = torch.bincount(2 * slot[ev[:, 0].long()] + (ev[:, 2] == 2), minlength=2 * len(pick)).view(-1, 2)   # kind 1 / 2
        events = ev.cpu().numpy()
        events = events[np.lexsort((events[:, 2], events[:, 1], events[:, 0]))][:DUMP_EVENTS]
    write_dump(out_dir, {"topics": pick, "route_count": route_count, "span_count": span_count, "offsets": offsets, "ranks": ranks,
                         "throttled_count": counts, "throttled": events})


def dump_inverse(out_dir, res):
    """the last timed step's bfq_rmatch result over a seeded sample of the query filters: total matches per filter and the
    returned topic ids, sorted within a filter (under a limit, WHICH ids come back is left open, as in the reference)"""
    import torch
    pick = cpu_sample_indices(res.n_filters, DUMP_ROWS)
    offsets, ids = sample_csr(torch.from_numpy(res.offsets), torch.from_numpy(res.ids), torch.from_numpy(pick), DUMP_VALUES)
    write_dump(out_dir, {"filters": pick, "totals": res.totals[pick], "offsets": offsets, "ids": ids})


_ORACLE_CACHE = {}


def oracle_for_sample(w, idx):
    """the oracle over ALL tenants' routes (a uniform topic sample touches every tenant) and the sampled topics as blobs"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    if _ORACLE_CACHE.get("w") is not w:
        kv = O.KV()
        kv.load(w.keys, w.key_off, w.vals, w.val_off)
        kv.freeze()
        _ORACLE_CACHE.update(w=w, kv=kv)
    kv = _ORACLE_CACHE["kv"]
    if len(idx) == w.n_topics:
        pb, poff = w.topics, np.ascontiguousarray(w.topic_off)
    else:
        off = np.asarray(w.topic_off)
        lens = (off[idx + 1] - off[idx]).astype(np.int64)
        poff = np.zeros(len(idx) + 1, np.int64)
        poff[1:] = np.cumsum(lens)
        pb = np.zeros(max(int(poff[-1]), 1), np.uint8)
        src = np.asarray(w.topics)
        for k, i in enumerate(idx.tolist()):   # <= a few hundred thousand short copies
            pb[poff[k]:poff[k + 1]] = src[off[i]:off[i + 1]]
    tt = np.ascontiguousarray(np.asarray(w.topic_tenant[:w.n_topics])[idx]).astype(np.int32)
    return O, kv, w.tenants, (pb, poff), tt


def run_cpu_baseline(w, args, mode_name, cached=False, n_passes=5, n_warm=0):
    """times the oracle on the host cores over a bounded, unbiased sample; returns the cpu_baseline dict and the per-topic
    algorithmic-byte figures (SURVEY.md §8d) measured on the same sample.
    mode_name: "trie" = the oracle's per-topic filter-trie walk over the WHOLE batch (also the exact V / P / ranges counters);
    "reference" = the literal TenantRouteMatcher.matchAll restatement, one call per topic (the production shape,
    DW/cache/TenantRouteCache.java:185-186) on a uniform random sample. cached=True puts a (tenant, topic) -> result map in
    front, the way TenantRouteCache (DW/cache/TenantRouteCache.java:100-139) serves repeated topics: every distinct pair is
    matched once, the repeats are lookups."""
    cores = os.cpu_count() or 1
    want = args.cpu_sample or (1 << 30 if mode_name == "trie" else 100000)
    idx = cpu_sample_indices(w.n_topics, want)
    O, kv, tenants, (pb, poff), tt = oracle_for_sample(w, idx)
    tb, toff = O.blob(tenants)
    n = len(idx)
    mode = O.MODE_TRIE if mode_name == "trie" else O.MODE_REFERENCE
    singleton = mode_name != "trie"
    n_unique = n
    if cached:
        # the cache's effect on the matcher's work: only the first occurrence of every (tenant, topic) pair reaches it
        seen, keep = set(), []
        mv = memoryview(np.ascontiguousarray(pb))
        for k in range(n):
            key = (int(tt[k]), bytes(mv[poff[k]:poff[k + 1]]))
            if key not in seen:
                seen.add(key)
                keep.append(k)
        keep = np.asarray(keep, np.int64)
        n_unique = len(keep)
        lens = (poff[keep + 1] - poff[keep]).astype(np.int64)
        poff2 = np.zeros(n_unique + 1, np.int64)
        poff2[1:] = np.cumsum(lens)
        pb2 = np.zeros(max(int(poff2[-1]), 1), np.uint8)
        for j, k in enumerate(keep.tolist()):
            pb2[poff2[j]:poff2[j + 1]] = pb[poff[k]:poff[k + 1]]
        pb, poff, tt_run = pb2, poff2, np.ascontiguousarray(tt[keep])
    else:
        tt_run = tt
    n_run = len(tt_run)
    # warm (also builds the oracle's trie outside the timed region)
    kv.match_blobs(tb, toff, pb, poff, tt_run, min(n_run, 256), 2 ** 31 - 1, 100, mode, singleton, cores)
    if n_warm > 0 and not cached:
        # the reference arm: bound the whole --steps K --warmup W run to ~3 minutes of matching by shrinking the sample (a
        # prefix of a uniform random sample is one) if a pilot pass says K + W passes would take longer
        kv.match_blobs(tb, toff, pb, poff, tt_run, n_run, 2 ** 31 - 1, 100, mode, singleton, cores)
        pilot = kv.last_match_seconds
        budget = 180.0
        if pilot * (n_passes + n_warm) > budget and n_run > 10000:
            n_run = max(10000, int(n_run * budget / (pilot * (n_passes + n_warm))))
            n = n_run
        n_warm -= 1
    for _ in range(n_warm):   # --warmup W: whole passes of the sample, untimed
        kv.match_blobs(tb, toff, pb, poff, tt_run, n_run, 2 ** 31 - 1, 100, mode, singleton, cores)
    # n_passes timed passes (5 for the cpu_baseline leg, --steps K for the reference arm), each repeated until it lasts >= 1 s
    # of wall time; the MEDIAN pass is reported
    passes, per_pass = [], []
    for _ in range(max(1, n_passes)):
        dt, reps = 0.0, 0
        while dt < 1.0 and reps < 64:
            out = kv.match_blobs(tb, toff, pb, poff, tt_run, n_run, 2 ** 31 - 1, 100, mode, singleton, cores)
            dt += kv.last_match_seconds   # the C++ matcher call alone (result marshalling to numpy excluded)
            reps += 1
        passes.append(dt / reps)
        per_pass.append(reps)
    dt = float(np.median(passes))
    stats = out.stats
    what = ("oracle filter-trie walk" if mode_name == "trie" else
            "literal TenantRouteMatcher.matchAll restatement, one call per topic (production shape)")
    res = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": "%s: %d topics (%s) against all %d routes; %s, std::thread x %d; median of %d passes of >= 1 s (%.3f s per "
                     "batch, spread %.3f-%.3f) = %.0f core-seconds per batch%s"
                     % (w.config, n, "the whole batch" if n == w.n_topics else "uniform random sample without replacement", len(kv), what, cores,
                        len(passes), dt, min(passes), max(passes), dt * cores,
                        ("; a (tenant, topic) result cache in front: %d distinct pairs matched, %d repeats served as lookups" % (n_unique, n - n_unique)) if cached else "")}
    return res, stats, n, float(poff[-1] - poff[0]) if not cached else None


def inverse_cpu_baseline(w, ids):
    """the oracle's TopicLevelTrie restatement (U/index/TopicLevelTrie.java:190-249 + RetainTopicIndex's selectors) over the same
    1M retained topics, every query filter, all host cores; also counts the trie nodes the lookups visit (V of SURVEY.md 8d)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    cores = os.cpu_count() or 1
    orc = O.TopicLevelIndex()
    tenants = w.tenants
    tl = w.topic_list()
    for i in range(w.n_topics):
        orc.add(tl[i], int(ids[i]), tenants[w.topic_tenant[i]])
    n = w.n_query_filters
    tb, toff = O.blob(tenants)
    counts = np.zeros(n, np.int64)
    vis = np.zeros(1, np.uint64)
    ft = np.ascontiguousarray(w.filter_tenant[:n])
    fo = np.ascontiguousarray(w.filter_off[:n + 1])
    passes = []
    for _ in range(5):
        dt, reps = 0.0, 0
        while dt < 1.0 and reps < 64:
            t0 = time.perf_counter()
            O.lib.orc_tli_match_batch(orc.h, tb.ctypes.data, toff, ft.ctypes.data, w.filters.ctypes.data, fo, n, cores, counts, vis.ctypes.data)
            dt += time.perf_counter() - t0
            reps += 1
        passes.append(dt / reps)
    dt = float(np.median(passes))
    return ({"value": n / dt, "unit": "filters/s", "cores": cores, "kind": "port",
             "sample": "C5: all %d query filters against the %d retained topics; oracle restatement of TopicLevelTrie.lookup with RetainTopicIndex's "
                       "selectors, std::thread x %d, unlimited results; median of 5 passes of >= 1 s (%.3f s per batch)" % (n, w.n_topics, cores, dt)},
            int(vis[0]), int(counts.sum()))


def main_inverse(args, rank, world, local):
    """BASELINE config C5: RetainStoreCoProc.match's index lookup (RS/RetainStoreCoProc.java:167-190 over
    RS/index/RetainTopicIndex.java:36-124) — 1M retained topics matched BY 100k wildcard SUBSCRIBE filters. The C-ABI of this
    direction takes host buffers only (bfq_rmatch), so `value` is the DEVICE time of its kernels, measured by the library with
    CUDA events on the call's stream from "inputs enqueued" to "ids expanded" (bfq_rresult_timings[4]), and `e2e` is the wall
    time of the whole call (H2D + kernels + D2H of the ids)."""
    import torch

    import bifromq_b200
    from bifromq_b200 import retain
    bifromq_b200.load_library()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local)
    w = make_workload(args, 0, 1)
    idx = retain.GpuTopicMatchIndex(local)
    tenants = w.tenants
    t0 = time.perf_counter()
    ids = idx.add_blobs(tenants, w.topics, w.topic_off, w.topic_tenant[:w.n_topics])
    idx.commit()
    t_build = time.perf_counter() - t0
    n = w.n_query_filters
    limit = np.full(n, args.retain_limit, np.int64) if args.retain_limit >= 0 else None
    f_blob = torch.from_numpy(np.ascontiguousarray(w.filters)).pin_memory().numpy()
    f_off = torch.from_numpy(np.ascontiguousarray(w.filter_off[:n + 1])).pin_memory().numpy()
    f_tt = torch.from_numpy(np.ascontiguousarray(w.filter_tenant[:n])).pin_memory().numpy()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        idx.match_blobs(tenants, f_blob, f_off, f_tt, limit)
    torch.cuda.synchronize(dev)
    sampler.begin()
    dev_ms, k_ms, wall, last = [], [], [], None
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        last = idx.match_blobs(tenants, f_blob, f_off, f_tt, limit)
        wall.append(time.perf_counter() - t0)
        dev_ms.append(last.timings_ms["device_all_kernels"])
        k_ms.append(last.timings_ms["device_rmatch_kernel"])
    sampler.end()
    clocks = sampler.stop() if rank == 0 else None
    idx.match_blobs(tenants, f_blob, f_off, f_tt, None)          # warm: the first unlimited call grows the id / range buffers
    unl = idx.match_blobs(tenants, f_blob, f_off, f_tt, None)
    if numa:
        try:
            os.sched_setaffinity(0, numa["previous"])
        except Exception:
            pass
    if rank != 0:
        return
    total_dev = float(sum(dev_ms)) / 1000.0
    value = n * args.steps / total_dev
    e2e = n * args.steps / float(sum(wall))
    fbytes = int(w.filter_off[n] - w.filter_off[0])
    line = {"metric": "retained-topic SUBSCRIBE filters matched/sec @1M retained topics (inverse path, BASELINE config C5)", "value": value,
            "unit": "filters/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1000.0 * total_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 (byte and integer work)", "data": "synthetic",
            "config": {"workload": workload_name(args, w), "retained_topics": w.n_topics, "filters_per_step": n, "tenants": w.n_tenants,
                       "limit": "RetainMessageMatchLimit = %d per filter" % args.retain_limit if args.retain_limit >= 0 else "unlimited",
                       "l2": "flushed between timed steps (256 MiB memset, untimed)", "build_s": round(t_build, 1),
                       "value_is": "device time of the call's kernels (CUDA events inside bfq_rmatch), inputs enqueued before the first event"},
            "e2e": {"value": e2e, "unit": "filters/s", "h2d_bytes_per_step": fbytes + 8 * (n + 1) + 4 * n + (8 * n if limit is not None else 0),
                    "d2h_bytes_per_step": 24 * n + 8 * int(len(last.ids)), "last_step_breakdown_ms": {k: round(v, 3) for k, v in last.timings_ms.items()}},
            "gpu_launches": 5 * args.steps, "ids_returned_per_step": int(len(last.ids)), "matches_total_per_step": int(last.totals.sum()),
            "unlimited": {"ids_returned": int(len(unl.ids)), "device_ms": unl.timings_ms["device_all_kernels"], "wall_ms": unl.timings_ms["total"],
                          "filters_per_s_e2e": n / (unl.timings_ms["total"] / 1000.0)},
            "tier2_filters_per_step": last.n_overflow_filters, "clocks": clocks}
    if not args.no_cpu_baseline:
        base, visited, matches = inverse_cpu_baseline(w, ids)
        # SURVEY.md 8(d), inverse path: per filter  len + 4 + 32 V + 8 ranges, V = topic-trie nodes the reference's lookup visits
        # (counted by the oracle), ranges = rank ranges the kernel emits (a '#' subtree or a final '+' level is ONE range)
        alg = fbytes + 4 * n + 32 * visited + 8 * last.n_ranges
        k = float(np.mean(k_ms))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        ach = alg / (k / 1000.0) / 1e9
        line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6650 GB/s",
                            "kernel": "rmatch_kernel (one warp per filter over the BFS-numbered topic trie)", "kernel_ms": k,
                            "alg_bytes_per_filter": alg / n, "alg_counters_per_filter": {"V": visited / n, "ranges": last.n_ranges / n},
                            "note": "V counted by the oracle over all %d filters; the reference's lookup visits EVERY child of a '+' level "
                                    "(TopicLevelTrie.java:200-249) while the kernel maps a '+' level to one id interval, so the achieved "
                                    "figure can exceed what the kernel really moves" % n,
                            "counts_check": {"oracle_matches": matches, "gpu_matches": int(unl.totals.sum()), "equal": matches == int(unl.totals.sum())}}
        line["cpu_baseline"] = base
    print(json.dumps(line))
    if args.dump_outputs:
        dump_inverse(args.dump_outputs, last)


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if args.config == "C5" and args.impl != "reference":
        return main_inverse(args, rank, world, local)
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.impl == "reference":
        # the reference's own algorithm (restated in C++, oracle/) on the host cores; rank 0 only
        if rank != 0:
            return
        w = make_workload(args, 0, 1)
        if args.config == "C5":
            base, visited, matches = inverse_cpu_baseline(w, np.arange(w.n_topics))
            v = base["value"]
            print(json.dumps({"metric": "retained-topic SUBSCRIBE filters matched/sec @1M retained topics (inverse path, BASELINE config C5)",
                              "value": v, "unit": "filters/s", "n_gpus": args.gpus, "steps": 5, "warmup": 1, "ms_per_step": 1000.0 * w.n_query_filters / v,
                              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 (byte and integer work)",
                              "data": "synthetic", "impl": "reference", "config": {"workload": workload_name(args, w),
                              "note": "C++ restatement of the Java reference, not the JVM (no JDK in the image)"}, "cpu_baseline": base,
                              "e2e": {"value": v, "unit": "filters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
            return
        # a step = one pass of the bounded sample (100k topics: seconds per pass on the box's cores); K timed, W untimed
        base, _, n, _ = run_cpu_baseline(w, args, "reference", n_passes=args.steps, n_warm=args.warmup)
        cached, _, _, _ = run_cpu_baseline(w, args, "reference", cached=True, n_passes=min(args.steps, 5))
        v = base["value"]
        line = {"metric": metric_name(args), "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1000.0 * n / v, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "u8/u32 (byte and integer work)", "data": "synthetic", "impl": "reference",
                "config": {"workload": workload_name(args, w), "note": "C++ restatement of the Java reference, not the JVM (no JDK in the image)"},
                "cpu_baseline": base, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "with_tenant_route_cache": {"value": cached["value"], "unit": UNIT, "sample": cached["sample"]},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    import bifromq_b200
    bifromq_b200.load_library()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local)

    t_gen = time.perf_counter()
    w = make_workload(args, rank, world)
    t_gen = time.perf_counter() - t_gen
    t_build = time.perf_counter()
    idx = bifromq_b200.GpuRouteIndex(local)
    idx.load(w.keys, w.key_off, w.vals, w.val_off)
    idx.commit()
    t_build = time.perf_counter() - t_build
    stats = idx.stats()
    tenants = idx.tenant_blob(w.tenants)   # marshalled once: the same tenant list serves every batch
    n = w.n_topics
    blob_bytes = int(w.topic_off[-1])

    # ---- device-resident batch (value) and pinned host batch (e2e)
    h_topics = torch.from_numpy(np.ascontiguousarray(w.topics[:max(blob_bytes, 1)])).pin_memory()
    h_off = torch.from_numpy(np.ascontiguousarray(w.topic_off)).pin_memory()
    h_tt = torch.from_numpy(np.ascontiguousarray(w.topic_tenant[:max(n, 1)])).pin_memory()
    d_topics, d_off, d_tt = h_topics.to(dev), h_off.to(dev), h_tt.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    stream = torch.cuda.current_stream(dev)

    nt = len(w.tenants)
    # the reference's defaults (Setting.MaxPersistentFanout = INT_MAX, MaxGroupFanout = 100), as in the CPU legs
    max_p, max_g = [args.max_pfanout] * nt, [args.max_gfanout] * nt

    def enqueue_device():
        """one step, enqueued without a host synchronisation (bfq_match_device_async): every count the later kernels need is
        read on the device; the result is waited for DEPTH steps later, so the host never idles the GPU between steps"""
        return idx.match_device(tenants, d_topics.data_ptr(), d_off.data_ptr(), d_tt.data_ptr(), n, max_p, max_g,
                                stream=stream.cuda_stream, wait=False)

    def step_e2e():
        r = idx.match(tenants, h_topics.numpy(), h_off.numpy(), h_tt.numpy(), max_p, max_g)
        d2h = 12 * n + 8 * len(r.ranges) + 12 * len(r.throttled)
        tm = r.timings_ms
        r.close()
        return d2h, tm

    from bifromq_b200 import dist as D
    xch = None
    if world > 1 and args.exchange != "none":
        xch = D.Exchange(local)   # NCCL communicator inside the library; the id travels over torch.distributed
        idx.set_option("tier0_ctas_per_sm", 6)   # one CTA slot per SM stays free for the exchange kernels of the previous step
    DEPTH = 3   # matches in flight (each on its own leased workspace)
    sampler = ClockSampler(",".join(str(i) for i in range(world)) if world > 1 else local)
    if rank == 0:
        sampler.start()
    kernel_ms, launches, n_ranges, n_overflow, n_distinct = [], 0, 0, 0, 0
    last = [None]
    gathered_info = {}

    def retire(res, keep=False, record=True):
        """wait for a step, note its counters, hand its workspace back (the timed loop must reuse the warm workspaces)"""
        nonlocal launches, n_ranges, n_overflow, n_distinct
        res.wait()
        if record:
            kernel_ms.append(res.tier0_ms)
            launches += res.n_launches
            n_ranges, n_overflow, n_distinct = res.n_ranges, res.n_overflow_topics, res.n_distinct_topics
        if keep:
            last[0] = res
        else:
            res.release()

    xs = torch.cuda.Stream(dev) if xch is not None else None   # the exchange runs on its own stream, AHEAD steps behind the matching
    pipe = {"pending": [], "gathered": None}
    AHEAD = max(1, args.exchange_lag)

    def pump(res_new, record):
        """N > 1, software-pipelined: the exchange of step i - AHEAD is issued after the matches of steps i - AHEAD + 1 .. i have
        been enqueued (no host sync in a match), so the exchange's one host synchronisation (the ranks' range counts size the
        payload all-gather) and its NCCL traffic overlap the next step's kernels. AHEAD = 1 by default; 2 (one more match
        queued while the host sits in that synchronisation) was measured equal at N = 2 — what the exchange adds to a step is
        device work (compaction of the sparse ranges + the all-gather), not a starved queue. The exchange (SURVEY.md 8e): every
        rank ends with every rank's per-topic counts (and ranges) — bfq_exchange_gather, NCCL inside the library.
        res_new = None drains one step."""
        if res_new is not None:
            pipe["pending"].append(res_new)
        if pipe["pending"] and (res_new is None or len(pipe["pending"]) > AHEAD):
            pend = pipe["pending"].pop(0)
            pend.wait()                      # waits for THAT match only (an event behind it), then reads its counters
            g = xch.gather(pend, ranges=args.exchange == "ranges", stream=xs.cuda_stream)
            gathered_info.update(topics=g.n_topics_total, ranges=g.n_ranges_total, bytes_received=g.bytes_received)
            if pipe["gathered"] is not None:
                pipe["gathered"].release()   # its gather finished before the synchronisation inside the gather just issued
            pipe["gathered"] = pend
            if record:
                kernel_ms.append(pend.tier0_ms)
        return (res_new.n_launches + 4) if (res_new is not None and record) else 0

    def drain(record):
        while pipe["pending"]:
            pump(None, record)

    inflight = []
    for _ in range(max(args.warmup, 3) + DEPTH):   # warm-up (also creates the workspaces the timed loop will reuse)
        if xch is not None:
            pump(enqueue_device(), False)
            continue
        inflight.append(enqueue_device())
        if len(inflight) >= DEPTH:
            retire(inflight.pop(0), record=False)
    while inflight:
        retire(inflight.pop(0), record=False)
    if xch is not None:
        drain(False)
        xs.synchronize()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler.begin()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize(dev)
    if xch is not None:
        # K steps back to back; timed as a whole (first match enqueued -> last exchange complete): the steps overlap by design.
        # No L2 flush here: every rank's index is far larger than L2 and each step streams new result buffers.
        t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin.record(stream)
        for i in range(args.steps):
            launches += pump(enqueue_device(), True)
        drain(True)
        t_end.record(xs)
        xs.synchronize()
        torch.cuda.synchronize(dev)
        step_total = t_begin.elapsed_time(t_end)
        ev = None
    else:
        for i in range(args.steps):
            flush.zero_()                     # L2 flush between timed iterations (untimed: outside the event pair)
            ev[i][0].record(stream)
            inflight.append(enqueue_device())
            ev[i][1].record(stream)
            if len(inflight) >= DEPTH:
                retire(inflight.pop(0))
        while inflight:
            r_ = inflight.pop(0)
            retire(r_, keep=not inflight)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    out = last[0] if xch is None else pipe["gathered"]
    if xch is not None:
        n_ranges, n_overflow, n_distinct = out.n_ranges, out.n_overflow_topics, out.n_distinct_topics
    step_ms = [a.elapsed_time(b) for a, b in ev] if ev is not None else [step_total / args.steps] * args.steps
    total_ms = float(sum(step_ms))
    # per-rank view (rank 0 prints it): where the max over ranks comes from
    per_rank, imbalance = None, None
    if world > 1:
        mine = {"rank": rank, "topics_per_step": n, "step_ms": total_ms / args.steps, "tier0_kernel_ms": float(np.mean(kernel_ms)),
                "routes": int(w.n_routes), "tenants": int(w.n_tenants)}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        imbalance = max(p["step_ms"] for p in per_rank) / (sum(p["step_ms"] for p in per_rank) / world)
    n_routes = int(torch.from_numpy(np.zeros(1)).sum()) if n == 0 else None
    # ---- e2e through the host-buffer call
    for _ in range(2):
        step_e2e()
    e2e_t, d2h_bytes, e2e_tm = [], 0, {}
    if world > 1:
        dist.barrier()
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        d2h_bytes, e2e_tm = step_e2e()
        e2e_t.append(time.perf_counter() - t0)
    sampler.end()
    clocks = sampler.stop() if rank == 0 else None
    if numa:   # the CPU baseline below uses every host core
        try:
            os.sched_setaffinity(0, numa["previous"])
        except Exception:
            pass
    e2e_total = float(sum(e2e_t))
    h2d_bytes = blob_bytes + 8 * (n + 1) + 4 * n

    # ---- whole-job numbers: MAX over ranks of the time, SUM over ranks of the topics
    from bifromq_b200 import dist as D
    total_ms_max, topics_all = D.aggregate(total_ms, n, dev)
    e2e_ms_max, _ = D.aggregate(e2e_total * 1000.0, n, dev)
    value = topics_all * args.steps / (total_ms_max / 1000.0)
    e2e_value = topics_all * args.steps / (e2e_ms_max / 1000.0)

    if rank == 0:
        # matched routes of one batch (for the fan-out routes/s figure)
        res = idx.match(tenants, h_topics.numpy(), h_off.numpy(), h_tt.numpy(), max_p, max_g)
        routes_per_batch = int(res.route_count.astype(np.int64).sum())
        ranges_per_batch = int(res.span_count.astype(np.int64).sum())   # matched filters with >= 1 route, over every topic
        res.close()
        stats = idx.stats()
        cpu_base, roof = None, None
        k_ms = float(np.mean(kernel_ms))
        if not args.no_cpu_baseline and world == 1:   # rank 0 at N = 1 only (at N > 1 `w` is one shard)
            cpu_base, st, ns, sample_topic_bytes = run_cpu_baseline(w, args, "trie")
            roof = make_roofline(sample_topic_bytes, st, ns, n, k_ms, ranges_per_batch, routes_per_batch, {"config": args.config})
        line = {"metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "u8/u32 (byte and integer work)", "data": "synthetic",
                "config": {"workload": workload_name(args, w), "routes_per_gpu": w.n_routes, "filters_per_gpu": w.n_filters,
                           "tenants_per_gpu": w.n_tenants, "topics_per_step_per_gpu": n, "topics_per_step_all_gpus": int(topics_all),
                           "parallelism": "tenant-sharded x%d" % world,
                           "l2": ("flushed between timed steps (256 MiB memset, untimed); index %.2f GB >> L2" if xch is None else
                                  "not flushed (the pipelined steps overlap); inputs larger than L2: index %.2f GB per rank") % (stats["device_bytes"] / 1e9),
                           "caps": "MaxPersistentFanout=%s, MaxGroupFanout=%s (reference defaults: INT_MAX, 100)" % (
                               "INT_MAX" if args.max_pfanout == 2 ** 31 - 1 else args.max_pfanout, "INT_MAX" if args.max_gfanout == 2 ** 31 - 1 else args.max_gfanout),
                           "order": "inside the timed region: duplicate (tenant, topic) pairs are found with a device hash table and answered from their "
                                    "first occurrence (%d of %d topics distinct), the distinct ones are matched in locality order (own counting sort)" % (n_distinct, n),
                           "pipelining": ("steps are enqueued without host synchronisation (bfq_match_device_async), %d in flight; timed per step with CUDA events on the launching stream" % DEPTH) if xch is None else
                                         ("software pipeline: the matches of steps i-%d+1 .. i are enqueued (no host sync) before the exchange of step i-%d (own stream, one host sync) is issued; the K steps are timed as a whole with CUDA events (first match -> last exchange complete); no L2 flush (index >> L2)" % (AHEAD, AHEAD)),
                           "host": ("rank pinned to NUMA node %d of its GPU (%d cpus) for the GPU legs" % (numa["node"], numa["cpus"])) if numa
                                   else "no NUMA pinning (topology not exposed or single node)",
                           "gen_s": round(t_gen, 1), "build_s": round(t_build, 1)},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "last_step_breakdown_ms": {k: round(v, 3) for k, v in e2e_tm.items()}},
                "gpu_launches": launches, "gpu_launches_note": "own kernels per step: order prep/scan/scatter + tier 0 + tier 1 + followers + caps (2)", "routes_per_s": routes_per_batch * world * args.steps / (total_ms_max / 1000.0),
                "tier0_kernel_ms": float(np.mean(kernel_ms)), "step_ms_min_median_max": [float(np.min(step_ms)), float(np.median(step_ms)), float(np.max(step_ms))],
                "ranges_per_step": n_ranges, "tier2_topics_per_step": n_overflow, "index": stats, "clocks": clocks}
        if world > 1:
            line["per_rank"] = per_rank
            line["load_imbalance_max_over_mean"] = imbalance
            line["exchange"] = ({"what": "inside the timed step: bfq_exchange_gather (NCCL all-gather inside the library, one host sync): every rank ends with "
                                         "every rank's per-topic route counts%s" % (", range counts and dense {first rank, count} ranges" if args.exchange == "ranges" else ""),
                                 "topics_gathered": gathered_info.get("topics"), "ranges_gathered": gathered_info.get("ranges"),
                                 "bytes_received_per_rank": gathered_info.get("bytes_received")} if xch is not None else
                                {"what": "none (--exchange none)"})
            line["config"]["sharding"] = ("ONE %s filter set: tenant -> rank by fnv1a64(tenantId) mod %d%s; a %d-topic batch (%s) split by owner" % (
                args.config, world, "" if args.no_replicate_hot else "; tenants above 1/(4 x ranks) of the batch are hosted by every rank, their topics dealt round-robin",
                int(topics_all), "%d x the config's batch: weak scaling" % world if args.scaling == "weak" else "the config's batch: strong scaling"))
        if roof:
            line["roofline"] = roof
        if cpu_base:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line))
        if args.dump_outputs:
            dump_forward(args.dump_outputs, out, dev, stream.cuda_stream)
    out.release()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def workload_name(args, w):
    names = {"C1": "C1: 1 tenant, 10k exact filters, 1k topics", "C2": "C2: 1 tenant, 1M filters (50% '+'), 100k-topic batch",
             "C3": "C3: 1000 tenants x 10k filters mixed +/#, 1M-topic batch",
             "C4": "C4: 10M filters over 1000 tenants (Zipf sizes, Zipf fan-out and topic popularity), 1M-topic batch",
             "C5": "C5: retain-store inverse match, 1M retained topics vs 100k wildcard SUBSCRIBE filters"}
    s = names[args.config]
    if args.scale != 1.0:
        s += " [scale %.4g — NOT a valid bench size]" % args.scale
    return s


if __name__ == "__main__":
    main()
