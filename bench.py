#!/usr/bin/env python3
"""bench.py — messages/s of the message-scan metric path on N B200s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config C1|C2|C3|C4] [--mode fused|hll|counters|alive]
  python bench.py --impl reference --gpus N --steps K ...   the reference's CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR    also writes the state the K timed steps computed as DIR/<name>.npy

Workloads (BASELINE.json configs; SURVEY.md §8 d) — the default at every N is C1, per-GPU work fixed (weak scaling):
  C1  64 partitions, 1e8 messages per GPU, 256 B mean value, 16-byte keys, 1e7 distinct keys per GPU, 1 % null keys,
      NO tombstones (SURVEY.md §8 d's "0 % variant for the in-stream-HLL case": on a tombstone-free topic the in-stream
      sketch of the default mode estimates exactly what the reference's -c BitSet counts, so both arms compute the same
      alive-key answer; --tombstones 500 gives the 5 % variant, --mode fused the exact table).  The configuration the
      metric is quoted on.
  C2  the alive-key path: 64 partitions, 1e9 messages per GPU, 1e7 distinct keys, every record keyed (mode alive).
  C3  the 8-GPU job as each of its ranks sees it: 256 partitions sharded p mod 8, 4e9 messages in all = 5e8 per rank,
      1 KiB mean value.  With N < 8 GPUs the first N of the 8 shards are scanned (per-GPU work is C3's at every N).
  C4  value-size sweep 64 B .. 64 KiB on the C1 shape (value bytes are never read — src/metric.rs:235 — so the kernel
      time does not depend on them; the logical topic GB/s grows linearly).  The JSON line carries the sweep.

Modes:
  hll       counters + histograms + extrema + FNV32 per key + in-stream HLL sketch of every (key, value) record — north_star's
            fused scan kernel.  The sketch equals the reference's alive-key count (within its standard error) on
            tombstone-free topics only; the default workload is one.  The headline.
  fused     the same with EXACT alive keys instead (seen cache + open-addressed last-writer table: the reference's -c
            answer on any topic, src/metric.rs:288-305) + HLL over the resolved alive set at finalize.
  alive     fused without the HLL extension (exactly the reference with -c).
  counters  MessageMetrics only (the reference without -c): no key bytes are read.

A "step" is one pass of the hot path over one batch: the fused scan kernel over the rank's shard resident in HBM, added to
the running topic state.  The K timed steps form one K-batch topic: state reset at the start, and — as the reference reads
its results once, after the poll loop (src/main.rs:117-170) — ONE merge (N > 1: one NCCL all-reduce) and ONE finalize
(state to host) at the end, all inside the timed region.  Inputs are >= 3.6 GB per GPU (>> 126 MB L2), so every step
streams from HBM.  `value` = all ranks' records / max-over-ranks device time (CUDA events on the scan stream).
`e2e` = the same metric through the C-ABI host entry point (kta_push_batch_host) with the batch in pinned HOST memory:
host->device copies every step and the state read-back (finalize) every step are inside the timed region.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "messages/sec scanned (fused metric scan)"
UNIT = "msg/s"
DEFAULT_MODE = "hll"

CONFIGS = {
    # partitions, records/GPU, value mean, distinct keys/GPU, null keys /10k, tombstones /10k, virtual world, mode
    "C1": dict(partitions=64, n=100_000_000, value_mean=256, distinct_keys=10_000_000, nulls=100, tombstones=0, shard_world=0, mode=None),
    "C2": dict(partitions=64, n=1_000_000_000, value_mean=256, distinct_keys=10_000_000, nulls=0, tombstones=500, shard_world=0, mode="alive"),
    # C3 is named "partition-sharded scan + NCCL histogram/HLL merge": the in-stream sketch mode.  (The exact table keeps 31
    # bits of seq; a sharded -c job needs absolute sequence numbers, and this topic has 4e9 of them.)
    "C3": dict(partitions=256, n=500_000_000, value_mean=1024, distinct_keys=10_000_000, nulls=100, tombstones=500, shard_world=8, mode="hll"),
    "C4": dict(partitions=64, n=100_000_000, value_mean=1024, distinct_keys=10_000_000, nulls=100, tombstones=0, shard_world=0, mode=None),
}
C4_VALUE_MEANS = [64, 256, 1024, 4096, 16384, 65536]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C1", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default=None, choices=["fused", "hll", "counters", "alive"])
    # overrides of the named configuration (shape studies; the workload string says what ran)
    ap.add_argument("--n", type=int, default=None, help="records per GPU")
    ap.add_argument("--partitions", type=int, default=None)
    ap.add_argument("--value-mean", type=int, default=None)
    ap.add_argument("--distinct-keys", type=int, default=None, help="distinct keys per GPU")
    ap.add_argument("--tombstones", type=int, default=None, help="tombstones per 10 000 records")
    ap.add_argument("--null-keys", type=int, default=None, help="null keys per 10 000 records")
    ap.add_argument("--shard-world", type=int, default=None, help="scan shard r of a topic sharded p mod W (W >= --gpus)")
    ap.add_argument("--run-len", type=int, default=1)
    ap.add_argument("--hll", type=int, default=14)
    ap.add_argument("--alive-table-kib", type=int, default=0, help="initial alive-key table size (0 = library default, 128 MiB)")
    ap.add_argument("--key-mode", type=int, default=0, help="0 = 16-byte binary keys, 1 = ASCII key-<id>, 2 = variable 0..40 B")
    ap.add_argument("--zipf-keys", action="store_true", help="stress case: log-uniform (Zipf s = 1 staircase) key ids")
    ap.add_argument("--geometric-values", action="store_true", help="stress case: geometric-tailed value lengths")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the post-run parity check of the (merged) state")
    ap.add_argument("--cpu-sample", type=int, default=0, help="records in the CPU baseline sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state they computed (what a caller reads back) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    c = CONFIGS[a.config]
    for k_arg, k_cfg in (("n", "n"), ("partitions", "partitions"), ("value_mean", "value_mean"), ("distinct_keys", "distinct_keys"),
                         ("tombstones", "tombstones"), ("null_keys", "nulls"), ("shard_world", "shard_world")):
        if getattr(a, k_arg) is None:
            setattr(a, k_arg, c[k_cfg])
    if a.mode is None:
        a.mode = c["mode"] or DEFAULT_MODE
    return a


MODE_TEXT = {"fused": "counters+histograms+FNV32+exact alive keys (seen cache + last-writer table: -c) +HLL p%d over the alive set",
             "alive": "counters+histograms+FNV32+exact alive keys (seen cache + last-writer table: -c)",
             "hll": "counters+histograms+FNV32+in-stream HLL p%d of every (key, value) record", "counters": "counters+histograms (no -c)"}
KERNEL = {"fused": "kta::scan_kernel<MODE_EXACT>", "alive": "kta::scan_kernel<MODE_EXACT>", "hll": "kta::scan_kernel<MODE_HLL>",
          "counters": "kta::scan_kernel<MODE_COUNTERS>"}


def virtual_world(a, world):
    return max(world, a.shard_world or 0)


def make_spec(a, world):
    from kafka_topic_analyzer_b200 import synth
    vw = virtual_world(a, world)
    return synth.make_spec(a.n * vw, a.partitions, run_len=a.run_len, distinct_keys=a.distinct_keys * vw, value_mean=a.value_mean,
                           key_mode=a.key_mode, zipf_keys=a.zipf_keys, geometric_values=a.geometric_values,
                           tombstone_per_10k=a.tombstones, null_key_per_10k=a.null_keys)


def config_dict(a, world):
    """Names the workload; a pure function of the arguments, identical for both arms (--impl ours / reference)."""
    keys = {0: "16 B", 1: "ASCII key-<id>", 2: "variable 0..40 B"}[a.key_mode & 0xFF] + " keys"
    if a.zipf_keys:
        keys += " (log-uniform ids)"
    vw = virtual_world(a, world)
    mode_text = MODE_TEXT[a.mode] % a.hll if "%d" in MODE_TEXT[a.mode] else MODE_TEXT[a.mode]
    return {
        "workload": "%s: %d partitions%s, %.0e msgs/GPU x %d GPU, %d B mean value%s, %s, %.0e distinct keys/GPU, %.1f %% null keys, "
                    "%.1f %% tombstones, run_len=%d, mode=%s (%s)" %
                    (a.config, a.partitions, " sharded p mod %d" % vw if vw > 1 else "", a.n, world, a.value_mean,
                     " (geometric tail)" if a.geometric_values else "", keys, a.distinct_keys, a.null_keys / 100, a.tombstones / 100,
                     a.run_len, a.mode, mode_text),
        "config": a.config, "mode": a.mode, "partitions": a.partitions, "records_per_gpu": a.n, "value_mean": a.value_mean,
        "distinct_keys_per_gpu": a.distinct_keys, "shard_world": vw,
        "step": "one scan of the rank's %.0e-record batch into the running topic state; the K timed steps are one K-batch topic "
                "closed by one merge (N>1) and one finalize inside the timed region" % a.n,
        "l2": "inputs %.1f GB/GPU, larger than L2 (126 MB): no flush needed" % (a.n * 36 / 1e9),
        "key_tile_base": "128-record tile offsets column supplied with the batch (feeder-side prefix sum, 0.06 B/record; the "
                         "library derives it with one extra pass when absent)",
    }


class ClockSampler:
    """nvidia-smi clocks + throttle reasons around the timed region.  The poller needs ~0.1 s to come up and samples every
    20 ms, while 20 steps of a 0.65 ms scan are over in 13 ms: so it is started BEFORE the warm-up steps (same kernels, back
    to back with the timed ones), the caller waits for its first line, and stop() reports the samples taken from then to the
    end of the timed region (`samples`) and how many of them fell inside the timed region itself (`samples_in_region`)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.rows, self.proc, self.load_from = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=2.0):
        """blocks until the poller has delivered a line (or `timeout` s); everything from now on counts as under load"""
        t_end = time.perf_counter() + timeout
        while self.proc and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.005)
        self.load_from = time.perf_counter()

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        lo = self.load_from if self.load_from is not None else float("-inf")
        hi = t1 + 0.025 if t1 is not None else float("inf")      # a sample describes the 20 ms before it
        rows = [r for (t, r) in list(self.rows) if lo <= t <= hi and len(r) >= 9] or [r for (_, r) in list(self.rows) if len(r) >= 9]
        inside = sum(1 for (t, r) in list(self.rows) if t0 is not None and t1 is not None and t0 <= t <= t1 + 0.025 and len(r) >= 9)
        sm = sorted(int(r[1]) for r in rows if r[1].isdigit())
        mx = [int(r[2]) for r in rows if r[2].isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_region": inside}


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (oracle port; the Rust original cannot be
# built here).  bench.py is one of the few places allowed to execute oracle/.  It never loads libkta_gpu.so:
# the topic comes from the host-only generator library (libkta_synth.so).
# --------------------------------------------------------------------------------------------------
def host_sample(a, world, sample):
    """The first `sample` records of rank 0's shard of the workload (same spec as the GPU arm: same key space)."""
    from kafka_topic_analyzer_b200 import synth
    spec = make_spec(a, world)
    return synth.fill_host(spec, rank=0, world=virtual_world(a, world), count=min(sample, a.n))


def cpu_reference_rate(topic, threads, count_alive_keys):
    """records/s of the C restatement of src/metric.rs:206-305 over `topic`.
    threads == 1 is the reference as designed (one consumer thread, src/kafka.rs:92-135); threads > 1 runs
    one independent handler set per thread over an equal slice (what a partition-sharded rewrite could do)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    import numpy as np
    n = topic.n
    kl = np.maximum(topic.key_len.astype(np.int64), 0)
    koff = np.concatenate([[0], np.cumsum(kl)])
    bounds = [n * i // threads for i in range(threads + 1)]
    oracles = [Oracle(count_alive_keys=count_alive_keys, no_hist=True) for _ in range(threads)]

    def work(i):
        lo, hi = bounds[i], bounds[i + 1]
        oracles[i].handle_batch(topic.partition[lo:hi], topic.ts_ms[lo:hi], topic.key_len[lo:hi], topic.value_len[lo:hi],
                                topic.key_bytes[int(koff[lo]):int(koff[hi])])

    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        [t.start() for t in ts]
        [t.join() for t in ts]
    return n / (time.perf_counter() - t0)


def cpu_baseline_text(a, sample, alive):
    return ("first %d records of rank 0's batch of this workload per step (same topic spec, same %d-key space; fresh handlers "
            "each step); C restatement of src/metric.rs:206-305 + src/fnv32.rs (%s); 1 thread because the reference is "
            "single-threaded by construction (src/kafka.rs:92-135); Rust original not buildable here (no toolchain)"
            % (sample, a.distinct_keys, "MessageMetrics + LogCompactionInMemoryMetrics (-c)" if alive else "MessageMetrics only"))


def run_reference(a):
    """--impl reference: the reference's own CPU path.  It is single-threaded by construction (one consumer
    thread drives both handlers, src/kafka.rs:92-135; the alive-key BitSet is one global structure,
    src/metric.rs:262-264), so "all the host threads it can use" is 1; a partition-sharded multi-thread
    figure for the counter handler alone is added for context."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    alive = a.mode != "counters"
    probe = host_sample(a, a.gpus, 1_000_000)
    rate = cpu_reference_rate(probe, 1, alive)
    # size the per-step sample so that warmup + steps take about two minutes in total
    sample = a.cpu_sample or int(min(20_000_000, max(1_000_000, rate * 120.0 / max(1, a.steps + a.warmup))))
    topic = host_sample(a, a.gpus, sample)
    sample = topic.n
    for _ in range(max(0, a.warmup - 1)):
        cpu_reference_rate(topic, 1, alive)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        cpu_reference_rate(topic, 1, alive)
    total = time.perf_counter() - t0
    value = sample * a.steps / total
    sharded = cpu_reference_rate(topic, cores, False)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * total / max(1, a.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_dict(a, a.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": cpu_baseline_text(a, sample, alive),
                         "counters_only_sharded_value": sharded, "counters_only_sharded_cores": cores},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
def make_engine(kta, a, mode, device, shard=None):
    """shard = (rank, world) for a partition-sharded scan: the kernel carves counter columns for the owned partitions only"""
    return kta.KtaEngine(a.partitions, count_alive_keys=mode in ("fused", "alive"),
                         hll_precision=a.hll if mode in ("fused", "hll") else 0, device=device, alive_table_kib=a.alive_table_kib,
                         shard=shard if shard and shard[1] > 1 else None)


def scan_topic(eng, topic, mode):
    keys = mode != "counters"
    eng.scan_batch_device(topic.partition, topic.ts_ms, topic.key_len, topic.value_len,
                          key_bytes=topic.key_bytes if keys else None, key_bytes_len=topic.key_bytes_len if keys else 0,
                          key_tile_base=topic.key_tile_base if keys else None, seq=topic.seq)


def state_of(eng, P, mode):
    """Everything the report reads (src/main.rs:130-170) plus the extensions, as one comparable structure."""
    mm = eng.message_metrics
    s = {"counters": [[eng.counter(i, p) for i in range(7)] for p in range(P)],
         "khist": [eng.hist(0, p).tolist() for p in range(P)], "vhist": [eng.hist(1, p).tolist() for p in range(P)],
         "globals": [mm.smallest_message(), mm.largest_message(), mm.overall_size(), mm.overall_count(), mm.latest_message(),
                     list(mm.earliest_message())]}
    if mode in ("fused", "alive"):
        s["alive_keys"] = eng.alive_keys()
    if mode in ("fused", "hll"):
        s["hll"] = eng.hll_registers().tolist()
    return s


DUMP_PARTITIONS = 4096   # per-partition outputs of larger topics are dumped for a seeded sample of this many partitions


def dump_outputs(eng, P, mode, out_dir, prefix=""):
    """Writes the finalized state of the timed path, everything a caller reads back from it, as out_dir/<prefix><name>.npy,
    so that two builds can be compared output for output on the same seeded topic.  Integer metrics are stored as float64
    (exact below 2^53), the HLL registers as float32.  A topic with more than DUMP_PARTITIONS partitions is represented by
    a fixed, seeded sample of them (partitions.npy names which), which keeps the files far below 64 MB."""
    import numpy as np
    parts = np.arange(P)
    if P > DUMP_PARTITIONS:
        parts = np.sort(np.random.default_rng(0).choice(P, DUMP_PARTITIONS, replace=False))
    out = {"partitions": parts,
           "counters": [[eng.counter(i, int(p)) for i in range(7)] for p in parts],
           "key_size_hist": [eng.hist(0, int(p)) for p in parts],
           "value_size_hist": [eng.hist(1, int(p)) for p in parts],
           "globals": [eng.global_(i) for i in range(4)],
           "timestamps": list(eng.timestamps())}
    if mode in ("fused", "alive"):
        out["alive_keys"] = [eng.alive_keys()]
    if mode in ("fused", "hll"):
        out["hll_registers"] = eng.hll_registers()
        out["alive_keys_hll"] = [eng.alive_keys_hll()]
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"),
                np.asarray(v, dtype=np.float32 if name == "hll_registers" else np.float64))


def run_ours(a):
    import torch
    import torch.distributed as dist
    import kafka_topic_analyzer_b200 as kta
    from kafka_topic_analyzer_b200 import synth
    from kafka_topic_analyzer_b200.distributed import allreduce_merge

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE %d" % (a.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    ctx = dict(torch=torch, dist=dist, kta=kta, synth=synth, merge=allreduce_merge, rank=rank, world=world, local=local, dev=dev,
               barrier=barrier)
    if a.config == "C4":
        line = run_sweep(a, ctx)
    else:
        line = measure(a, ctx, full=True)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def measure(a, ctx, full, dump_prefix=""):
    torch, dist, kta, synth, allreduce_merge = ctx["torch"], ctx["dist"], ctx["kta"], ctx["synth"], ctx["merge"]
    rank, world, local, dev, barrier = ctx["rank"], ctx["world"], ctx["local"], ctx["dev"], ctx["barrier"]
    # ---- the rank's shard of the topic, generated in HBM ----
    P = a.partitions
    vw = virtual_world(a, world)
    spec = make_spec(a, world)
    n_all = a.n * world                      # records scanned per step by all ranks together
    exact = a.mode in ("fused", "alive")
    topic = synth.DeviceTopic(spec, rank=rank, world=vw, device=local, with_seq=(exact and vw > 1))
    n = topic.n
    assert n == a.n
    alg_bytes = 20 * n + (topic.key_bytes_len if a.mode != "counters" else 0)   # SURVEY.md §8(d)

    # a sharded handle carves counter columns for its own partitions only: worth its few instructions per record when the
    # topic has many partitions (C3: 256 -> 32 columns per rank), not for C1's 64
    eng = make_engine(kta, a, a.mode, local, shard=(rank, vw) if a.partitions > 64 else None)
    stream = torch.cuda.current_stream(dev)
    eng.set_stream(stream.cuda_stream)

    def topic_pass(steps):
        """one K-batch topic: reset, K scans, one merge, one finalize"""
        eng.reset()
        for _ in range(steps):
            scan_topic(eng, topic, a.mode)
        if world > 1:
            allreduce_merge(eng)
        eng.finalize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first()          # the poller is up before the warm-up steps: they and the timed steps are its "under load"
    topic_pass(max(1, a.warmup))
    barrier()
    eng.set_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_region0 = time.perf_counter()
    e0.record(stream)
    topic_pass(a.steps)
    e1.record(stream)
    launches = eng.stats()[0]
    barrier()
    clocks = sampler.stop(t_region0, time.perf_counter()) if rank == 0 else None
    ms = e0.elapsed_time(e1)
    kern_ms, kern_n = eng.scan_time_ms()
    eng.set_timing(False)
    kavg = kern_ms / max(1, kern_n)
    t = torch.tensor([ms, kavg, -kavg], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, kern_max_ms, kern_min_ms = t[0].item(), t[1].item(), -t[2].item()
    value = n_all * a.steps / (ms / 1e3)
    # sanity on the timed topic itself: K batches were counted (on every rank after the merge)
    assert eng.message_metrics.overall_count() == n_all * a.steps, (eng.message_metrics.overall_count(), n_all * a.steps)
    if a.dump_outputs and rank == 0:
        dump_outputs(eng, P, a.mode, a.dump_outputs, dump_prefix)
    table = eng.alive_table_stats() if exact else None

    merge_ms = None
    if world > 1:
        # the merge alone (export kernel + ONE NCCL all-reduce + import kernel), 20 back-to-back calls
        barrier()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record(stream)
        for _ in range(20):
            allreduce_merge(eng, counters_only=True)
        m1.record(stream)
        barrier()
        mt = torch.tensor([m0.elapsed_time(m1) / 20], dtype=torch.float64, device=dev)
        dist.all_reduce(mt, op=dist.ReduceOp.MAX)
        merge_ms = mt.item()

    verified = None
    if full and not a.no_verify:
        verified = verify(a, ctx, eng, topic, spec, vw)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (kern_max_ms / 1e3) / 1e9
    traffic = None
    try:
        if a.config == "C1":      # the committed ncu captures are of the C1 shape
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get({"fused": "alive"}.get(a.mode, a.mode))
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": config_dict(a, world),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": KERNEL[a.mode], "kernel_ms": kern_max_ms, "kernel_ms_min_rank": kern_min_ms,
                     "algorithmic_bytes_per_launch": alg_bytes, "mean_key_bytes": topic.key_bytes_len / n,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650"},
        "logical_topic_gb_s": value * (topic.key_bytes_len / n + a.value_mean) / 1e9,
        "gpu_launches": launches, "clocks": clocks,
    }
    if table:
        line["alive_table"] = {"slots": table[0], "bytes": table[0] * 8, "occupied": table[1], "grows": table[2], "reruns": table[3]}
    if merge_ms is not None:
        line["merge_ms"] = merge_ms
    if verified is not None:
        line["verified"] = verified
    if not full:
        eng.close()
        return line

    if rank == 0 and world == 1 and not a.no_extra:
        line["extra_modes"] = extra_modes(a, topic, kta, torch, dev, peak)

    # ---- e2e: same metric through the host entry point, inputs in pinned host memory ----
    if not a.no_e2e:
        e2e_steps = a.steps
        cols = {}
        for name in ("partition", "ts_ms", "key_len", "value_len", "key_tile_base"):
            src = getattr(topic, name)
            cols[name] = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
            cols[name].copy_(src)
        seq_host = None
        if topic.seq is not None:
            seq_host = torch.empty(topic.seq.shape, dtype=topic.seq.dtype, pin_memory=True)
            seq_host.copy_(topic.seq)
        kb = torch.empty(topic.key_bytes_len, dtype=torch.uint8, pin_memory=True)
        kb.copy_(topic.key_bytes[: topic.key_bytes_len])
        use_keys = a.mode != "counters"
        h2d = sum(cols[c].numel() * cols[c].element_size() for c in ("partition", "ts_ms", "key_len", "value_len"))
        if use_keys:
            h2d += kb.numel() + cols["key_tile_base"].numel() * 8
        if seq_host is not None:
            h2d += seq_host.numel() * 8
        d2h = (P * 67 + 1) * 8 + 32 + ((1 << a.hll) * 4 if a.mode in ("fused", "hll") else 0) + (8 if exact else 0)

        def e2e_step():
            eng.reset()
            eng.push_batch_host(cols["partition"], cols["ts_ms"], cols["key_len"], cols["value_len"],
                                kb if use_keys else None, cols["key_tile_base"] if use_keys else None, seq=seq_host)
            if world > 1:
                allreduce_merge(eng)
            eng.finalize()

        e2e_step()
        barrier()
        sampler2 = ClockSampler(local)
        if rank == 0:
            sampler2.start()
            sampler2.wait_first()
        barrier()
        e0.record(stream)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        if rank == 0:
            line["clocks_e2e"] = sampler2.stop(t0, t0 + wall)
        t = torch.tensor([max(e0.elapsed_time(e1) / 1e3, wall)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert eng.message_metrics.overall_count() == n_all
        line["e2e"] = {"value": n_all * e2e_steps / t.item(), "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                       "path": "per step: kta_reset + kta_push_batch_host (pinned host SoA -> chunked cudaMemcpyAsync -> scan) "
                               "[+ NCCL merge] + kta_finalize (state to host)"}
    eng.close()

    # ---- cpu_baseline: the oracle port on the GPU box's host cores (rank 0, N=1 only) ----
    if rank == 0 and world == 1 and not a.no_cpu:
        alive = a.mode != "counters"
        m = min(n, a.cpu_sample or 20_000_000)
        host = synth.HostTopic(topic.partition[:m].cpu().numpy(), None, topic.ts_ms[:m].cpu().numpy(),
                               topic.key_len[:m].cpu().numpy(), topic.value_len[:m].cpu().numpy(), None,
                               topic.key_bytes[: topic.key_bytes_len].cpu().numpy(), None)
        rate1 = cpu_reference_rate(host, 1, alive)
        cores = os.cpu_count() or 1
        rateN = cpu_reference_rate(host, cores, False)   # counter handler only, equal slices
        line["cpu_baseline"] = {"value": rate1, "unit": UNIT, "cores": 1, "kind": "port", "sample": cpu_baseline_text(a, m, alive),
                                "counters_only_sharded_value": rateN, "counters_only_sharded_cores": cores}
        if not a.no_extra:
            line["extra"] = {"e2e_push": e2e_push(a)}
    return line


def verify(a, ctx, eng, topic, spec, vw):
    """Parity of the measured path outside the timed region: one pass (reset, scan, merge, finalize) must give
    (i) the closed-form shares of the generator and the counter identities of src/metric.rs, and (ii) at N > 1, on every
    rank, bit for bit the state that ONE engine on rank 0 reaches by scanning all N shards itself without any merge —
    every counter, histogram bucket, extremum, the exact alive-key count and every HLL register."""
    torch, dist, kta, synth, allreduce_merge = ctx["torch"], ctx["dist"], ctx["kta"], ctx["synth"], ctx["merge"]
    rank, world, local, dev = ctx["rank"], ctx["world"], ctx["local"], ctx["dev"]
    P = a.partitions
    eng.reset()
    scan_topic(eng, topic, a.mode)
    if world > 1:
        allreduce_merge(eng)
    eng.finalize()
    got = state_of(eng, P, a.mode)
    owned = set(p for p in range(P) if p % vw < world)
    per_part = a.n * vw // P
    for p in range(P):
        tot, tomb, alive, knull, knn, ksum, vsum = got["counters"][p]
        assert tot == (per_part if p in owned else 0), ("total", p, tot)
        assert knull + knn == tot == alive + tomb, ("identities", p)
        assert sum(got["khist"][p]) == knn and sum(got["vhist"][p]) == alive, ("histogram sums", p)
        if a.key_mode == 0:
            assert ksum == 16 * knn
        if not a.geometric_values:
            assert (a.value_mean // 2) * alive <= vsum <= (a.value_mean // 2 + a.value_mean) * alive
    assert got["globals"][3] == a.n * world
    out = {"closed_form_shares_and_identities": True}
    if world == 1 and a.mode == "hll" and a.tombstones == 0:
        # tombstone-free topic: the sketch must estimate the EXACT alive-key count (the reference's -c answer, computed here
        # by the exact engine over the same topic) within 4 sigma, sigma = 1.04 / sqrt(2^p)
        b = argparse.Namespace(**vars(a))
        ex = make_engine(kta, b, "alive", local)
        ex.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        scan_topic(ex, topic, "alive")
        ex.finalize()
        exact_keys = ex.alive_keys()
        ex.close()
        est = eng.alive_keys_hll()
        assert abs(est - exact_keys) <= 4 * 1.04 / (2 ** (a.hll / 2)) * exact_keys, (est, exact_keys)
        out["hll_estimate"] = est
        out["exact_alive_keys"] = exact_keys
        out["hll_within_4_sigma_of_exact"] = True
    if world > 1:
        ref_state = None
        if rank == 0:
            ref = make_engine(kta, a, a.mode, local)
            ref.set_stream(torch.cuda.current_stream(dev).cuda_stream)
            exact = a.mode in ("fused", "alive")
            for r in range(world):
                t_r = topic if r == rank else synth.DeviceTopic(spec, rank=r, world=vw, device=local, with_seq=exact)
                scan_topic(ref, t_r, a.mode)
                ref.sync()
                del t_r
            ref.finalize()
            ref_state = state_of(ref, P, a.mode)
            ref.close()
        box = [ref_state]
        dist.broadcast_object_list(box, src=0)
        same = box[0] == got
        flags = torch.tensor([1 if same else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if not same:
            diff = [k for k in got if got[k] != box[0][k]]
            raise AssertionError("rank %d: merged state differs from the single-engine scan in %s" % (rank, diff))
        assert flags.item() == 1
        out["merged_state_equals_single_engine_scan_on_every_rank"] = True
    return out


def run_sweep(a, ctx):
    """C4: the value-size sweep.  One line; `value` is the 1 KiB point (north_star's target shape)."""
    points, head = [], None
    for vm in C4_VALUE_MEANS:
        b = argparse.Namespace(**vars(a))
        b.value_mean = vm
        line = measure(b, ctx, full=False, dump_prefix="value_mean_%d_" % vm)
        points.append({"value_mean": vm, "value": line["value"], "ms_per_step": line["ms_per_step"],
                       "kernel_ms": line["roofline"]["kernel_ms"], "frac": line["roofline"]["frac"],
                       "logical_topic_gb_s": line["logical_topic_gb_s"]})
        if vm == a.value_mean:
            head = line
    head = head or line
    head["sweep"] = points
    return head


def extra_modes(a, topic, kta, torch, dev, peak):
    """Kernel-only numbers for the other modes on the same topic (informational)."""
    out = {}
    for mode in ("counters", "hll", "alive", "fused"):
        if mode == a.mode:
            continue
        try:
            eng = make_engine(kta, a, mode, dev.index)
            eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)

            def topic_pass(k):
                eng.reset()
                for _ in range(k):
                    scan_topic(eng, topic, mode)
                eng.finalize()
            topic_pass(max(1, a.warmup))
            eng.set_timing(True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            topic_pass(a.steps)
            e1.record()
            torch.cuda.synchronize(dev)
            kms, kn = eng.scan_time_ms()
            alg = 20 * topic.n + (topic.key_bytes_len if mode != "counters" else 0)
            ach = alg / (kms / kn / 1e3) / 1e9
            out[mode] = {"msg_per_s": topic.n * a.steps / (e0.elapsed_time(e1) / 1e3), "kernel_ms": kms / kn,
                         "achieved_gb_s": ach, "frac": ach / peak,
                         "alive_keys": eng.alive_keys() if mode in ("alive", "fused") else None}
            eng.close()
        except Exception as ex:  # informational only
            out[mode] = {"error": repr(ex)}
    return out


def e2e_push(a):
    """The reference's own call shape, one handle_message per polled record (src/kafka.rs:107-109): the C++ host driver
    (csrc/cli, a separate binary over libkta_gpu.so) calls kta_push once per record, keys included, kta_finalize inside
    the timed region.  Library time only (the synthetic generator is excluded)."""
    cli = os.path.join(ROOT, "kafka_topic_analyzer_b200", "csrc", "cli", "kafka-topic-analyzer")
    if not os.path.exists(cli):
        return {"unavailable": "csrc/cli/kafka-topic-analyzer not built"}
    n = 20_000_000
    synthetic = ("n=%d,partitions=%d,value_mean=%d,run_len=%d,distinct_keys=%d,key_mode=%d,tombstone_per_10k=%d,null_key_per_10k=%d"
                 % (n, a.partitions, a.value_mean, a.run_len, min(a.distinct_keys, n // 2), a.key_mode, a.tombstones, a.null_keys))
    out = {"records": n, "path": "kafka-topic-analyzer --feed push: one kta_push call per record + kta_finalize"}
    for name, flags in (("counters", []), ("count_alive_keys", ["-c"])):
        try:
            r = subprocess.run([cli, "-t", "bench", "-b", "none", "--synthetic", synthetic, "--feed", "push", *flags],
                               capture_output=True, text=True, timeout=600)
            m = re.search(r"feed=push: (\d+) records through the handlers in ([0-9.]+) s = ([0-9.e+]+) msg/s", r.stderr)
            out[name] = {"value": float(m.group(3)), "unit": UNIT, "seconds": float(m.group(2))} if m else {"error": r.stderr[-300:]}
        except Exception as ex:
            out[name] = {"error": repr(ex)}
    return out


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
