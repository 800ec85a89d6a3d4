#!/usr/bin/env python3
"""
bench.py -- reads/sec of the adapter-trimming hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C]     this repo's CUDA path
    python bench.py --impl reference ...                                  the reference's CPU path

--config 2 (default, the configuration BASELINE.json's metric is quoted on): 100 M x 150 bp single-end synthetic
reads per GPU, one 3' adapter AGATCGGAAGAGC, e = 0.1.  --config 3 / 4 / 5: the other single-GPU configurations of
BASELINE.json with the workloads of SURVEY.md section 8(d) (cutadapt_b200/configs.py): five adapters incl. IUPAC +
linked at e = 0.15; 50 M pairs 2 x 150 bp with -q 20 (a pair counts as two reads); 96 anchored 5' barcodes with
indels through the device index, 25 M reads per GPU (the 200 M-read job of 8 GPUs).  Weak scaling: every rank
trims its own shard, no data-path collective; the trim statistics are all-reduced once per step.

One "step" = one pass of the hot path over the whole per-GPU batch.
  value  : whole-job reads/s with the batch resident in HBM (CUDA events, max over ranks).
  e2e    : the same through the host-facing C ABI (cg_process_batch): pinned host buffers, the library's host-side
           packing (reads travel partly as a 3-bases-per-byte stream), H2D copies, kernels, D2H copy of the match
           records all inside the timed region; the byte counts come from the library (cg_ctx_transfer_bytes),
           raw_transfer_value is the same call with CUTADAPT_B200_H2D_PACK=0.
  roofline.achieved : algorithmic bytes (190 B/read: 150 sequence + 8 offset + 32 result; 340 with qualities)
           x reads per pass / mean device time of ALL kernels of the trimming pass, measured with CUDA events on the
           launching stream inside the library -- i.e. the whole hot path, not just its largest kernel.
  parity_checked : every 1000th read of the batch is re-computed with the oracle after the timed region and
           compared with the device's record (bit-exact); a mismatch fails the run.
  cpu_baseline : the reference's own compiled hot path (oracle/_ref) on the host cores, bounded sample, rank 0 at
           N=1 only.

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0's shard), as float64 .npy files:
  matches[2]   : the match records (adapter, astart, astop, rstart, rstop, score, errors, info per slot) of a fixed,
                 seeded sample of DUMP_SAMPLE reads, shape [sample, slots, 8]; "2" = the second mate (config 4)
  qtrim[2]     : the quality-trimming interval of the same reads (config 4)
  statistics[2]: the whole statistics vector of the step (after the all-reduce)
  read_index   : which reads the sample holds
The inputs depend on the arguments only, so two builds can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ADAPTER = "AGATCGGAAGAGC"
ERROR_RATE = 0.1
READ_LEN = 150
# SURVEY.md section 8(d): sequence + offset + record (+ qualities when quality trimming is fused)
ALGO_BYTES = {2: READ_LEN + 8 + 32, 3: READ_LEN + 8 + 32, 4: 2 * READ_LEN + 8 + 32, 5: READ_LEN + 8 + 32}
# ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of all kernels of one pass divided by the reads
# (profiles/README.md); measured once per round, not in the timed run.  None: not captured for that configuration.
NCU_DRAM_BYTES_PER_READ = {2: 259, 3: None, 4: None, 5: 189}     # profiles/r2_launches_config{2_16M,5_25M}.csv
DEFAULT_READS = {2: 100_000_000, 3: 100_000_000, 4: 50_000_000, 5: 25_000_000}   # config 4: pairs
CONFIG_TEXT = {
    2: "one 3' adapter AGATCGGAAGAGC, e=0.1",
    3: "5 adapters (2 plain, IUPAC, N run, linked), e=0.15, reads from the five constructs",
    4: "paired-end 2x150bp, 3' adapters on R1/R2 + quality trimming -q 20 (a pair = 2 reads)",
    5: "demultiplexing, 96 anchored 5' barcodes with indels (device index), e=0.1",
}
HOST_WINDOW_READS = 20_000_000           # pinned host window streamed repeatedly in the e2e leg
DUMP_SAMPLE = 1 << 18                    # reads in --dump-outputs: at most 44 MB of float64 for any configuration
DUMP_SEED = 20240923


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference (oracle/_ref) or, if it did not travel, the C oracle port
# ------------------------------------------------------------------------------------------------

_WORKER = {}


def _cpu_init(kind, path, index, n_workers, config):
    """Pool initializer: every worker loads its slice of the sample once and builds the adapters of the configuration."""
    with open(path) as f:
        rows = [r.split("\t") for r in f.read().split("\n") if r]
    per = max(1, len(rows) // n_workers)
    with index.get_lock():
        me = index.value
        index.value += 1
    _WORKER["rows"] = rows[me * per:(me + 1) * per] or rows[:per]
    _WORKER["config"] = config
    if kind == "reference":
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        import cutadapt.adapters as RA
        from cutadapt_b200 import configs as CF

        e = CF.CONFIG_ERROR_RATE[config]
        if config == 2:
            _WORKER["adapter"] = RA.BackAdapter(ADAPTER, max_errors=e, min_overlap=3)
        elif config == 3:
            objs = [RA.BackAdapter(s, max_errors=e, min_overlap=3, name=f"a{i}") for i, s in enumerate(CF.CONFIG3_BACK)]
            objs.append(RA.LinkedAdapter(RA.PrefixAdapter(CF.CONFIG3_LINKED[0], max_errors=e, min_overlap=3, name="lf"),
                                         RA.BackAdapter(CF.CONFIG3_LINKED[1], max_errors=e, min_overlap=3, name="lb"),
                                         True, False, "linked"))
            _WORKER["adapter"] = RA.MultipleAdapters(objs)
        elif config == 4:
            _WORKER["adapter"] = RA.BackAdapter(CF.CONFIG4_R1, max_errors=e, min_overlap=3)
            _WORKER["adapter2"] = RA.BackAdapter(CF.CONFIG4_R2, max_errors=e, min_overlap=3)
        else:
            _WORKER["adapter"] = RA.IndexedPrefixAdapters(
                [RA.PrefixAdapter(b, max_errors=e, indels=True, name=f"bc{i}") for i, b in enumerate(CF.config5_barcodes())])
    else:
        from oracle import oracle as O
        from cutadapt_b200.kmer_heuristic import create_positions_and_kmers

        _WORKER["oracle"] = O
        _WORKER["tables"] = O.KmerTables(create_positions_and_kmers(ADAPTER, 3, ERROR_RATE, True, False))
    _WORKER["kind"] = kind


def _cpu_worker(repeat):
    """The reference hot path per read: (quality_trim_index,) Adapter.match_to (prefilter + locate) and Match.trimmed."""
    import time as _t

    rows = _WORKER["rows"]
    kept = 0
    t0 = _t.perf_counter()
    n_reads = 0
    if _WORKER["kind"] == "reference":
        adapter = _WORKER["adapter"]
        if _WORKER["config"] == 4:
            from cutadapt.qualtrim import quality_trim_index

            adapter2 = _WORKER["adapter2"]
            for _ in range(repeat):
                for r1, q1, r2, q2 in rows:
                    for ad, read, q in ((adapter, r1, q1), (adapter2, r2, q2)):
                        s, e = quality_trim_index(q, 0, 20, 33)
                        read = read[s:e]
                        m = ad.match_to(read)
                        kept += len(read) if m is None else len(m.trimmed(read))
                n_reads += 2 * len(rows)
        else:
            for _ in range(repeat):
                for (read,) in rows:
                    m = adapter.match_to(read)
                    if m is not None:
                        kept += len(m.trimmed(read))
                n_reads += len(rows)
    else:
        O, kt = _WORKER["oracle"], _WORKER["tables"]
        for _ in range(repeat):
            for row in rows:
                read = row[0]
                if kt.present(read):
                    r = O.locate(ADAPTER, read, ERROR_RATE, 14, min_overlap=3)
                    if r is not None:
                        kept += r[2]
            n_reads += len(rows)
    return _t.perf_counter() - t0, n_reads, kept


def reference_kind():
    ref_dir = os.path.join(ROOT, "oracle", "_ref", "cutadapt")
    if os.path.isdir(ref_dir) and any(f.startswith("_align") and f.endswith(".so") for f in os.listdir(ref_dir)):
        return "reference"
    return "port"


def cpus_available():
    """CPUs this process may use: the affinity mask, cut down by a cgroup CPU quota (containers on a shared host)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, round(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                n = min(n, max(1, round(q / p)))
        except Exception:
            pass
    return n


class CpuArm:
    """All host cores running the reference hot path on pre-parsed reads (spawned workers)."""

    def __init__(self, sample_rows, cores=None, config=2):
        """sample_rows: one tab-separated row per read (config 4: read 1, qualities 1, read 2, qualities 2)."""
        import multiprocessing as mp
        import tempfile

        self.kind = reference_kind()
        if self.kind != "reference" and config != 2:
            raise RuntimeError("the C oracle port only times configuration 2; oracle/_ref is needed for the others")
        # one process per CPU this job may actually use (the affinity mask cut down by a cgroup quota): more would
        # only oversubscribe the baseline
        self.cores = cores or cpus_available()
        self.cores = max(1, min(self.cores, len(sample_rows)))
        fd, self.path = tempfile.mkstemp(suffix=".reads")
        with os.fdopen(fd, "w") as f:
            f.write("\n".join(sample_rows))
        ctx = mp.get_context("spawn")
        index = ctx.Value("i", 0)
        self.pool = ctx.Pool(self.cores, initializer=_cpu_init, initargs=(self.kind, self.path, index, self.cores, config))
        # warm up + calibrate: one pass over each worker's slice
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [1] * self.cores, chunksize=1)
        self.pass_reads = sum(r[1] for r in res)
        self.pass_seconds = max(r[0] for r in res)

    def run(self, seconds_target):
        # calibrate on a warm, multi-pass run (a single pass is dominated by stragglers / dispatch)
        if not getattr(self, "rate", None):
            t0 = time.perf_counter()
            res = self.pool.map(_cpu_worker, [4] * self.cores, chunksize=1)
            self.rate = sum(r[1] for r in res) / (time.perf_counter() - t0)
        # timed rounds until the sample is long enough (the rate estimate improves with every round)
        total_n, total_wall = 0, 0.0
        while total_wall < 0.8 * seconds_target:
            remaining = seconds_target - total_wall
            repeat = max(1, int(round(remaining * self.rate / max(self.pass_reads, 1))))
            t0 = time.perf_counter()
            res = self.pool.map(_cpu_worker, [repeat] * self.cores, chunksize=1)
            wall = time.perf_counter() - t0
            n = sum(r[1] for r in res)
            self.rate = n / wall
            total_n += n
            total_wall += wall
        return total_n / total_wall, total_n, total_wall

    def close(self):
        self.pool.close()
        self.pool.join()
        try:
            os.unlink(self.path)
        except OSError:
            pass


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits"],
                    capture_output=True, text=True, timeout=5).stdout.strip().split("\n")[0]
                parts = [p.strip() for p in out.split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for p in self.samples:
            try:
                sm.append(float(p[0])); mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------

def numa_nodes():
    """{node: set of CPUs this process may use} for the NUMA nodes of the host."""
    nodes = {}
    try:
        allowed = os.sched_getaffinity(0)
        for entry in sorted(os.listdir("/sys/devices/system/node")):
            if not entry.startswith("node") or not entry[4:].isdigit():
                continue
            cpus = set()
            for part in open(f"/sys/devices/system/node/{entry}/cpulist").read().strip().split(","):
                if part:
                    a, _, b = part.partition("-")
                    cpus.update(range(int(a), int(b or a) + 1))
            if cpus & allowed:
                nodes[int(entry[4:])] = cpus & allowed
    except Exception:
        return {}
    return nodes


def best_numa_node_for(dev, torch):
    """
    The NUMA node whose memory the GPU reads fastest, MEASURED: pinned buffers are allocated by a thread running on
    each node in turn (first touch puts them there) and copied to the device.  A deployment would place its read
    buffers like this; the topology files are not reliable inside containers.  Returns (node or None, {node: GB/s}).
    """
    nodes = numa_nodes()
    if len(nodes) < 2:
        return None, {}
    saved = os.sched_getaffinity(0)
    rates = {}
    try:
        dst = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for node, cpus in nodes.items():
            os.sched_setaffinity(0, cpus)
            src = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
            src.fill_(65)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            rates[node] = 4 * src.numel() / (e0.elapsed_time(e1) / 1000.0) / 1e9
            del src
    except Exception:
        rates = {}
    finally:
        os.sched_setaffinity(0, saved)
    if not rates:
        return None, {}
    return max(rates, key=rates.get), {k: round(v, 1) for k, v in rates.items()}


def sample_rows(config, n, shard=0):
    """Bounded CPU sample of the configuration's workload as tab-separated rows (CpuArm)."""
    from cutadapt_b200.configs import make_config_batch, to_strings

    b = make_config_batch(config, n, shard=shard, device="cpu")
    if config == 4:
        cols = [to_strings(b[k]) for k in ("seq", "qual", "seq2", "qual2")]
        return ["\t".join(r) for r in zip(*cols)]
    return to_strings(b["seq"])


def parity_check(config, mates, results, stride=1000):
    """
    Every `stride`-th read of every mate, re-computed with the oracle (C loop on the host threads / the oracle's
    own index for config 5) and compared with the device's records.  Returns (reads checked, mismatches).
    """
    import numpy as np
    import torch
    from oracle import oracle
    from cutadapt_b200 import _lib
    from cutadapt_b200.configs import config5_barcodes

    checked = mismatches = 0
    for mate, res in zip(mates, results):
        n = res.n_reads
        idx = torch.arange(0, n, stride, device=mate["seq"].device)
        rows = mate["seq"].view(n, READ_LEN)[idx].cpu().numpy()
        data = np.ascontiguousarray(rows).reshape(-1)
        offsets = np.arange(idx.numel() + 1, dtype=np.int64) * READ_LEN
        slots = mate["batch"].adapter_set.slots
        got = res.matches.view(n, slots, 8)[idx].cpu().numpy().view(_lib.MATCH_DTYPE).reshape(idx.numel(), 1, slots)
        spec = mate["batch"].spec
        if config == 5:
            exp = oracle.oracle_index_process(config5_barcodes(), ERROR_RATE, True, True, data, offsets, spec.adapters)
            same = np.ones(idx.numel(), dtype=bool)
            for f in ("adapter", "astart", "astop", "rstart", "rstop", "score", "errors"):
                same &= got[f][:, 0, 0] == exp[f]
        else:
            qdata = None
            if mate["qual"] is not None:
                qdata = np.ascontiguousarray(mate["qual"].view(n, READ_LEN)[idx].cpu().numpy()).reshape(-1)
            exp, eqt = oracle.oracle_process_packed(spec.adapters, spec.groups, data, offsets, qdata,
                                                    quality_trim=qdata is not None, cutoff_front=0, cutoff_back=20)
            same = (got == exp).all(axis=(1, 2))
            if qdata is not None:
                same &= (res.qtrim[idx].cpu().numpy() == eqt).all(axis=1)
        checked += int(idx.numel())
        mismatches += int((~same).sum())
    return checked, mismatches


def dump_outputs(out_dir, mates, results, all_stats):
    """--dump-outputs: the step's results as float64 .npy files (see the module docstring)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n = results[0].n_reads
    index = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_SAMPLE, replace=False))
    idx = torch.from_numpy(index).to(results[0].matches.device)
    arrays = {"read_index": index}
    pos = 0
    for k, (m, res) in enumerate(zip(mates, results)):
        suffix = "2" if k else ""
        arrays["matches" + suffix] = res.matches.view(n, -1, 8)[idx].cpu().numpy()
        if res.qtrim is not None:
            arrays["qtrim" + suffix] = res.qtrim[idx].cpu().numpy()
        arrays["statistics" + suffix] = all_stats[pos:pos + m["stats"].numel()].cpu().numpy()
        pos += m["stats"].numel()
    assert sum(a.size for a in arrays.values()) * 8 <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("BENCH_CONFIG", 2)), choices=[2, 3, 4, 5],
                    help="BASELINE.json configuration (SURVEY.md section 8(d) numbering); 2 = the headline metric")
    ap.add_argument("--reads", type=int, default=int(os.environ.get("BENCH_READS", 0)),
                    help="reads (config 4: pairs) per GPU; default: the size BASELINE.json names for the configuration")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --reads per GPU (default); strong: --reads in total, split evenly over the GPUs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64, a fixed sample of reads)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    cfg = args.config
    if not args.reads:
        args.reads = DEFAULT_READS[cfg]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.scaling == "strong":
        args.reads = max(1, args.reads // world)       # the job stays the same size, every GPU gets its share
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    reads_per_unit = 2 if cfg == 4 else 1
    unit = "pairs" if cfg == 4 else "reads"
    workload = f"config {cfg}: {args.reads} {unit} x {READ_LEN}bp synthetic per GPU, {CONFIG_TEXT[cfg]}"
    metric = "reads/sec (150bp SE, 1 adapter, e=0.1)" if cfg == 2 else f"reads/sec (BASELINE config {cfg}: {CONFIG_TEXT[cfg]})"

    if args.impl == "reference":
        if rank != 0:
            return 0
        arm = CpuArm(sample_rows(cfg, 400_000 if cfg != 4 else 200_000), config=cfg)
        kind, cores = arm.kind, arm.cores
        vals = []
        for i in range(args.warmup + args.steps):
            v, n, wall = arm.run(5.0)
            if i >= args.warmup:
                vals.append((v, n, wall))
        arm.close()
        value = sum(n for _, n, _ in vals) / sum(w for _, _, w in vals)
        line = {
            "impl": "reference", "metric": metric, "value": value, "unit": "reads/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * sum(w for _, _, w in vals) / len(vals), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "sample": f"{vals[0][1]} reads per step over {cores} host cores"},
            "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": kind,
                             "cpus_available": cpus_available(),
                             "sample": f"{vals[0][1]} pre-parsed reads per step, "
                                       f"{'quality_trim_index + ' if cfg == 4 else ''}Adapter.match_to + Match.trimmed"},
            "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from cutadapt_b200 import _lib
    from cutadapt_b200.configs import config_adapters, make_config_batch
    from cutadapt_b200.pipeline import DeviceBatch, allreduce_statistics

    n = args.reads
    # CPU baseline first (spawned workers; rank 0, N=1 only), before the GPU is busy
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        arm = CpuArm(sample_rows(cfg, 400_000 if cfg != 4 else 200_000), config=cfg)
        v, nproc, wall = arm.run(12.0)
        arm.close()
        cpu = {"value": v, "unit": "reads/s", "cores": arm.cores, "kind": arm.kind, "cpus_available": cpus_available(),
               "sample": f"{nproc} pre-parsed reads in {wall:.1f}s: {'quality_trim_index + ' if cfg == 4 else ''}"
                         f"Adapter.match_to + Match.trimmed over {arm.cores} processes"}

    data = make_config_batch(cfg, n, shard=rank, device=str(dev))
    offsets = torch.arange(n + 1, device=dev, dtype=torch.int64) * READ_LEN
    ad1, ad2 = config_adapters(cfg)
    qc = (0, 20) if cfg == 4 else None
    mates = []
    for key, qkey, ads in (("seq", "qual", ad1), ("seq2", "qual2", ad2)):
        if ads is None:
            continue
        batch = DeviceBatch(ads, quality_cutoff=qc, device=local_rank)
        slots = batch.adapter_set.slots
        mates.append({
            "seq": data[key].reshape(-1), "qual": data[qkey].reshape(-1) if qc else None, "batch": batch,
            "out": torch.empty((n * slots, 8), dtype=torch.int32, device=dev),
            "qt": torch.empty((n, 2), dtype=torch.int32, device=dev) if qc else None,
            "stats": torch.zeros(int(_lib.lib().cg_stats_size(batch.n_adapters, READ_LEN, 3)), dtype=torch.int64, device=dev),
        })
    del data
    all_stats = torch.zeros(sum(m["stats"].numel() for m in mates), dtype=torch.int64, device=dev)

    def step():
        results = []
        pos = 0
        for m in mates:
            m["stats"].zero_()
            res, _ = m["batch"].run_with_statistics(m["seq"], offsets, m["qual"], max_read_len=READ_LEN, out=m["out"],
                                                    qtrim_out=m["qt"], max_len=READ_LEN, kmax=3, into=m["stats"])
            all_stats[pos:pos + m["stats"].numel()] = m["stats"]
            pos += m["stats"].numel()
            results.append(res)
        allreduce_statistics(all_stats)          # one all-reduce carries the statistics of both mates
        return results

    for _ in range(args.warmup):
        step()
    barrier()
    stage_on = bool(os.environ.get("CUTADAPT_B200_STAGE_TIMES"))
    for m in mates:
        m["batch"].ctx.kernel_time(reset=True)
        if stage_on:
            m["batch"].ctx.stage_times(reset=True)
    launches0 = sum(m["batch"].ctx.launch_count() for m in mates)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        results = step()
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = sum(m["batch"].ctx.launch_count() for m in mates) - launches0
    kern_ms = 0.0
    stage_ms = None
    for m in mates:
        ms, _ = m["batch"].ctx.kernel_time(reset=True)
        kern_ms += ms
        if stage_on:
            st = m["batch"].ctx.stage_times(reset=True)
            stage_ms = st if stage_ms is None else {k: stage_ms[k] + v for k, v in st.items()}
    kern_per_step = kern_ms / args.steps
    t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    with_adapters = [int(m["stats"][2].item()) for m in mates]
    total_reads_stat = int(sum(int(m["stats"][0].item()) for m in mates))
    reads_per_step = n * reads_per_unit
    value = reads_per_step * world * args.steps / (elapsed_ms / 1000.0)
    jit = [m["batch"].adapter_set.jit_status() for m in mates]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, mates, results, all_stats)

    # ---- parity of the timed batch: a fixed 1-in-1000 sample against the oracle (outside the timed region) -----
    checked, mismatches = parity_check(cfg, mates, results)
    if mismatches:
        print(json.dumps({"error": f"{mismatches} of {checked} sampled reads differ from the oracle"}))
        return 3

    # ---- end-to-end through the host-facing C ABI ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        hw = min(n, HOST_WINDOW_READS)
        passes = (n + hw - 1) // hw
        # host buffers on the NUMA node the GPU reads fastest (measured), like a deployment would place them
        gpu_node, node_rates = best_numa_node_for(dev, torch)
        saved_affinity = os.sched_getaffinity(0)
        if gpu_node is not None:
            os.sched_setaffinity(0, numa_nodes()[gpu_node])
        host = []
        for m in mates:
            h_seq = torch.empty(hw * READ_LEN, dtype=torch.uint8, pin_memory=True)
            h_seq.copy_(m["seq"][: hw * READ_LEN])
            h_qual = None
            if m["qual"] is not None:
                h_qual = torch.empty(hw * READ_LEN, dtype=torch.uint8, pin_memory=True)
                h_qual.copy_(m["qual"][: hw * READ_LEN])
            slots = m["batch"].adapter_set.slots
            h_out = torch.empty((hw * slots, 8), dtype=torch.int32, pin_memory=True)
            h_out.zero_()
            h_qt = torch.empty((hw, 2), dtype=torch.int32, pin_memory=True) if h_qual is not None else None
            host.append((h_seq, h_qual, h_out, h_qt))
        h_off = torch.empty(hw + 1, dtype=torch.int64, pin_memory=True)
        h_off.copy_(offsets[: hw + 1])
        os.sched_setaffinity(0, saved_affinity)
        # worker threads of the library's host side (packing for the compressed transfer): this rank's
        # share of the host cores
        if world > 1:
            os.environ.setdefault("CUTADAPT_B200_HOST_THREADS",
                                  str(max(2, min(32, _lib.lib().cg_host_cpus_available() // world))))
        host_threads = int(_lib.lib().cg_host_threads())
        host_ctx = _lib.Context(local_rank)
        host_sets = [_lib.AdapterSet(m["batch"].spec, host_ctx) for m in mates]
        import ctypes as C

        h_stats = [np.zeros(m["stats"].numel(), dtype=np.int64) for m in mates]

        def e2e_step(off=None, count=None):
            # records AND the statistics vector of every chunk come back (cg_process_batch_stats): the payload a
            # worker of the reference hands to the end-of-run merge
            off = h_off if off is None else off
            done = 0
            for p in range(passes):
                cnt = min(hw, n - done) if count is None else count
                for m, hs, (h_seq, h_qual, h_out, h_qt), st in zip(mates, host_sets, host, h_stats):
                    _lib.check(_lib.lib().cg_process_batch_stats(
                        host_ctx.handle, hs.handle, h_seq.data_ptr(), h_qual.data_ptr() if h_qual is not None else None,
                        off.data_ptr(), cnt, C.byref(m["batch"].params), h_out.data_ptr(),
                        h_qt.data_ptr() if h_qt is not None else None, READ_LEN, 3, st.ctypes.data))
                done += cnt

        e2e_step()
        # for the record: one step with the raw (uncompressed) transfer
        os.environ["CUTADAPT_B200_H2D_PACK"] = "0"
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        e2e_step()
        barrier()
        raw_wall = time.perf_counter() - t0
        os.environ["CUTADAPT_B200_H2D_PACK"] = os.environ.get("BENCH_E2E_PACK", "1")     # "0.xx": a fixed share (sweeps)
        e2e_step()             # lets the compressed share of the transfer settle
        e2e_step()
        barrier()
        host_ctx.transfer_bytes(reset=True)
        host_ctx.host_profile(reset=True)
        l0 = host_ctx.launch_count()
        t0 = time.perf_counter()
        e2e_steps = args.steps
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        wall = time.perf_counter() - t0
        tw = torch.tensor([wall], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.item())
        h2d_bytes, d2h_bytes = host_ctx.transfer_bytes()
        # ragged variant: the same bytes cut into reads of 100..150 characters, so that the int64 offsets travel too
        # (equally long reads get their offsets regenerated on the device)
        rng = np.random.default_rng(7)
        lens = rng.integers(100, READ_LEN + 1, size=hw)
        roff = np.zeros(hw + 1, dtype=np.int64)
        np.cumsum(lens, out=roff[1:])
        n_rag = int(np.searchsorted(roff, hw * READ_LEN, side="right") - 1)
        r_off = torch.empty(n_rag + 1, dtype=torch.int64, pin_memory=True)
        r_off.copy_(torch.from_numpy(roff[: n_rag + 1]))
        e2e_step(r_off, n_rag)
        barrier()
        host_ctx.transfer_bytes(reset=True)
        t0 = time.perf_counter()
        e2e_step(r_off, n_rag)
        barrier()
        rag_wall = time.perf_counter() - t0
        rag_h2d, _ = host_ctx.transfer_bytes()
        e2e = {"value": reads_per_step * world * e2e_steps / wall, "unit": "reads/s",
               # counted by the library from the copies it issues (cg_ctx_transfer_bytes): the reads travel as a
               # base-6 stream, three characters per byte, packed by the library's host threads inside the timed
               # region and expanded to the caller's bytes on the device; the offsets of equally long reads are
               # regenerated on the device from (first offset, length)
               "h2d_bytes_per_step": h2d_bytes // e2e_steps, "d2h_bytes_per_step": d2h_bytes // e2e_steps,
               "steps": e2e_steps, "launches": host_ctx.launch_count() - l0,
               "host_threads": host_threads, "host_cpus_available": int(_lib.lib().cg_host_cpus_available()),
               "host_numa_node": int(_lib.lib().cg_ctx_numa_node(host_ctx.handle)), "host_buffer_node": gpu_node, "h2d_GBps_by_node": node_rates,
               "host_profile": {k: (round(v, 4) if isinstance(v, float) else v)
                                for k, v in host_ctx.host_profile().items()},
               "raw_transfer_value": reads_per_step * world / raw_wall,
               "ragged": {"value": n_rag * passes * reads_per_unit * world / rag_wall, "unit": "reads/s",
                          "reads": "100..150 characters, int64 offsets shipped", "h2d_bytes_per_step": rag_h2d},
               "statistics": "reduced on the device per chunk and returned with the records (cg_process_batch_stats)",
               "how": f"cg_process_batch on pinned host buffers (sequences{' + qualities' if qc else ''} + int64 offsets in, "
                      f"32-byte records out), compressed host-to-device transfer (raw_transfer_value: the same with "
                      f"CUTADAPT_B200_H2D_PACK=0); the {n}-{unit} step streams a {hw}-{unit} pinned window {passes}x"}
    sampler.stop()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        algo = ALGO_BYTES[cfg]
        achieved = algo * reads_per_step / (kern_per_step / 1000.0) / 1e9 if kern_per_step > 0 else None
        dram = NCU_DRAM_BYTES_PER_READ.get(cfg)
        line = {
            "metric": metric, "value": value, "unit": "reads/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "baseline_config": cfg, f"{unit}_per_gpu": n, "reads_per_step_per_gpu": reads_per_step,
                       "l2": f"inputs ({reads_per_step * algo / 1e9:.1f} GB/GPU touched per step) larger than L2",
                       "step": "trimming pass of every mate (first stage, plan, DP rounds / per-adapter passes + selection / "
                               "index lookups) + statistics reduction + one int64 all-reduce of the statistics",
                       "with_adapters": with_adapters, "reads_counted": total_reads_stat,
                       "first_stage_specialised": jit},
            "parity_checked": checked, "parity_mismatches": mismatches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None,
                         # ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of the pipeline's kernels
                         # (profiles/README.md), scaled to the reads of one pass: bytes per launch
                         "traffic": dram * reads_per_step if dram else None,
                         "traffic_unit": "bytes per pass (ncu DRAM bytes per read x reads)",
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                         "kernel": "all kernels of one trimming pass (per-kernel shares in profiles/)",
                         "kernel_ms_per_launch": kern_per_step,
                         "stage_ms_per_launch": ({k: v / args.steps for k, v in stage_ms.items()} if stage_ms else None),
                         "algorithmic_bytes_per_read": algo},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches,
            "clocks": sampler.summary(),
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
