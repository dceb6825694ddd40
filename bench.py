#!/usr/bin/env python3
"""bench.py — reads/s decoded on the barcode classification path, on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1] [--configs c2,c3,c4,c5] [--impl reference]

One "step" is one pass of the hot path over one batch of synthetic reads resident in HBM:
reset accumulators -> classify every read of the batch against every barcode of every decoder of the
workload (one kernel set per decoder) -> collect: the accumulator planes all-reduced across ranks
(phq_collect, the path's only collective). Reads are sharded per rank (weak scaling: sizes are per GPU).

Prints ONE JSON line (rank 0). The top level of the line is BASELINE.json's headline configuration, c1
(96 x [8,8] dual index PAMLD): `value` is device-timed (CUDA events on the launching stream, max over
ranks); `e2e` is the same metric through the host-buffer C-ABI call that starts from the bytes a feed
holds (FASTQ bytes of the barcode segments in, packing on the device, per-read records out, every copy
inside the timed region), next to a plain pinned-copy ceiling measured in the same run; `roofline` relates
the dominant kernel to the measured HBM peak and names the binding resource; `cpu_baseline` is the
reference's own decoder classes (oracle/_ref, else the C port) timed on this host's cores on a bounded
sample of the same reads.

`configs` carries the other four BASELINE.json configurations, each a short run of the same step with its
own clock sample: c2 (MDD), c3 (SPLiT-seq), c4 (sci-RNA-seq: pass 1 -> collect -> Classifier::finalize ->
priors installed -> pass 2, the two-pass workflow of docs/pamld.md:38-44, collective timed separately) and
c5 (737,280 barcode whitelist at 1.25 x 10^8 reads per GPU = 10^9 reads on 8 GPUs, with its 47 MB
all-reduce). At N > 1 every config also verifies, outside the timed region, that the collected planes equal
the sum of the per-rank planes and that the counts cover N x the shard.

`--impl reference` times only the CPU implementation of the headline config (all host threads).

`--dump-outputs DIR` writes what the last timed step of the headline config computed on rank 0 as DIR/<name>.npy:
per tiled decoder k the index, distance and confidence of a fixed, seeded sample of the reads (d<k>_*), the qcfail
flags of the same reads, which reads they are (reads.npy), and every decoder's accumulator tables (d<k>_counts,
d<k>_sums) and the chain totals. The synthetic inputs depend only on the arguments, so two builds run with the same
arguments can be compared file for file: exactly, except the f64 confidence sums (d<k>_sums), which the kernels add
atomically in no fixed order and so agree to rounding.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "reads/sec decoded (PAMLD)"
UNIT = "reads/s"
C5_READS = 125_000_000                      # 10^9 reads over 8 GPUs (BASELINE.json configs[4])
DEFAULT_READS = {"c1": 1 << 28, "c2": 1 << 28, "c3": 1 << 26, "c4": 1 << 26, "c5": C5_READS}
# the short runs of the `configs` object: (reads per GPU, warm-up reads, steps)
SHORT_RUN = {"c1": (1 << 26, None, 5), "c2": (1 << 26, None, 5), "c3": (1 << 24, None, 5), "c4": (1 << 24, None, 5), "c5": (C5_READS, 148 * 15 * 32 * 8, 1)}
WORKLOAD_LABEL = {
    "c1": "C1: Illumina dual-index (i7+i5, 8 bp each) 96-sample PAMLD, noise 0.05, confidence threshold 0.95",
    "c2": "C2: same 96-sample dual-index set, MDD, distance tolerance [1,1]",
    "c3": "C3: SPLiT-seq 3 x 96 x [8] + 4 x [6] PAMLD cellular + naive 10 bp UMI",
    "c4": "C4: sci-RNA-seq 96 x [10] + 196 x [10,10] PAMLD cellular + naive 8 bp UMI, two passes with prior estimation",
    "c5": "C5: 16 bp cellular PAMLD against a 737,280 barcode whitelist + naive 12 bp UMI",
}
NCU_SUMMARY = os.path.join(ROOT, "profiles", "ncu_summary.json")
ORIGINAL_AFFINITY = None
# --dump-outputs: per-read outputs of this many reads (drawn with DUMP_SEED), so that the files of the largest
# configuration (c5: 47 MB of accumulator tables) stay under 64 MB in all
DUMP_READS = 1 << 19
DUMP_SEED = 20240601
DUMP_LIMIT_BYTES = 64_000_000


def algorithmic_bytes_per_read(chain, compiled) -> int:
    """SURVEY.md §8d: per tiled decoder ceil(L/4) + ceil(L/8) bytes of bases and no-call mask, L quality bytes and
    16 bytes out; + 1 byte qcfail in and out per read. An MDD decoder without quality masking never needs the quality
    plane (absent positions travel in the base words), so its L quality bytes are not counted."""
    total = 2
    for info in chain.info:
        if info.has_tile:
            topic = compiled[{0: "sample", 1: "molecular", 2: "cellular"}[info.topic]]
            spec = topic[info.index] if isinstance(topic, list) else topic
            L = info.nucleotide_cardinality
            total += (L + 3) // 4 + (L + 7) // 8 + 16
            if not (info.algorithm == 1 and int(spec.get("quality masking threshold", 0)) <= 0):
                total += L
    return total


def pair_words_per_read(chain) -> int:
    """SURVEY.md §8d: one (read, barcode) pair-word per 16 bases of barcode: C1 96, C3 292, C4 96 + 2 x 196 = 488."""
    return sum(info.barcode_cardinality * info.word_cardinality for info in chain.info if info.has_tile)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe): one
    `nvidia-smi -lms 100` process streaming CSV lines while the timed steps run."""
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.process = None
        self.thread = None
        self.active = threading.Event()

    def _run(self):
        for line in self.process.stdout:
            if self.active.is_set():
                self.samples.append([x.strip() for x in line.strip().split(",")])

    def __enter__(self):
        try:
            self.process = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-lms", "100"],
                                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
            time.sleep(0.35)            # let the first samples arrive before the timed region starts
        except Exception:
            self.process = None
        return self

    def begin(self):
        self.active.set()

    def end(self):
        self.active.clear()

    def __exit__(self, *a):
        if self.process is not None:
            self.process.terminate()
            try:
                self.process.wait(timeout=5)
            except Exception:
                self.process.kill()

    def summary(self):
        rows = [s for s in self.samples if len(s) >= 7 and s[0].replace(".", "").isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(s[0]) for s in rows)
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in rows)]
        power = [float(s[2]) for s in rows if s[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(power) if power else None}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_summary(workload_name):
    """What the committed `ncu --set full` capture of this workload's dominant kernel says (profiles/ncu_summary.json,
    written by scripts/ncu_summary.py from the .ncu-rep): DRAM bytes per read and the counters that name the binding
    resource. File constants from an offline capture, labelled as such; {} when no capture exists."""
    for path in (NCU_SUMMARY, os.path.join(ROOT, "profiles", "traffic.json")):
        try:
            entry = json.load(open(path)).get(workload_name)
            if entry:
                return entry
        except Exception:
            pass
    return {}


def pin_to_gpu_numa_node(local_rank):
    """Bind this rank's threads (and so the first-touch placement of its pinned staging) to the CPUs NVML reports as
    local to its GPU. Returns a short description for the JSON line."""
    global ORIGINAL_AFFINITY
    ORIGINAL_AFFINITY = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"gpu_local_cpus": len(cpus), "bound_cpus": len(allowed), "host_cpus": os.cpu_count()}
    except Exception as e:
        return {"gpu_local_cpus": None, "bound_cpus": None, "host_cpus": os.cpu_count(), "note": "affinity not set: %s" % type(e).__name__}


def host_sample(compiled, spec, n_reads, seed):
    from pheniqs_b200 import workload
    return workload.synthesize(compiled, spec["input segment length"], n_reads, seed=seed, sampling="zipf" if spec["name"] == "c4" else "prior")


def time_cpu(compiled, spec, seconds_target=12.0, threads=None, seed=99):
    """The reference's CPU implementation of the path on this host's cores, on a bounded sample."""
    from oracle import oracle as O
    if ORIGINAL_AFFINITY is not None:
        os.sched_setaffinity(0, ORIGINAL_AFFINITY)      # the CPU arm gets every core of the host, not just the GPU's NUMA node
    threads = threads or (os.cpu_count() or 1)
    probe_n = 2000 if spec["name"] != "c5" else 16
    code, quality, offset, _ = host_sample(compiled, spec, probe_n, seed)
    checker = O.best_oracle(compiled, len(code))
    probe = checker.decode(O.ReadBatch(code, quality, offset), threads=1, want_outputs=False)
    rate = probe_n / max(probe.seconds, 1e-9)
    n = int(min(max(rate * threads * seconds_target, threads * 4), 4e7))
    code, quality, offset, _ = host_sample(compiled, spec, n, seed + 1)
    checker = O.best_oracle(compiled, len(code))
    out = checker.decode(O.ReadBatch(code, quality, offset), threads=threads, want_outputs=False)
    return {"value": n / out.seconds, "unit": UNIT, "cores": threads, "kind": checker.kind,
            "sample": "%d synthetic reads of the same workload, %d threads each with private decoders (transcode.cpp:2296), %.1f s" % (n, threads, out.seconds)}


def run_reference(args, rank, world):
    """The reference's own decoder classes on all host threads: one bounded sample of the workload (synthesized once),
    decoded args.warmup + args.steps times with fresh decoder sets; sized so the whole run stays within a few minutes.
    Nothing of the product is loaded here: the job is compiled by the oracle's own restatement of the compile step."""
    from oracle import oracle as O
    from pheniqs_b200 import workload          # numpy only: the synthetic read generator and the decoder directives
    if rank != 0:
        return
    spec = workload.load(args.workload)
    compiled = O.compile_job(spec["job"])
    threads = os.cpu_count() or 1
    passes = max(args.steps + args.warmup, 1)
    per_step = max(1.5, min(15.0, 100.0 / passes))
    probe_n = 2000 if spec["name"] != "c5" else 16
    code, quality, offset, _ = host_sample(compiled, spec, probe_n, 999)
    probe = O.best_oracle(compiled, len(code)).decode(O.ReadBatch(code, quality, offset), threads=1, want_outputs=False)
    rate = probe_n / max(probe.seconds, 1e-9)
    n = int(min(max(rate * threads * per_step, threads * 4), 4e7))
    code, quality, offset, _ = host_sample(compiled, spec, n, 1000)
    batch = O.ReadBatch(code, quality, offset)
    total_seconds, kind = 0.0, None
    for step in range(passes):
        checker = O.best_oracle(compiled, len(code))
        kind = checker.kind
        out = checker.decode(batch, threads=threads, want_outputs=False)
        if step >= args.warmup:
            total_seconds += out.seconds
    steps = max(passes - args.warmup, 1)
    value = n * steps / max(total_seconds, 1e-9)
    baseline = {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                "sample": "%d synthetic reads of the same workload per step, %d threads each with private decoders (transcode.cpp:2296), %.1f s per step" % (n, threads, total_seconds / steps)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total_seconds / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": {"workload": WORKLOAD_LABEL[args.workload], "reads_per_step": n},
            "cpu_baseline": baseline, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


class Bench:
    """Everything one rank needs to run one configuration after another on its GPU."""

    def __init__(self, args, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        self.device = torch.device("cuda", local_rank)
        self.stream = torch.cuda.current_stream(self.device)
        self.sm_count = torch.cuda.get_device_properties(self.device).multi_processor_count
        self.peak, self.peak_source = measured_peaks()
        self.flush = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.device)

    def max_over_ranks(self, value):
        if self.world == 1:
            return float(value)
        t = self.torch.tensor([value], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def l2_flush(self):
        if self.flush is None:
            self.flush = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.device)
        self.flush.zero_()

    # ------------------------------------------------------------------ one pass, timed
    def timed_steps(self, chain, tiles, n, flags, results, steps, warmup, flush, warm_reads=None, capture=False):
        """`warmup` untimed steps (over the first warm_reads reads when given), then `steps` timed ones between barriers.
        Returns (elapsed ms max over ranks, clocks summary, launches inside the timed region, device ms of the last
        timed step's kernels alone, the last timed step's outputs when `capture` else None)."""
        torch = self.torch

        def step(m, collect=True):
            if flush:
                self.l2_flush()
            flags.zero_()
            chain.reset(self.stream)
            chain.decode_device(tiles, m, flags, results, self.stream)
            if self.world > 1 and collect:
                chain.collect(stream=self.stream)

        for _ in range(warmup):
            step(warm_reads or n)
        self.barrier()
        launches_before = chain.statistics()["kernel_launches"]
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(self.local_rank) as clocks:
            self.barrier()
            clocks.begin()
            start.record(self.stream)
            for _ in range(steps):
                step(n)
            stop.record(self.stream)
            self.barrier()
            launches = chain.statistics()["kernel_launches"] - launches_before
            last_kernel_ms = chain.last_kernel_milliseconds()
            outputs = None
            if capture:
                # read before anything below decodes again (over other reads for c5) or resets the accumulators; the copy
                # leaves the GPU idle, so it stays out of the clock samples
                clocks.end()
                outputs = self.step_outputs(chain, n, flags, results)
                clocks.begin()
            # keep the GPU under the same load a little longer when the timed region was too short to sample
            # (without the collective: every rank decides for itself how long it keeps going)
            extra = 0
            deadline = time.time() + 2.0
            while len(clocks.samples) < 3 and time.time() < deadline:
                step(warm_reads or n, collect=False)
                extra += 1
                if extra % 4 == 0:
                    torch.cuda.synchronize(self.device)
            torch.cuda.synchronize(self.device)
            clocks.end()
        return self.max_over_ranks(start.elapsed_time(stop)), clocks.summary(), int(launches), last_kernel_ms, outputs

    def step_outputs(self, chain, n, flags, results):
        """What a caller of the timed path receives from one step, as float arrays for --dump-outputs: per-read results
        and qcfail flags of DUMP_READS reads drawn with DUMP_SEED (all reads when fewer), every decoder's accumulator
        tables and the chain totals."""
        torch = self.torch
        from pheniqs_b200 import RESULT_DTYPE
        reads = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_READS), replace=False))
        rows = torch.from_numpy(reads).to(self.device)
        out = {"reads": reads.astype(np.float64), "qcfail": flags[rows].cpu().numpy().astype(np.float32)}
        for k in range(chain.n_decoders):
            if results[k] is not None:
                record = results[k][rows].cpu().numpy().view(RESULT_DTYPE).reshape(-1)
                out["d%d_index" % k] = record["index"].astype(np.float32)
                out["d%d_distance" % k] = record["distance"].astype(np.float32)
                out["d%d_confidence" % k] = record["confidence"].astype(np.float64)
            u, f = chain.accumulators(k)
            out["d%d_counts" % k] = u.astype(np.float64)
            out["d%d_sums" % k] = f
        out["totals"] = np.array(chain.totals(), dtype=np.float64)
        return out

    @staticmethod
    def dump_bytes(chain, n):
        """The bytes step_outputs returns for this chain and batch, known before anything runs."""
        sampled = min(n, DUMP_READS)
        per_read = 8 + 4 + sum(4 + 4 + 8 for info in chain.info if info.has_tile)
        tables = sum((info.barcode_cardinality + 1) * (6 + 2) * 8 for info in chain.info)
        return sampled * per_read + tables + 2 * 8

    def kernel_only(self, chain, tiles, n, flags, results, repeats):
        """The decoders' kernels alone (no reset, flush or collective), CUDA events on the launching stream."""
        out = []
        for _ in range(repeats):
            flags.zero_()
            chain.reset(self.stream)
            chain.decode_device(tiles, n, flags, results, self.stream)
            out.append(chain.last_kernel_milliseconds())
        return float(np.mean(out))

    def collect_only(self, chain, repeats=5):
        """The collective alone: reset -> phq_collect between CUDA events (the planes hold zeros: an all-reduce moves the
        same bytes whatever they hold)."""
        if self.world == 1:
            return None
        torch = self.torch
        times = []
        for _ in range(repeats):
            chain.reset(self.stream)
            self.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(self.stream)
            chain.collect(stream=self.stream)
            b.record(self.stream)
            torch.cuda.synchronize(self.device)
            times.append(a.elapsed_time(b))
        chain.reset(self.stream)
        return self.max_over_ranks(float(np.median(times)))

    def verify_sums(self, chain, tiles, n, flags, results):
        """Outside the timed region: one more pass whose per-rank planes are kept, collected, gathered and compared —
        the collected u64 plane must equal the sum of the ranks' planes bit for bit, the f64 plane to 1e-12, and every
        tiled decoder's counts must cover world x n reads."""
        torch, dist = self.torch, self.dist
        flags.zero_()
        chain.reset(self.stream)
        chain.decode_device(tiles, n, flags, results, self.stream)
        u64_plane, f64_plane = chain.accumulator_tensors()
        report = {"reads_covered": None}
        if self.world > 1:
            mine_u, mine_f = u64_plane.clone(), f64_plane.clone()
            chain.collect(stream=self.stream)
            torch.cuda.synchronize(self.device)
            # the per-rank planes travel to rank 0 one plane at a time (c5: 47 MB per rank)
            gathered_u = [torch.empty_like(mine_u) for _ in range(self.world)] if self.rank == 0 else None
            gathered_f = [torch.empty_like(mine_f) for _ in range(self.world)] if self.rank == 0 else None
            dist.gather(mine_u, gathered_u, dst=0)
            dist.gather(mine_f, gathered_f, dst=0)
            if self.rank == 0:
                total_u = torch.stack(gathered_u).sum(dim=0)
                total_f = torch.stack(gathered_f).sum(dim=0)
                assert torch.equal(total_u, u64_plane), "collected u64 plane differs from the sum of the ranks' planes"
                assert torch.allclose(total_f, f64_plane, rtol=1e-12, atol=0), "collected f64 plane differs from the sum of the ranks' planes"
                report["collected_equals_sum_of_ranks"] = True
        torch.cuda.synchronize(self.device)
        covered = []
        for k, info in enumerate(chain.info):
            if info.has_tile:
                u, _ = chain.accumulators(k)
                covered.append(int(u[:, 0].sum()))
        assert all(c == n * self.world for c in covered), "accumulators do not cover world x batch: %r" % covered
        assert chain.totals()[0] == n * self.world
        report["reads_covered"] = n * self.world
        chain.reset()
        return report

    # ------------------------------------------------------------------ roofline
    def roofline(self, name, chain, compiled, n, kernel_ms, clock_summary):
        bytes_per_read = algorithmic_bytes_per_read(chain, compiled)
        achieved = bytes_per_read * n / (kernel_ms * 1e-3) / 1e9
        pairs = pair_words_per_read(chain)
        sm_mhz = clock_summary.get("sm_mhz") or 0
        captured = ncu_summary(name)
        per_read = captured.get("dram_bytes_per_read")
        out = {"bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak,
               "traffic": per_read * n if per_read is not None else None, "peak_source": self.peak_source,
               "kernel": "; ".join(chain.kernel_description(k) for k in range(chain.n_decoders)),
               "kernel_ms_per_launch_set": kernel_ms, "algorithmic_bytes_per_read": bytes_per_read,
               "pair_words_per_read": pairs, "pair_words_per_s": pairs * n / (kernel_ms * 1e-3),
               "pair_words_per_clk_per_sm": (pairs * n / (kernel_ms * 1e-3)) / (sm_mhz * 1e6 * self.sm_count) if sm_mhz else None}
        # The path is NOT HBM bound (SURVEY.md §8d): the HBM fraction above is what the contract asks for. The binding
        # resource is named from the committed ncu capture of the dominant kernel (offline counters, file constants).
        if captured.get("binding"):
            out["binding"] = dict(captured["binding"], source=captured.get("source"))
        # SURVEY.md §8d's integer roofline: the exhaustive formulation costs 19 integer-pipe operations per (read,
        # barcode) pair-word for PAMLD and 7 for MDD; the chip issues 4 warp instructions per clock and SM (measured:
        # profiles/r01_microbench.txt). The kernels restructure the arithmetic (separable grids, lookups, pruned bit-sliced
        # scans, f32 prefilters), so this EQUIVALENT rate can exceed the peak: it measures work avoided, not pipe use.
        equivalent_ops = sum((19 if info.algorithm == 0 else 7) * info.barcode_cardinality * info.word_cardinality for info in chain.info if info.has_tile)
        if sm_mhz:
            issue_peak = self.sm_count * 4 * 32 * sm_mhz * 1e6
            out["int_equivalent"] = {"ops_per_read": equivalent_ops, "ops_per_s": equivalent_ops * n / (kernel_ms * 1e-3),
                                     "issue_peak_lane_ops_per_s": issue_peak, "frac": equivalent_ops * n / (kernel_ms * 1e-3) / issue_peak,
                                     "note": "operations of SURVEY.md §8d's exhaustive formulation per second over the measured issue peak; above 1 = work the kernels avoid"}
        return out

    # ------------------------------------------------------------------ one configuration
    def run(self, name, n, steps, warmup, warm_reads=None, headline=False):
        torch = self.torch
        from pheniqs_b200 import DecoderChain, compile_job, workload
        t_setup = time.perf_counter()
        spec = workload.load(name)
        compiled = compile_job(spec["job"])
        chain = DecoderChain(compiled, device=self.local_rank)
        sampling = "zipf" if name == "c4" else "prior"
        tiles = workload.synthesize_device_tiles(chain, compiled, n, self.device, seed=workload.SEED + 17 * self.rank, sampling=sampling)
        flags = torch.zeros(n, dtype=torch.uint8, device=self.device)
        results = [torch.empty((n, 2), dtype=torch.float64, device=self.device) if info.has_tile else None for info in chain.info]
        setup_seconds = time.perf_counter() - t_setup
        bytes_per_read = algorithmic_bytes_per_read(chain, compiled)
        # timing rule: inputs larger than L2, or L2 flushed between steps (a 256 MB write inside the step)
        flush = bytes_per_read * n < (192 << 20)
        capture = headline and self.args.dump_outputs is not None and self.rank == 0
        if capture and self.dump_bytes(chain, n) > DUMP_LIMIT_BYTES:
            raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (self.dump_bytes(chain, n), DUMP_LIMIT_BYTES))

        elapsed_ms, clocks, launches, last_kernel_ms, outputs = self.timed_steps(chain, tiles, n, flags, results, steps, warmup, flush, warm_reads, capture)
        # the kernels alone: a few more passes, or (long single-step configs) the events of the timed step itself
        kernel_ms = self.kernel_only(chain, tiles, n, flags, results, min(steps, 5)) if steps >= 3 else last_kernel_ms
        collect_ms = self.collect_only(chain)
        entry = {"workload": WORKLOAD_LABEL[name], "value": n * self.world * steps / (elapsed_ms * 1e-3), "unit": UNIT, "ms_per_step": elapsed_ms / steps,
                 "steps": steps, "warmup": warmup, "reads_per_gpu": n, "reads_total": n * self.world,
                 "decoders": chain.n_decoders, "barcodes": [info.barcode_cardinality for info in chain.info],
                 "l2": ("inputs (%d MB per GPU) exceed L2; no flush needed" % (bytes_per_read * n >> 20)) if not flush else
                       ("inputs are %d MB per GPU: L2 flushed with a 256 MB write between steps (inside the timed region)" % (bytes_per_read * n >> 20)),
                 "roofline": self.roofline(name, chain, compiled, n, kernel_ms, clocks), "gpu_launches": launches, "clocks": clocks,
                 "setup_seconds": round(setup_seconds, 1)}
        if collect_ms is not None:
            u64_plane, f64_plane = chain.accumulator_tensors()
            entry["collect"] = {"ms": collect_ms, "bytes": int(8 * (u64_plane.numel() + f64_plane.numel())), "call": "phq_collect: one grouped ncclAllReduce(sum) over the u64 and f64 accumulator planes"}
        entry["verified"] = self.verify_sums(chain, tiles, min(n, 1 << 24), flags, results)

        if name in ("c1", "c4"):
            # c4 is the configuration that asks for it; c1's second pass shows the headline decoder off the equal-prior special case
            entry["two_pass"] = self.two_pass(chain, compiled, spec, tiles, n, flags, results, steps, warmup, flush, sampling)
        if self.rank == 0 and self.world == 1 and not self.args.no_cpu_baseline:
            entry["cpu_baseline"] = time_cpu(compiled, spec, seconds_target=12.0 if headline else 4.0)
        return entry, (spec, compiled, chain, tiles, outputs)

    def two_pass(self, chain, compiled, spec, tiles, n, flags, results, steps, warmup, flush, sampling):
        """The two-pass workflow (docs/pamld.md:38-44; C4 names it): pass 1 under the configured (uniform) priors -> collect (NCCL) ->
        Classifier::finalize (classifier.h:94-124) -> adjust_prior (classifier.h:125-160) -> pass 2 under the estimated
        priors. Each piece timed on its own; the priors every rank derives from the collected tables are compared with
        a one-GPU run over the shards of all ranks."""
        torch = self.torch
        stage = {}
        wall = time.perf_counter()
        flags.zero_()
        chain.reset(self.stream)
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        self.barrier()
        a.record(self.stream)
        chain.decode_device(tiles, n, flags, results, self.stream)
        b.record(self.stream)
        if self.world > 1:
            chain.collect(stream=self.stream)
        c.record(self.stream)
        torch.cuda.synchronize(self.device)
        stage["pass1_ms"] = self.max_over_ranks(a.elapsed_time(b))
        stage["collect_ms"] = self.max_over_ranks(b.elapsed_time(c)) if self.world > 1 else 0.0
        t0 = time.perf_counter()
        priors = {k: chain.estimate_priors(k) for k, info in enumerate(chain.info) if info.algorithm == 0}
        for k, (noise, concentration) in priors.items():
            chain.set_priors(k, noise, concentration)
        chain.reset()
        stage["finalize_and_install_ms"] = self.max_over_ranks(1e3 * (time.perf_counter() - t0))
        flags.zero_()
        self.barrier()
        a.record(self.stream)
        chain.decode_device(tiles, n, flags, results, self.stream)
        b.record(self.stream)
        torch.cuda.synchronize(self.device)
        stage["pass2_ms"] = self.max_over_ranks(a.elapsed_time(b))
        stage["workflow_ms"] = self.max_over_ranks(1e3 * (time.perf_counter() - wall))
        stage["workflow_reads_per_s"] = n * self.world / (stage["workflow_ms"] * 1e-3)
        stage["estimated_noise"] = {str(k): v[0] for k, v in priors.items()}
        stage["kernels_pass2"] = "; ".join(chain.kernel_description(k) for k in range(chain.n_decoders))

        # pass 2 as a timed run of its own, same rules as pass 1
        elapsed_ms, clocks, launches, _, _ = self.timed_steps(chain, tiles, n, flags, results, steps, warmup, flush)
        kernel_ms = self.kernel_only(chain, tiles, n, flags, results, min(steps, 5))
        stage["pass2"] = {"value": n * self.world * steps / (elapsed_ms * 1e-3), "unit": UNIT, "ms_per_step": elapsed_ms / steps, "steps": steps,
                          "roofline": self.roofline("c4_pass2", chain, compiled, n, kernel_ms, clocks), "gpu_launches": launches, "clocks": clocks}

        # the same estimates from ONE GPU over the shards of every rank (rank 0, untimed): integer tables identical,
        # priors to 1e-12 (the f64 planes are not consulted by the estimate)
        if self.world > 1 and self.rank == 0 and n <= (1 << 24):
            from pheniqs_b200 import DecoderChain, workload
            single = DecoderChain(compiled, device=self.local_rank)
            for r in range(self.world):
                shard = workload.synthesize_device_tiles(single, compiled, n, self.device, seed=workload.SEED + 17 * r, sampling=sampling)
                flags.zero_()
                single.decode_device(shard, n, flags, None, self.stream)
                torch.cuda.synchronize(self.device)
                del shard
            worst = 0.0
            for k, (noise, concentration) in priors.items():
                one_noise, one_concentration = single.estimate_priors(k)
                worst = max(worst, abs(one_noise - noise) / max(abs(noise), 1e-300))
                scale = np.maximum(np.abs(concentration), 1e-300)
                worst = max(worst, float(np.max(np.abs(one_concentration - concentration) / scale)))
            assert worst <= 1e-12, "priors from the collected tables differ from the one-GPU run: %g" % worst
            stage["priors_vs_one_gpu_max_relative_difference"] = worst
            single.close()
        # back to the configured priors: what follows (the end to end forms) measures the job as configured
        from pheniqs_b200 import workload
        for k, (_, decoder) in enumerate(workload.chain_of(compiled)):
            if chain.info[k].algorithm == 0:
                _, configured = workload.barcode_matrix(decoder)
                chain.set_priors(k, float(decoder["noise"]), configured)
        chain.reset()
        return stage

    # ------------------------------------------------------------------ end to end (headline config)
    def copy_ceiling(self, h2d_bytes, d2h_bytes, repeats=3):
        """Plain pinned-memory copies of the same byte counts, both directions at once on two streams, all ranks at the
        same time: what the host <-> device links of this box sustain for this rank with no kernel and no API in between."""
        torch = self.torch
        up_host = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
        down_host = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
        up_device = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=self.device)
        down_device = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=self.device)
        s_up, s_down = torch.cuda.Stream(self.device), torch.cuda.Stream(self.device)

        def once():
            with torch.cuda.stream(s_up):
                up_device.copy_(up_host, non_blocking=True)
            with torch.cuda.stream(s_down):
                down_host.copy_(down_device, non_blocking=True)
        once()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(repeats):
            once()
        torch.cuda.synchronize(self.device)
        seconds = self.max_over_ranks(time.perf_counter() - t0)
        return seconds / repeats

    def end_to_end(self, line, spec, compiled, chain, tiles, n, brief=False, brief_reads=1 << 24):
        """Host buffers in, per-read results out, every copy inside the timed region, through the C-ABI calls a host makes.
        Forms, by what the timed region starts from:
          e2e        phq_decode_batch_raw_compact: the FASTQ bytes of the barcode segments (what a feed holds); the device
                     does the decoding, slicing and packing (pack_kernel). The headline.
          e2e_bam    phq_decode_batch_bam_compact: the reference's decoded Segment buffers (BAM codes + Phred bytes)
          e2e_tags   phq_decode_batch_raw_tags: FASTQ bytes in, the BAM auxiliary block of every read out
          e2e_full   phq_decode_batch: tiles packed beforehand (Phred bytes), 16-byte results + qcfail byte
          e2e_packed phq_decode_batch_compact: tiles packed beforehand with codebook qualities, 8-byte records — starts
                     from the device's own format: packing is NOT inside its timed region
        The per-rank batch is the same at every N. `brief` (the short runs under `configs`): e2e and e2e_full only, on 2^24
        reads (four sub-batches in flight over three staging slots; 2^22 for the whitelist config, which is kernel bound)."""
        torch = self.torch
        from pheniqs_b200 import COMPACT_DTYPE, RESULT_DTYPE, workload
        m = min(n, brief_reads) if brief else (self.args.e2e_reads or min(n, 1 << 25))
        e2e_steps = max(3, min(self.args.steps, 5))
        keep = []

        def time_host(call):
            for _ in range(2):
                call()
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                call()
            torch.cuda.synchronize(self.device)
            return self.max_over_ranks(time.perf_counter() - t0) / e2e_steps

        def pinned_results(dtype, width):
            out = []
            for info in chain.info:
                if info.has_tile:
                    buffer = torch.zeros((m, width), dtype=torch.float64).pin_memory()
                    keep.append(buffer)
                    out.append(buffer.numpy().view(dtype).reshape(-1))
                else:
                    out.append(None)
            return out

        def describe(seconds, h2d, d2h, call):
            ceiling = self.copy_ceiling(int(h2d), int(d2h))
            return {"value": m * self.world / seconds, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "reads_per_gpu_per_step": m, "steps": e2e_steps, "call": call,
                    "copy_ceiling": {"value": m * self.world / ceiling, "unit": UNIT, "per_rank_h2d_gbs": h2d / ceiling / 1e9, "per_rank_d2h_gbs": d2h / ceiling / 1e9,
                                     "note": "plain pinned copies of the same bytes in both directions at once, all ranks together"},
                    "frac_of_copy_ceiling": ceiling / seconds}

        tiled = [info.has_tile for info in chain.info]
        topics = [info.topic for info in chain.info if info.has_tile]
        one_decoder_per_topic = len(topics) == len(set(topics))     # the 8-byte records are then lossless w.r.t. the reference's output
        chain.reset()

        # ---- tiles packed beforehand
        host_tiles = chain.allocate_tiles(m, pinned=True)
        for k, t in enumerate(tiles):
            if t is None:
                continue
            host_tiles[k].bases[:] = t[0][:, :m].cpu().numpy().view(np.uint32)
            host_tiles[k].nmask[:] = t[1][:, :m].cpu().numpy().view(np.uint16)
            host_tiles[k].quality[:] = t[2][:, :m].cpu().numpy().view(np.uint32)
        full_results = pinned_results(RESULT_DTYPE, 2)
        qc_buffer = torch.zeros(m, dtype=torch.uint8).pin_memory()
        keep.append(qc_buffer)
        seconds = time_host(lambda: chain.decode(host_tiles, m, None, results=full_results, qcfail_out=qc_buffer.numpy()))
        line["e2e_full"] = describe(seconds, sum(t.bytes_per_read() * m for t in host_tiles if t is not None), 16 * m * sum(tiled) + m,
                                    "phq_decode_batch (tiles packed beforehand, Phred bytes; 16-byte results + qcfail byte out)")
        compact_results = None
        if one_decoder_per_topic and not brief:
            forms = [t.compress_quality() for t in host_tiles if t is not None]
            compact_results = pinned_results(COMPACT_DTYPE, 1)
            seconds = time_host(lambda: chain.decode_compact(host_tiles, m, None, results=compact_results))
            line["e2e_packed"] = describe(seconds, sum(t.bytes_per_read() * m for t in host_tiles if t is not None), 8 * m * sum(tiled),
                                          "phq_decode_batch_compact (tiles packed beforehand with %s-bit codebook qualities; 8-byte records out) — starts from the device's own format" % forms)
        del host_tiles

        # ---- the bytes a feed holds
        raw = workload.raw_segments_from_device_tiles(chain, compiled, tiles, m)
        if raw is None:
            line["e2e"] = dict(line["e2e_full"], note="the raw byte forms are not generated for this workload (reverse complemented tokens); tiles packed beforehand")
            return
        segments = [None if g is None else g[:4] for g in raw]
        raw_bytes = sum(2 * g[3] * m for g in raw if g is not None)
        if one_decoder_per_topic:
            raw_results = pinned_results(COMPACT_DTYPE, 1)
            seconds = time_host(lambda: chain.decode_raw(segments, m, 33, None, compact=True, results=raw_results))
            if compact_results is not None:
                assert all(a is None or np.array_equal(a["packed"], b["packed"]) for a, b in zip(raw_results, compact_results)), "raw and packed forms disagree"
            else:
                assert all(a is None or np.array_equal(a["packed"] & 0xffffff, b["index"].astype(np.uint32)) for a, b in zip(raw_results, full_results)), "raw and packed forms disagree"
            d2h, record = 8 * m * sum(tiled), "8-byte records out"
        else:
            raw_results = pinned_results(RESULT_DTYPE, 2)
            seconds = time_host(lambda: chain.decode_raw(segments, m, 33, None, results=raw_results, qcfail_out=qc_buffer.numpy()))
            assert all(a is None or np.array_equal(a["index"], b["index"]) for a, b in zip(raw_results, full_results)), "raw and packed forms disagree"
            d2h, record = 16 * m * sum(tiled) + m, "16-byte results + qcfail byte out (several decoders per topic)"
        line["e2e"] = describe(seconds, raw_bytes, d2h, "phq_decode_batch_raw%s (FASTQ bytes of the barcode segments in, decoded / sliced / packed on the device; %s)" % ("_compact" if one_decoder_per_topic else "", record))

        if brief:
            chain.reset()
            return
        # the reference's decoded Segment buffers: BAM codes and Phred bytes (sequence.h:264-300), same byte count
        bam_of_ascii = np.full(256, 15, dtype=np.uint8)
        for letter, code in ((b"A", 1), (b"C", 2), (b"G", 4), (b"T", 8)):
            bam_of_ascii[letter[0]] = code
        bam_segments = []
        for g in raw:
            if g is None:
                bam_segments.append(None)
                continue
            code_host = torch.empty(g[0].shape[0], dtype=torch.uint8).pin_memory()
            phred_host = torch.empty(g[1].shape[0], dtype=torch.uint8).pin_memory()
            code_host.numpy()[:] = bam_of_ascii[g[0]]
            phred_host.numpy()[:] = g[1] - 33
            keep += [code_host, phred_host]
            bam_segments.append((code_host.numpy(), phred_host.numpy(), None, g[3]))
        bam_results = pinned_results(COMPACT_DTYPE if one_decoder_per_topic else RESULT_DTYPE, 1 if one_decoder_per_topic else 2)
        if one_decoder_per_topic:
            seconds = time_host(lambda: chain.decode_raw(bam_segments, m, 0, None, compact=True, results=bam_results, bam=True))
            assert all(a is None or np.array_equal(a["packed"], b["packed"]) for a, b in zip(bam_results, raw_results)), "BAM and FASTQ forms disagree"
        else:
            seconds = time_host(lambda: chain.decode_raw(bam_segments, m, 0, None, results=bam_results, qcfail_out=qc_buffer.numpy(), bam=True))
        line["e2e_bam"] = describe(seconds, raw_bytes, d2h, "phq_decode_batch_bam%s (the reference's Segment buffers in: one BAM code and one Phred byte per base; %s)" % ("_compact" if one_decoder_per_topic else "", record))

        # FASTQ bytes in, the auxiliary block of every read out (on a smaller batch: the records are 80+ bytes per read)
        m_tags = min(m, 1 << 24)
        stride = chain.tag_record_bytes()
        aux_buffer = torch.zeros((m_tags, stride), dtype=torch.uint8).pin_memory()
        length_buffer = torch.zeros(m_tags, dtype=torch.int32).pin_memory()
        keep += [aux_buffer, length_buffer]
        tag_segments = [None if g is None else (g[0][:g[3] * m_tags], g[1][:g[3] * m_tags], None, g[3]) for g in raw]
        m_saved, m = m, m_tags
        seconds = time_host(lambda: chain.decode_raw_tags(tag_segments, m_tags, 33, None, stride=stride, aux=aux_buffer.numpy(), aux_length=length_buffer.numpy(), qcfail_out=qc_buffer.numpy()[:m_tags]))
        line["e2e_tags"] = describe(seconds, raw_bytes // m_saved * m_tags, m_tags * (stride + 5),
                                    "phq_decode_batch_raw_tags (FASTQ bytes of the barcode segments in; the auxiliary block RG BC QT XB ... of every read + its length + qcfail out)")
        line["e2e_tags"]["record_bytes"] = stride
        m = m_saved
        chain.reset()


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=10)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--workload", default="c1", choices=sorted(DEFAULT_READS), help="the headline configuration (default c1, BASELINE.json's)")
    parser.add_argument("--configs", default="c2,c3,c4,c5", help="configurations reported as short runs under `configs` ('' for none)")
    parser.add_argument("--reads", type=int, default=0, help="reads per GPU per step of the headline configuration (default: per workload)")
    parser.add_argument("--e2e-reads", type=int, default=0, help="reads per GPU per end-to-end step (default min(reads, 2^25), the same at every N)")
    parser.add_argument("--impl", default="b200", choices=["b200", "reference"])
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--no-e2e", action="store_true")
    parser.add_argument("--dump-outputs", metavar="DIR", default=None,
                        help="write what the last timed step of the headline configuration computed as DIR/<name>.npy")
    args = parser.parse_args()
    if args.steps < 1:
        parser.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        parser.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    host = pin_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the classification path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    bench = Bench(args, rank, local_rank, world)
    n = args.reads or DEFAULT_READS[args.workload]
    warm_reads = SHORT_RUN["c5"][1] if args.workload == "c5" else None
    entry, (spec, compiled, chain, tiles, outputs) = bench.run(args.workload, n, args.steps, args.warmup, warm_reads=warm_reads, headline=True)
    if outputs is not None and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, array in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), array)
    del outputs
    line = {"metric": METRIC, "value": entry["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": entry["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": entry["workload"], "reads_per_gpu": n, "decoders": entry["decoders"], "barcodes": entry["barcodes"], "l2": entry["l2"],
                       "parallelism": "reads sharded x%d, accumulators collected by phq_collect (NCCL all-reduce)" % world, "host": host},
            "roofline": entry["roofline"], "gpu_launches": entry["gpu_launches"], "clocks": entry["clocks"], "verified": entry["verified"]}
    for key in ("collect", "two_pass", "cpu_baseline"):
        if key in entry:
            line[key] = entry[key]
    if not args.no_e2e:
        bench.end_to_end(line, spec, compiled, chain, tiles, n)
    chain.close()
    del chain, tiles, entry
    torch.cuda.empty_cache()

    configs = {}
    for name in [c for c in args.configs.split(",") if c and c != args.workload]:
        reads, warm, steps = SHORT_RUN[name]
        try:
            entry, (spec_k, compiled_k, chain, tiles, _) = bench.run(name, reads, steps, 3, warm_reads=warm)
            if not args.no_e2e:
                bench.end_to_end(entry, spec_k, compiled_k, chain, tiles, reads, brief=True, brief_reads=(1 << 22) if name == "c5" else (1 << 24))
            configs[name] = entry
            chain.close()
            del chain, tiles
        except Exception as e:                  # a config that cannot run is reported, not hidden
            if world > 1:
                raise
            configs[name] = {"workload": WORKLOAD_LABEL[name], "error": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    if configs:
        line["configs"] = configs
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
