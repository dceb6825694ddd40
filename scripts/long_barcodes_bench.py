"""Reads per second of long decoders (33-64 nt) on the device path, next to a 40 nt MDD decoder and the card it ran on.

    python scripts/long_barcodes_bench.py [--reads N] [--steps K] [--warmup W]

Each configuration is one decoder of 96 random barcodes with unequal priors. Its reads are synthesized, packed on the
host and uploaded once; the timed steps call phq_decode_batch_device on the resident tiles, timed with CUDA events over
all K steps. Prints one JSON line per configuration, with the card's name and power limit read in the same run.
Writes nothing."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from pheniqs_b200 import DecoderChain, compile_job, workload  # noqa: E402

CONFIGS = (("pamld 96 x [20, 20]", "pamld", (20, 20)), ("pamld 96 x [64]", "pamld", (64,)), ("mdd 96 x [20, 20]", "mdd", (20, 20)))


def job(algorithm, segments, seed):
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    codec = {}
    for i in range(96):
        codec["@%02d" % i] = {"barcode": [letters[rng.integers(0, 4, size=n)].tobytes().decode() for n in segments],
                              "concentration": float(rng.integers(1, 5))}
    return {"sample": {"algorithm": algorithm, "codec": codec, "noise": 0.05, "confidence threshold": 0.9,
                       "transform": {"token": ["%d:0:%d" % (i, n) for i, n in enumerate(segments)]}}}


def card():
    query = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in query.stdout.strip().split(",")]
    return name, power


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--reads", type=int, default=1 << 22)
    parser.add_argument("--steps", type=int, default=10)
    parser.add_argument("--warmup", type=int, default=2)
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    name, power = card()
    for label, algorithm, segments in CONFIGS:
        compiled = compile_job(job(algorithm, segments, sum(segments)))
        n = args.reads
        code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=3)
        chain = DecoderChain(compiled, device=0)
        tiles = chain.upload(chain.pack(code, quality, offset), n)
        flags = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
        results = [torch.zeros((n, 2), dtype=torch.float64, device="cuda:0")]
        for _ in range(args.warmup):
            chain.decode_device(tiles, n, flags, results)
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(args.steps):
            chain.decode_device(tiles, n, flags, results)
        stop.record()
        torch.cuda.synchronize()
        seconds = start.elapsed_time(stop) / 1000.0
        print(json.dumps({"config": label, "kernels": chain.kernel_description(0), "reads": n, "steps": args.steps,
                          "reads_per_second": n * args.steps / seconds, "exact_path_reads": chain.statistics()["exact_path_reads"],
                          "card": name, "power_limit": power}), flush=True)
        chain.close()


if __name__ == "__main__":
    main()
