"""The C restatement against the reference's own classes (oracle/_ref) on seeded synthetic reads.

MDD, multi-segment PAMLD, reverse complement knits and barcode counts above 5 have no stored vector in the
reference's tests (SURVEY.md §8c); here the restatement is pinned on them by the live reference build where oracle/_ref
is built, and everywhere by tests/golden/reference_outputs.json: a SHA-256 of every array compared below
(tests/golden/make_reference_vectors.py; its "source" names the checker that computed them)."""
import hashlib
import zlib

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import workload

VARIANTS = ["pamld", "pamld_hq", "pamld_rc2", "mdd", "mdd_masked", "mdd_rc"]


def outputs(oracle, batch):
    """Everything a checker reports for one batch, by name: per-read results, accumulators, estimated priors, totals."""
    out = oracle.decode(batch)
    arrays = {name: getattr(out, name) for name in ("index", "distance", "confidence", "qcfail", "read_distance", "read_confidence", "channel")}
    for k in range(oracle.n_decoders):
        arrays["counts%d" % k], arrays["sums%d" % k] = oracle.accumulators(k)
        if oracle.chain[k][1]["algorithm"] == "pamld":
            noise, concentration = oracle.estimate_priors(k)
            arrays["noise%d" % k] = np.array([noise], dtype=np.float64)
            arrays["concentration%d" % k] = concentration
    arrays["totals"] = np.array(oracle.totals(), dtype=np.uint64)
    return arrays


def digests(arrays):
    """SHA-256 of each array's dtype, shape and bytes: equal digests = bit identical arrays."""
    out = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        out[name] = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()
    return out


def both(case, compiled, batch, n_segments):
    port = outputs(O.PortOracle(compiled), batch)
    stored = helpers.golden("reference_outputs.json")[case]
    got = digests(port)
    assert sorted(got) == sorted(stored), case
    assert [name for name in stored if got[name] != stored[name]] == [], case + ": differs from the stored outputs"
    if O.ref_available():
        ref = outputs(O.RefOracle(compiled, n_segments), batch)
        assert sorted(ref) == sorted(port)
        for name in port:
            assert np.array_equal(port[name], ref[name]), case + " " + name          # same operation order -> bit identical
    return port


def baseline_inputs(name):
    spec = workload.load(name)
    compiled = O.compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 3000, seed=11)
    return compiled, O.ReadBatch(code, quality, offset), len(code)


def random_inputs(variant, short):
    rng = np.random.default_rng(zlib.crc32(variant.encode()) % 1000)
    if variant == "pamld":
        decoder = helpers.random_job(rng, "pamld", (8,), 24)
    elif variant == "pamld_hq":
        decoder = helpers.random_job(rng, "pamld", (6, 7), 40, **{"high quality threshold": 20, "high quality distance threshold": 1})
    elif variant == "pamld_rc2":
        decoder = helpers.random_job(rng, "pamld", (10, 10), 60, reverse=True)
    elif variant == "mdd":
        decoder = helpers.random_job(rng, "mdd", (8, 8), 48, minimum_distance=3)
    elif variant == "mdd_masked":
        decoder = helpers.random_job(rng, "mdd", (9,), 30, minimum_distance=5, **{"quality masking threshold": 13})
    else:
        decoder = helpers.random_job(rng, "mdd", (7, 5), 20, reverse=True, minimum_distance=3)
    job = {"sample": decoder, "molecular": [{"algorithm": "naive", "transform": {"token": ["0::4"]}}],
           "cellular": [helpers.random_job(rng, "pamld", (8,), 12), helpers.random_job(rng, "mdd", (8,), 12, minimum_distance=3)]}
    job["cellular"][0]["transform"]["token"] = ["0:3:11"]
    job["cellular"][1]["transform"]["token"] = ["1:0:8"]
    compiled = O.compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], 2500, seed=5, short_fraction=short)
    qcfail = (rng.random(2500) < 0.1).astype(np.uint8)
    return compiled, O.ReadBatch(code, quality, offset, qcfail), len(code)


def degenerate_inputs():
    rng = np.random.default_rng(3)
    job = {"sample": helpers.random_job(rng, "pamld", (8,), 10)}
    for record in job["sample"]["codec"].values():
        record["concentration"] = 1
    compiled = O.compile_job(job)
    n = 64
    code = np.full((n, 10), 15, dtype=np.uint8)
    quality = np.full((n, 10), 30, dtype=np.uint8)
    code[16:32] = 1
    quality[16:32] = 0
    code[32:48] = np.array([1, 2, 4, 8, 1, 2, 4, 8, 1, 2], dtype=np.uint8)
    quality[32:48] = 2
    code[48:] = np.array([1, 2, 4, 8, 1, 2, 4, 8, 1, 2], dtype=np.uint8)
    quality[48:] = rng.integers(0, 42, size=(16, 10))
    return compiled, O.ReadBatch.from_fixed([code], [quality]), 1


def whitelist_inputs():
    spec = workload.load("c5", whitelist_cardinality=4000)
    compiled = O.compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 400, seed=5)
    return compiled, O.ReadBatch(code, quality, offset), len(code)


def cases():
    """(key in reference_outputs.json, inputs) of every test below."""
    for name in ("c1", "c2", "c3", "c4"):
        yield "baseline_" + name, lambda name=name: baseline_inputs(name)
    for variant in VARIANTS:
        for short in (0.0, 0.2):
            yield "random_%s_%g" % (variant, short), lambda variant=variant, short=short: random_inputs(variant, short)
    yield "degenerate", degenerate_inputs
    yield "whitelist_reduced", whitelist_inputs


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_baseline_configs(name):
    out = both("baseline_" + name, *baseline_inputs(name))
    assert (out["index"] > 0).any()


@pytest.mark.parametrize("short", [0.0, 0.2])
@pytest.mark.parametrize("variant", VARIANTS)
def test_random_decoders(variant, short):
    compiled, batch, n_segments = random_inputs(variant, short)
    out = both("random_%s_%g" % (variant, short), compiled, batch, n_segments)
    assert out["qcfail"].sum() >= batch.qcfail.sum()


def test_degenerate_observations():
    """all-N, all-Q0 and all-Q2 observations: the noise filter and the first-maximum rule on exact ties."""
    both("degenerate", *degenerate_inputs())


def test_whitelist_config_reduced():
    """Config 5's shape (16 nt cellular whitelist + naive UMI) on 4,000 barcodes: the restatement and the reference's own
    classes agree bit for bit there too (the full 737,280 barcode table is covered on the GPU box against oracle/_ref)."""
    out = both("whitelist_reduced", *whitelist_inputs())
    assert (out["index"] > 0).any()
