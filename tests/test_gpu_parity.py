"""Parity of the CUDA path (through the C ABI) with the CPU oracle. Run on the B200 box: pytest -m gpu.

Bar (BASELINE.json north_star, SURVEY.md §8d): barcode index, distance and qcfail bit-exact for MDD and
PAMLD; PAMLD posterior within 1e-6 in log space (and the error probability 1 - conf within 1e-6 relative,
floored at the 2^-53 quantum of the reference's own `1.0 - confidence`); u64 accumulators identical;
f64 accumulators and estimated priors within 1e-9 relative."""
import copy

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import DecoderChain, compile_job, workload

pytestmark = pytest.mark.gpu


def run_both(job, code, quality, offset, qcfail=None, compiled=None, device_path=False, oracle_threads=1):
    compiled = compiled or compile_job(job)
    n = int(offset[0].shape[0] - 1)
    chain = DecoderChain(compiled, device=0)
    tiles = chain.pack(code, quality, offset)
    if device_path:
        import torch
        device_tiles = chain.upload(tiles, n)
        flags = torch.zeros(n, dtype=torch.uint8, device="cuda:0") if qcfail is None else torch.from_numpy(np.ascontiguousarray(qcfail)).to("cuda:0")
        device_results = [torch.zeros((n, 2), dtype=torch.float64, device="cuda:0") for _ in range(chain.n_decoders)]
        chain.decode_device(device_tiles, n, flags, device_results)
        torch.cuda.synchronize()
        from pheniqs_b200 import RESULT_DTYPE
        results = [r.cpu().numpy().view(RESULT_DTYPE).reshape(-1) for r in device_results]
        flags_out = flags.cpu().numpy()
    else:
        results, flags_out = chain.decode(tiles, n, qcfail)
    checker = O.best_oracle(compiled, len(code))
    expected = checker.decode(O.ReadBatch(code, quality, offset, qcfail), threads=oracle_threads)
    return chain, checker, results, flags_out, expected


def check(chain, checker, results, flags_out, expected):
    for k, info in enumerate(chain.info):
        label = "decoder %d" % k
        if info.algorithm == 0:
            helpers.compare_pamld(results[k], expected.index[:, k], expected.distance[:, k], expected.confidence[:, k], label)
        else:
            assert np.array_equal(results[k]["index"], expected.index[:, k]), label
            assert np.array_equal(results[k]["distance"], expected.distance[:, k]), label
            assert np.all(results[k]["confidence"] == 0), label
        u, f = chain.accumulators(k)
        eu, ef = checker.accumulators(k)
        assert np.array_equal(u, eu), label + " integer accumulators"
        assert np.allclose(f, ef, rtol=1e-9, atol=0), label + " confidence accumulators"
        if info.algorithm == 0:
            noise, concentration = chain.estimate_priors(k)
            enoise, econcentration = checker.estimate_priors(k)
            # no read classified and passing filter, none below the random barcode probability: both sides form 0 / 0
            assert noise == pytest.approx(enoise, rel=1e-9, nan_ok=True)
            assert np.allclose(concentration, econcentration, rtol=1e-9, atol=0, equal_nan=True)
    assert np.array_equal(flags_out, expected.qcfail)
    assert chain.totals() == checker.totals()


@pytest.mark.parametrize("device_path", [False, True])
@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_baseline_configs(name, device_path):
    spec = workload.load(name)
    compiled = compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 60000, seed=21, sampling="zipf" if name == "c4" else "prior")
    state = run_both(None, code, quality, offset, compiled=compiled, device_path=device_path)
    check(*state)
    # prefilter scan + exact scan + tie pass per PAMLD decoder, lookup + queued scan per MDD decoder, one count kernel per naive decoder
    chain = state[0]
    assert all("pamld_fast" in chain.kernel_description(k) for k, info in enumerate(chain.info) if info.algorithm == 0)
    assert chain.statistics()["kernel_launches"] == sum(3 if info.algorithm == 0 else (2 if info.algorithm == 1 else 1) for info in chain.info)


@pytest.mark.parametrize("name", ["c1", "c3", "c4"])
def test_exact_scans_without_the_prefilter(name, monkeypatch):
    """PHQ_DISABLE_FAST=1: every read goes through the f64 scans (the path the prefilter leaves its hard reads to)."""
    monkeypatch.setenv("PHQ_DISABLE_FAST", "1")
    spec = workload.load(name)
    compiled = compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 40000, seed=22, sampling="zipf" if name == "c4" else "prior")
    state = run_both(None, code, quality, offset, compiled=compiled)
    check(*state)
    chain = state[0]
    assert not any("pamld_fast" in chain.kernel_description(k) for k in range(chain.n_decoders))
    assert chain.statistics()["kernel_launches"] == sum(2 if info.algorithm in (0, 1) else 1 for info in chain.info)


def test_whitelist_config_reduced():
    """Config 5's shape (16 bp cellular barcodes, chunked TMA staging of the table, global accumulators) on a 20,000 barcode whitelist."""
    spec = workload.load("c5", whitelist_cardinality=20000)
    compiled = compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 3000, seed=4)
    check(*run_both(None, code, quality, offset, compiled=compiled))


@pytest.mark.parametrize("variant", ["single", "two_segments_hq", "reverse_short", "flat_priors_no_noise"])
def test_whitelist_kernel_on_small_codecs(variant, monkeypatch):
    """pamld_whitelist_kernel (bit sliced pruning scan + exact path) forced onto small codecs, where the oracle is
    cheap: several blocks per chunk with a ragged last block, the high quality filter, short reads (absent
    positions are not counted), reverse complemented tokens, a decoder without noise (no absolute floor for
    the pruning threshold) and unequal priors."""
    monkeypatch.setenv("PHQ_WHITELIST_MINIMUM", "1")
    rng = np.random.default_rng(77)
    short = 0.0
    if variant == "single":
        decoder = helpers.random_job(rng, "pamld", (8,), 150, minimum_distance=2)
    elif variant == "two_segments_hq":
        decoder = helpers.random_job(rng, "pamld", (6, 7), 100, **{"high quality threshold": 20, "high quality distance threshold": 1})
    elif variant == "reverse_short":
        decoder = helpers.random_job(rng, "pamld", (9, 7), 700, reverse=True, minimum_distance=2)
        short = 0.2
    else:
        decoder = helpers.random_job(rng, "pamld", (12,), 1100, noise=0.0, minimum_distance=2)
        for record in decoder["codec"].values():
            record["concentration"] = 1.0
    job = {"sample": decoder, "cellular": [helpers.random_job(rng, "pamld", (16,), 40)]}
    job["cellular"][0]["transform"]["token"] = ["0:1:17"]
    compiled = compile_job(job)
    n = 12000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=9, short_fraction=short)
    qcfail = (rng.random(n) < 0.1).astype(np.uint8)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    assert all("pamld_whitelist_kernel" in state[0].kernel_description(k) for k in range(state[0].n_decoders))
    check(*state)


def test_whitelist_config_full_size():
    """Config 5 at its full table size: 737,280 x 16 nt, 1,440 chunks streamed per tile of reads; a few
    hundred reads, which is what the CPU oracle finishes in seconds."""
    spec = workload.load("c5")
    compiled = compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 600, seed=11)
    import os
    state = run_both(None, code, quality, offset, compiled=compiled, oracle_threads=os.cpu_count() or 1)
    assert "pamld_whitelist_kernel" in state[0].kernel_description(1) or "pamld_whitelist_kernel" in state[0].kernel_description(0)
    check(*state)


def test_bdggg_golden_through_the_gpu():
    batch, decoders, expected = helpers.bdggg()
    compiled = compile_job(decoders)
    chain, checker, results, flags, oracle_out = run_both(None, batch.code, batch.quality, batch.offset, batch.qcfail, compiled=compiled)
    check(chain, checker, results, flags, oracle_out)
    rg = ["undetermined"] + [k[1:] for k in sorted(compiled["sample"]["codec"])]
    for i, e in enumerate(expected):
        assert (589 if flags[i] else 77) == e["flag"], e["name"]
        assert rg[results[0]["index"][i]] == e["RG"].split(":")[-1], e["name"]
        # Read-level confidence of one decoder per type = the decoder's confidence (read.h:279-285)
        assert helpers.error_tag(results[0]["confidence"][i]) == e["XB"], e["name"]
        assert helpers.error_tag(results[2]["confidence"][i]) == e["XC"], e["name"]
    report = helpers.golden("bdggg_report.json")
    noise, concentration = chain.estimate_priors(0)
    assert noise == pytest.approx(report["sample"]["estimated noise"], abs=2e-15)


@pytest.mark.parametrize("short", [0.0, 0.2])
@pytest.mark.parametrize("variant", ["pamld", "pamld_hq", "pamld_rc2", "pamld_long", "mdd", "mdd_masked", "mdd_rc", "mdd_3seg"])
def test_random_decoders(variant, short):
    rng = np.random.default_rng(abs(hash(variant)) % 1000 + 1)
    if variant == "pamld":
        decoder = helpers.random_job(rng, "pamld", (8,), 24)
    elif variant == "pamld_hq":
        decoder = helpers.random_job(rng, "pamld", (6, 7), 40, **{"high quality threshold": 20, "high quality distance threshold": 1})
    elif variant == "pamld_rc2":
        decoder = helpers.random_job(rng, "pamld", (10, 10), 60, reverse=True)
    elif variant == "pamld_long":
        decoder = helpers.random_job(rng, "pamld", (16, 15), 50, minimum_distance=6)
    elif variant == "mdd":
        decoder = helpers.random_job(rng, "mdd", (8, 8), 48, minimum_distance=3)
    elif variant == "mdd_masked":
        decoder = helpers.random_job(rng, "mdd", (9,), 30, minimum_distance=5, **{"quality masking threshold": 13})
    elif variant == "mdd_rc":
        decoder = helpers.random_job(rng, "mdd", (7, 5), 20, reverse=True, minimum_distance=3)
    else:
        decoder = helpers.random_job(rng, "mdd", (6, 12, 9), 64, minimum_distance=3)
    job = {"sample": decoder, "molecular": [{"algorithm": "naive", "transform": {"token": ["0::4"]}}],
           "cellular": [helpers.random_job(rng, "pamld", (8,), 12), helpers.random_job(rng, "mdd", (8,), 12, minimum_distance=3)]}
    job["cellular"][0]["transform"]["token"] = ["0:3:11"]
    job["cellular"][1]["transform"]["token"] = ["1:0:8"]
    compiled = compile_job(job)
    n = 20000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=5, short_fraction=short)
    qcfail = (rng.random(n) < 0.1).astype(np.uint8)
    check(*run_both(None, code, quality, offset, qcfail, compiled=compiled))


@pytest.mark.parametrize("shape", [(6, 6, 5, 7, 0.8, False), (8, 8, 6, 9, 0.8, False), (10, 10, 14, 14, 0.8, False), (12, 12, 3, 11, 0.8, False),
                                   (8, 8, 5, 8, 1.0, True), (8, 8, 7, 6, 1.0, False), (10, 10, 4, 16, 1.0, True), (8, 8, 9, 7, 0.9, True),
                                   (6, 6, 4, 5, 1.0, True), (12, 12, 3, 20, 1.0, True), (8, 8, 12, 3, 1.0, True)])
def test_combinatorial_codecs(shape):
    """Dual-index style codecs (distinct first-segment words x distinct second-segment words) take the
    combinatorial scan kernel: sparse grids (runs not a multiple of four), dense grids with absent
    combinations, and full grids with equal priors (the separable form: KA + KB word products per read)."""
    compiled = compile_job(helpers.grid_job(*shape))
    code, quality, offset, _ = workload.synthesize(compiled, [0], 30000, seed=8)
    check(*run_both(None, code, quality, offset, compiled=compiled))


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_codebook_qualities_and_compact_results(name):
    """Qualities travelling as 2-bit codebook indices and results travelling as 8-byte records give exactly
    what the byte / 16-byte forms give (the compact error probability is float(1 - confidence), read.h:189)."""
    spec = workload.load(name)
    compiled = compile_job(spec["job"])
    n = 50000
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], n, seed=13)
    chain = DecoderChain(compiled, device=0)
    plain = chain.pack(code, quality, offset)
    results, flags = chain.decode(plain, n)
    u_plain = [chain.accumulators(k) for k in range(chain.n_decoders)]
    chain.reset()
    small = DecoderChain(compiled, device=-1).pack(code, quality, offset, quality_bits=-1)
    assert all(t is None or t.quality_bits == 2 for t in small)
    again, flags_again = chain.decode(small, n)
    for k in range(chain.n_decoders):
        assert np.array_equal(again[k], results[k])
        u, f = chain.accumulators(k)
        assert np.array_equal(u, u_plain[k][0])
    assert np.array_equal(flags, flags_again)
    chain.reset()
    compact = chain.decode_compact(small, n)
    running = np.zeros(n, dtype=np.uint8)
    for k, info in enumerate(chain.info):
        if not info.has_tile:
            continue
        packed = compact[k]["packed"]
        assert np.array_equal(packed & 0xffffff, results[k]["index"].astype(np.uint32))
        assert np.array_equal((packed >> 24) & 0x3f, results[k]["distance"].astype(np.uint32))
        assert np.array_equal(compact[k]["error_probability"], (1.0 - results[k]["confidence"]).astype(np.float32))
        last = k
    assert np.array_equal((compact[last]["packed"] >> 30) & 1, flags.astype(np.uint32))
    # a 4-bit codebook: more than four distinct qualities
    rng = np.random.default_rng(2)
    quality9 = [np.array([2, 7, 11, 14, 22, 25, 30, 33, 37], dtype=np.uint8)[rng.integers(0, 9, size=q.shape)] for q in quality]
    chain.reset()
    wide = chain.pack(code, quality9, offset)
    want, want_flags = chain.decode(wide, n)
    four = DecoderChain(compiled, device=-1).pack(code, quality9, offset, quality_bits=-1)
    assert all(t is None or t.quality_bits == 4 for t in four)
    got, got_flags = chain.decode(four, n)
    for k in range(chain.n_decoders):
        assert np.array_equal(got[k], want[k])
    assert np.array_equal(got_flags, want_flags)


def test_structural_ties_take_the_exact_path():
    """Uniform priors + all-N / low quality observations: many exactly tied barcodes; first maximum must match."""
    rng = np.random.default_rng(3)
    job = {"sample": helpers.random_job(rng, "pamld", (8,), 10, minimum_distance=2)}
    for record in job["sample"]["codec"].values():
        record["concentration"] = 1
    n = 4096
    code = np.full((n, 10), 15, dtype=np.uint8)
    quality = np.full((n, 10), 30, dtype=np.uint8)
    code[1024:2048] = 1
    quality[1024:2048] = 0
    pattern = np.array([1, 2, 4, 8, 1, 2, 4, 8, 1, 2], dtype=np.uint8)
    code[2048:3072] = pattern
    quality[2048:3072] = 2
    code[3072:] = np.array([1, 2, 4, 8], dtype=np.uint8)[rng.integers(0, 4, size=(1024, 10))]
    quality[3072:] = np.array([37, 2], dtype=np.uint8)[rng.integers(0, 2, size=(1024, 10))]
    batch = O.ReadBatch.from_fixed([code], [quality])
    state = run_both(job, batch.code, batch.quality, batch.offset)
    check(*state)
    assert state[0].statistics()["exact_path_reads"] >= 2048


def test_two_pass_prior_estimation():
    """Config 4's workflow: pass 1 with uniform priors, estimate, pass 2 with the estimated priors (docs/pamld.md:38-44)."""
    spec = workload.load("c4")
    compiled = compile_job(spec["job"])
    code, quality, offset, _ = workload.synthesize(compiled, spec["input segment length"], 40000, seed=9, sampling="zipf")
    chain, checker, results, flags, expected = run_both(None, code, quality, offset, compiled=compiled)
    check(chain, checker, results, flags, expected)
    # oracle side of pass 2: rewrite the compiled priors with the oracle's own estimates (classifier.h:125-160)
    adjusted = O.compile_job(spec["job"])
    for k, (topic, decoder) in enumerate(O.decoder_chain(adjusted)):
        if decoder["algorithm"] != "pamld":
            continue
        noise, concentration = checker.estimate_priors(k)
        decoder["noise"] = noise
        decoder["undetermined"]["concentration"] = noise
        for record in decoder["codec"].values():
            record["concentration"] = float(concentration[record["index"] - 1])
    chain.adjust_priors()
    chain.reset()
    tiles = chain.pack(code, quality, offset)
    results2, flags2 = chain.decode(tiles, 40000)
    second = O.best_oracle(adjusted, len(code))
    expected2 = second.decode(O.ReadBatch(code, quality, offset))
    check(chain, second, results2, flags2, expected2)
    assert not np.array_equal(results2[1]["confidence"], results[1]["confidence"])


def priors(compiled):
    """The sample decoder's barcode priors in index order."""
    codec = compiled["sample"]["codec"]
    return np.array([r["concentration"] for r in sorted(codec.values(), key=lambda r: r["index"])])


def check_with_priors(chain, compiled, tiles, concentration, code, quality, offset, qcfail):
    """Give the sample decoder `concentration` through set_priors, decode `tiles` again and compare with the oracle
    under the same priors."""
    chain.set_priors(0, compiled["sample"]["noise"], concentration)
    job = copy.deepcopy(compiled)
    for record in job["sample"]["codec"].values():
        record["concentration"] = float(concentration[record["index"] - 1])
    chain.reset()
    results, flags = chain.decode(tiles, len(qcfail), qcfail)
    checker = O.best_oracle(job, len(code))
    check(chain, checker, results, flags, checker.decode(O.ReadBatch(code, quality, offset, qcfail)))


def test_set_priors_rebuilds_the_grid_form():
    """A full 6 + 6 grid takes the separable form and the prefilter under equal priors, the sparse form without the
    prefilter under unequal ones, and the separable form again when equal priors come back: the grid table is
    rebuilt at another size each time, and the prefilter table stays allocated while the sparse form gates it off."""
    compiled = compile_job(helpers.grid_job(6, 6, 4, 5, 1.0, True))
    n = 20000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=10)
    qcfail = (np.random.default_rng(10).random(n) < 0.1).astype(np.uint8)
    chain = DecoderChain(compiled, device=0)
    tiles = chain.pack(code, quality, offset)
    equal = priors(compiled)
    unequal = equal * (1 + np.arange(equal.size) % 3)
    unequal *= equal.sum() / unequal.sum()
    assert chain.kernel_description(0).startswith("pamld_fast_grid_kernel<6, 6, 0>")
    for concentration, separable in ((equal, True), (unequal, False), (equal, True)):
        check_with_priors(chain, compiled, tiles, concentration, code, quality, offset, qcfail)
        description = chain.kernel_description(0)
        if separable:
            assert description.startswith("pamld_fast_grid_kernel<6, 6, 0>"), description
        else:
            assert description.startswith("pamld_grid_kernel<6, 6, 2, 0, 0> + ") and "pamld_fast" not in description, description


def test_set_priors_rebuilds_the_whitelist_bound(monkeypatch):
    """The whitelist scan prunes with the largest prior as its bound: a prior raised above every other through
    set_priors must raise the bound, or reads of that barcode are pruned away."""
    monkeypatch.setenv("PHQ_WHITELIST_MINIMUM", "1")
    rng = np.random.default_rng(79)
    compiled = compile_job({"sample": helpers.random_job(rng, "pamld", (10,), 300, minimum_distance=2)})
    n = 12000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=11)
    qcfail = (rng.random(n) < 0.1).astype(np.uint8)
    chain = DecoderChain(compiled, device=0)
    tiles = chain.pack(code, quality, offset)
    concentration = priors(compiled)
    concentration[np.argmax(concentration)] = 0.5
    concentration *= (1 - compiled["sample"]["noise"]) / concentration.sum()
    assert concentration.max() > 20 * priors(compiled).max()
    check_with_priors(chain, compiled, tiles, concentration, code, quality, offset, qcfail)
    assert chain.kernel_description(0).startswith("pamld_whitelist_kernel")


def test_large_batch_properties():
    """Size-independent properties on a batch far beyond what the oracle finishes in seconds (2^22 reads):
    every read lands in exactly one accumulator row, pf <= count, totals match, decode is idempotent, and a
    random slice of it is bit-compared with the oracle."""
    import torch
    spec = workload.load("c1")
    compiled = compile_job(spec["job"])
    chain = DecoderChain(compiled, device=0)
    n = 1 << 22
    tiles = workload.synthesize_device_tiles(chain, compiled, n, torch.device("cuda:0"), seed=77)
    flags = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
    results = [torch.zeros((n, 2), dtype=torch.float64, device="cuda:0")]
    chain.decode_device(tiles, n, flags, results)
    torch.cuda.synchronize()
    u, f = chain.accumulators(0)
    assert int(u[:, 0].sum()) == n and chain.totals()[0] == n
    assert np.all(u[:, 1] <= u[:, 0])
    assert chain.totals()[1] == int((flags == 0).sum().item())
    first = results[0].clone()
    flags.zero_()
    chain.decode_device(tiles, n, flags, results)
    torch.cuda.synchronize()
    assert torch.equal(first, results[0])
    from pheniqs_b200 import RESULT_DTYPE
    begin = 1234567
    count = 50000
    bases, nmask, quality = [t[:, begin:begin + count].cpu().numpy() for t in tiles[0]]
    code, q = workload.unpack_tile(bases, nmask, quality, 16)
    batch = O.ReadBatch.from_fixed([np.zeros((count, 0), np.uint8), code[:, :8], code[:, 8:], np.zeros((count, 0), np.uint8)],
                                   [np.zeros((count, 0), np.uint8), q[:, :8], q[:, 8:], np.zeros((count, 0), np.uint8)])
    expected = O.best_oracle(compiled, 4).decode(batch)
    got = results[0][begin:begin + count].cpu().numpy().view(RESULT_DTYPE).reshape(-1)
    helpers.compare_pamld(got, expected.index[:, 0], expected.distance[:, 0], expected.confidence[:, 0], "slice")
    assert np.array_equal(flags[begin:begin + count].cpu().numpy(), expected.qcfail)


def test_reference_power_is_the_libm_pow():
    """The tie pass compares p = pow(B, sigma) * prior where the reference's decision hangs on the rounding of pow itself
    (barcode.h:163, pamld.cpp:73). The device evaluates pow in double-double arithmetic, correctly rounded; glibc's pow is
    correctly rounded except in about one case in a thousand, where it is one ulp off: so the two agree bit for bit
    on at least 99.8 % of random exponents and never differ by more than one ulp."""
    import math
    rng = np.random.default_rng(5)
    # the last band: ties of 24-32 nt barcodes at Q60-Q93
    sigma = np.concatenate([rng.random(100000) * 8, rng.random(100000) * 64, rng.random(100000) * 1200, np.arange(0, 130, dtype=np.float64), np.array([0.0, 3000.0]),
                            1200.0 + rng.random(100000) * 1800.0])
    job = {"sample": helpers.random_job(rng, "pamld", (8,), 12)}
    chain = DecoderChain(compile_job(job), device=0)
    got = chain.reference_power(sigma)
    base = math.pow(10.0, -0.1)
    want = np.array([math.pow(base, x) for x in sigma])
    same = got == want
    assert same.mean() >= 0.998, same.mean()
    assert np.all(np.abs(got - want) <= np.spacing(want)), "more than one ulp from libm"
    chain.close()


def test_ties_between_sigmas_one_ulp_apart_keep_the_first_barcode():
    """Two barcodes one low quality mismatch away from the read, at different positions: their Kahan sums hold the same
    values in a different order and can differ in the last bit while pow() of both is the same double, and the reference
    then keeps the FIRST barcode (strict >, pamld.cpp:73). Small sigma is where that happens (one ulp of sigma is less
    than one ulp of pow below sigma = 8)."""
    rng = np.random.default_rng(99)
    letters = "ACGT"
    base_word = "ACGTTGCAAC"
    codec = {}
    # pairs of barcodes that differ from a common word at one position each
    words = []
    for i in range(10):
        w = list(base_word)
        w[i] = letters[(letters.index(w[i]) + 1) % 4]
        words.append("".join(w))
    for i, w in enumerate(words):
        codec["@%02d" % i] = {"barcode": [w], "concentration": 1.0}
    job = {"sample": {"algorithm": "pamld", "transform": {"token": ["0:0:10"]}, "codec": codec, "noise": 0.02, "confidence threshold": 0.05}}
    n = 6000
    lut = {c: v for c, v in zip("ACGT", (1, 2, 4, 8))}
    code = np.tile(np.array([lut[c] for c in base_word], dtype=np.uint8), (n, 1))
    quality = rng.integers(2, 41, size=(n, 10)).astype(np.uint8)       # every read mismatches each barcode at exactly one position
    same_quality = rng.random(n) < 0.7
    quality[same_quality] = quality[same_quality, :1]                  # ... mostly with one quality everywhere: ten way structural ties
    low = rng.random(n) < 0.5
    quality[low] = np.minimum(quality[low], 7)
    batch = O.ReadBatch.from_fixed([code], [quality])
    state = run_both(job, batch.code, batch.quality, batch.offset)
    check(*state)
    assert state[0].statistics()["exact_path_reads"] > n // 2
