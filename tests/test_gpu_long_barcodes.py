"""Decoders of 33 to 64 nucleotides on the long kernels (pamld_long_kernel + pamld_long_tie_kernel, mdd_long_kernel),
through every entry point, against the oracle at the bar of test_gpu_parity.py. Every case asserts which kernels ran.

Domain (test_gpu_quality_range.py): the reference's p = B^sigma * prior must be a normal double, so a PAMLD decoder of L
nucleotides with priors of 10^-7 or more draws qualities of at most 3000 / L. The synthetic Q37 / Q23 / Q12 / Q2 bins
are inside that at every L <= 64; MDD takes the whole byte range. One case goes outside the rule: reads within three
mismatches of their barcode at Q42..Q93, where the winner's p stays normal and distant barcodes underflow."""
import copy

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import DecoderChain, compile_job, workload
from pheniqs_b200.decoder import parse_auxiliary
from test_gpu_parity import check, run_both
from test_gpu_quality_range import chain_job, reads, uniform_priors
from test_gpu_raw import to_fastq_bytes

pytestmark = pytest.mark.gpu

LETTER = np.frombuffer(b"=ACMGRSVTWYHKDBN", dtype=np.uint8)


def pamld_description(L):
    H = (L + 7) // 8
    return "pamld_long_kernel<%d> + pamld_long_tie_kernel<%d>" % (H, H)


def long_pamld(rng, segments, n_barcodes=48, uniform=False, reverse=False, **extra):
    d = helpers.random_job(rng, "pamld", segments, n_barcodes, minimum_distance=6, reverse=reverse, **extra)
    return uniform_priors(d) if uniform else d


def synthesize(compiled, n, seed, short=0.0):
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=seed, short_fraction=short)
    qcfail = (np.random.default_rng(seed).random(n) < 0.1).astype(np.uint8)
    return code, quality, offset, qcfail


PAMLD_SHAPES = [(33,), (40,), (48,), (64,), (20, 20), (32, 32), (16, 16, 16, 16), (8,) * 8]


@pytest.mark.parametrize("uniform", [False, True])
@pytest.mark.parametrize("segments", PAMLD_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_pamld(segments, uniform):
    """Host tiles, a fifth of the reads short (the PAMLD terminator and stale bytes); the 4 x 16 decoder reverse
    complements its tokens (`~`)."""
    rng = np.random.default_rng(sum(segments) * 2 + uniform)
    job = {"sample": long_pamld(rng, segments, uniform=uniform, reverse=len(segments) == 4, **{"high quality threshold": 30, "high quality distance threshold": 3})}
    compiled = compile_job(job)
    code, quality, offset, qcfail = synthesize(compiled, 6000, seed=11 + len(segments), short=0.2)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    assert state[0].kernel_description(0) == pamld_description(sum(segments))
    check(*state)


def test_pamld_streams_a_large_codec():
    """4,096 barcodes of 40 nt: the table streams through shared memory in chunks, the tie runs span many barcodes."""
    rng = np.random.default_rng(4096)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    codec = {"@%04d" % i: {"barcode": [letters[rng.integers(0, 4, size=40)].tobytes().decode()], "concentration": float(rng.integers(1, 4))} for i in range(4096)}
    job = {"sample": {"algorithm": "pamld", "transform": {"token": ["0:0:40"]}, "codec": codec, "noise": 0.05, "confidence threshold": 0.9}}
    compiled = compile_job(job)
    code, quality, offset, qcfail = synthesize(compiled, 8000, seed=17, short=0.1)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    assert state[0].kernel_description(0) == pamld_description(40)
    check(*state)


@pytest.mark.parametrize("ways", [10, 16])
def test_built_ties(ways):
    """`ways` barcodes of 40 nt one mismatch away from every read, equal priors, most reads one quality at every
    position: ties the tie pass resolves by the reference's Kahan sums, more than the 11 candidates a record names."""
    rng = np.random.default_rng(ways)
    letters = "ACGT"
    base_word = "".join(letters[i] for i in rng.integers(0, 4, size=40))
    codec = {}
    for i in range(ways):
        w = list(base_word)
        w[2 * i] = letters[(letters.index(w[2 * i]) + 1) % 4]
        codec["@%02d" % i] = {"barcode": ["".join(w)], "concentration": 1.0}
    job = {"sample": {"algorithm": "pamld", "transform": {"token": ["0:0:40"]}, "codec": codec, "noise": 0.02, "confidence threshold": 0.05}}
    n = 6000
    lut = {c: v for c, v in zip("ACGT", (1, 2, 4, 8))}
    code = np.tile(np.array([lut[c] for c in base_word], dtype=np.uint8), (n, 1))
    quality = rng.integers(30, 76, size=(n, 40)).astype(np.uint8)
    same = rng.random(n) < 0.7
    quality[same] = quality[same, :1]
    batch = O.ReadBatch.from_fixed([code], [quality])
    state = run_both(job, batch.code, batch.quality, batch.offset)
    assert state[0].kernel_description(0) == pamld_description(40)
    check(*state)
    assert state[0].statistics()["exact_path_reads"] > n // 2


def test_high_qualities_outside_the_domain_rule():
    """64 nt reads within three mismatches of their barcode at Q42..Q93: sigma of the winner stays far below the
    underflow, distant barcodes underflow on both sides."""
    rng = np.random.default_rng(64)
    job = {"sample": long_pamld(rng, (64,), 40)}
    job["sample"]["transform"]["token"] = ["0:0:64"]
    compiled = compile_job(job)
    barcodes, _ = workload.barcode_matrix(compiled["sample"])
    n = 6000
    chosen = rng.integers(0, barcodes.shape[0], size=n)
    code = barcodes[chosen].astype(np.uint8).copy()
    for r in range(n):
        for j in rng.choice(64, size=int(rng.integers(0, 4)), replace=False):
            code[r, j] = workload.BAM_OF_2BIT[(int(np.log2(code[r, j])) + int(rng.integers(1, 4))) % 4]
    quality = rng.integers(42, 94, size=(n, 64)).astype(np.uint8)
    batch = O.ReadBatch.from_fixed([code], [quality])
    state = run_both(job, batch.code, batch.quality, batch.offset)
    assert state[0].kernel_description(0) == pamld_description(64)
    check(*state)


def test_two_pass_prior_estimation():
    """Pass 1 with uniform priors, estimate, pass 2 with the estimated priors (docs/pamld.md:38-44)."""
    rng = np.random.default_rng(91)
    job = {"sample": long_pamld(rng, (24, 24), 32, uniform=True)}
    compiled = compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], 20000, seed=19, sampling="zipf")
    chain, checker, results, flags, expected = run_both(None, code, quality, offset, compiled=compiled)
    check(chain, checker, results, flags, expected)
    adjusted = O.compile_job(job)
    noise, concentration = checker.estimate_priors(0)
    decoder = adjusted["sample"]
    decoder["noise"] = noise
    decoder["undetermined"]["concentration"] = noise
    for record in decoder["codec"].values():
        record["concentration"] = float(concentration[record["index"] - 1])
    chain.adjust_priors()
    chain.reset()
    results2, flags2 = chain.decode(chain.pack(code, quality, offset), 20000)
    second = O.best_oracle(adjusted, len(code))
    check(chain, second, results2, flags2, second.decode(O.ReadBatch(code, quality, offset)))
    assert chain.kernel_description(0) == pamld_description(48)
    # the second pass ran under the estimates: zipf sampling leaves them far from the uniform priors of the first
    assert concentration.max() > 4 * concentration.min()


MDD_SHAPES = {(20, 20): "mdd_long_kernel<2>", (16, 16, 16, 16): "mdd_long_kernel<0>", (64,): "mdd_long_kernel<1>"}


@pytest.mark.parametrize("threshold", [0, 30, 255])
@pytest.mark.parametrize("segments", list(MDD_SHAPES), ids=lambda s: "x".join(map(str, s)))
def test_mdd(segments, threshold):
    """The long MDD scan over the whole quality byte range with short reads; 4 x 16 nt would qualify for the lookup
    tables by its segments, and takes the scan."""
    rng = np.random.default_rng(sum(segments) + threshold)
    extra = {"quality masking threshold": threshold} if threshold else {}
    job = chain_job([helpers.random_job(rng, "mdd", segments, 40, minimum_distance=7, **extra)])
    compiled, code, quality, offset, qcfail = reads(job, "byte", 8000, seed=23 + threshold, short_fraction=0.2)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    assert state[0].kernel_description(0) == MDD_SHAPES[segments]
    check(*state)


def forms_job(rng):
    """A long PAMLD and a long MDD decoder of at most 63 nt, and a short PAMLD decoder: the chain the input forms run."""
    return chain_job([long_pamld(rng, (20, 20), 40, **{"high quality threshold": 30, "high quality distance threshold": 3}),
                      helpers.random_job(rng, "mdd", (30, 30), 40, minimum_distance=9, **{"quality masking threshold": 20}),
                      helpers.random_job(rng, "pamld", (12,), 32)])


def forms_reads(seed):
    compiled = compile_job(forms_job(np.random.default_rng(seed)))
    code, quality, offset, qcfail = synthesize(compiled, 6000, seed=seed, short=0.2)
    return compiled, code, quality, offset, qcfail


def assert_forms_kernels(chain):
    assert chain.kernel_description(0) == pamld_description(40)
    assert chain.kernel_description(1) == "mdd_long_kernel<2>"
    assert chain.kernel_description(2).startswith("pamld_fast_kernel<3, 0> + pamld_kernel<3>")


def test_device_resident_tiles():
    compiled, code, quality, offset, qcfail = forms_reads(29)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled, device_path=True)
    assert_forms_kernels(state[0])
    check(*state)


@pytest.mark.parametrize("sub_batch", [0, 333])
def test_bam_segments(sub_batch, monkeypatch):
    if sub_batch:
        monkeypatch.setenv("PHQ_SUB_BATCH_READS", str(sub_batch))
    compiled, code, quality, offset, qcfail = forms_reads(31)
    n = qcfail.shape[0]
    chain = DecoderChain(compiled, device=0)
    assert_forms_kernels(chain)
    results, flags = chain.decode_raw([(code[i], quality[i], offset[i], 0) for i in range(len(code))], n, 0, qcfail, bam=True)
    checker = O.best_oracle(compiled, len(code))
    check(chain, checker, results, flags, checker.decode(O.ReadBatch(code, quality, offset, qcfail)))


def assert_identical(chain, results, flags, want, want_flags, want_tables):
    assert np.array_equal(flags, want_flags)
    for k in range(chain.n_decoders):
        for field in ("index", "distance"):
            assert np.array_equal(results[k][field], want[k][field]), (k, field)
        assert np.array_equal(results[k]["confidence"].view(np.uint64), want[k]["confidence"].view(np.uint64)), k
        u, f = chain.accumulators(k)
        assert np.array_equal(u, want_tables[k][0]), k
        assert np.allclose(f, want_tables[k][1], rtol=1e-9, atol=0), k


@pytest.mark.parametrize("phred_offset, sub_batch", [(33, 0), (64, 0), (33, 333)])
def test_fastq_bytes(phred_offset, sub_batch, monkeypatch):
    """phq_decode_batch_raw from FASTQ bytes: bit for bit what host packed tiles give, and those as the oracle does;
    at offset 64 bytes below '@' wrap to 225..255 (fastq.h:73)."""
    if sub_batch:
        monkeypatch.setenv("PHQ_SUB_BATCH_READS", str(sub_batch))
    compiled, code, quality, offset, qcfail = forms_reads(37)
    if phred_offset == 64:
        rng = np.random.default_rng(64)
        printable = np.arange(33, 127, dtype=np.int64)
        quality = [((printable[rng.integers(0, printable.size, size=q.shape)] - 64) % 256).astype(np.uint8) for q in quality]
        # PAMLD scores bytes above 127 as q = 0, which the restatement defines (test_gpu_quality_range.py)
        monkeypatch.setattr(O, "best_oracle", lambda compiled, input_segment_cardinality=0: O.PortOracle(compiled))
    n = qcfail.shape[0]
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    check(*state)
    packed_chain, _, want, want_flags, _ = state
    sequence, ascii_quality = to_fastq_bytes(code, quality, phred_offset)
    chain = DecoderChain(compiled, device=0)
    assert_forms_kernels(chain)
    results, flags = chain.decode_raw([(sequence[i], ascii_quality[i], offset[i], 0) for i in range(len(code))], n, phred_offset, qcfail)
    assert_identical(chain, results, flags, want, want_flags, [packed_chain.accumulators(k) for k in range(chain.n_decoders)])


def test_compact_records(monkeypatch):
    """Compact records of a <= 63 nt chain equal the full records, across sub-batch boundaries; a 64 nt decoder refuses
    the compact forms (a 6-bit distance)."""
    monkeypatch.setenv("PHQ_SUB_BATCH_READS", "1000")
    compiled, code, quality, offset, qcfail = forms_reads(41)
    n = qcfail.shape[0]
    chain = DecoderChain(compiled, device=0)
    tiles = chain.pack(code, quality, offset)
    results, flags = chain.decode(tiles, n, qcfail)
    chain.reset()
    compact = chain.decode_compact(tiles, n, qcfail)
    for k in range(chain.n_decoders):
        packed = compact[k]["packed"]
        assert np.array_equal(packed & 0xffffff, results[k]["index"]), k
        assert np.array_equal((packed >> 24) & 0x3f, results[k]["distance"]), k
        assert np.array_equal(compact[k]["error_probability"], (1.0 - results[k]["confidence"]).astype(np.float32)), k
    assert np.array_equal((compact[-1]["packed"] >> 30) & 1, flags)
    rng = np.random.default_rng(63)
    for L, refused in ((63, False), (64, True)):
        c = compile_job({"sample": long_pamld(rng, (L,), 8)})
        codes, quals, offs, _ = synthesize(c, 100, seed=L)
        long_chain = DecoderChain(c, device=0)
        t = long_chain.pack(codes, quals, offs)
        if refused:
            with pytest.raises(Exception) as error:
                long_chain.decode_compact(t, 100)
            assert "6 bit distance" in str(error.value)
            assert long_chain.decode(t, 100)[0][0]["index"].shape == (100,)
        else:
            long_chain.decode_compact(t, 100)
        long_chain.close()


def expected_tags(job, compiled, code, quality, offset, expected):
    """The auxiliary block of every read built from the oracle's verdicts and the input bytes (the format
    test_bdggg_golden_tags pins): a PAMLD sample decoder (RG BC QT XB) and a PAMLD cellular decoder (CB CR CY XC)."""
    port = O.PortOracle(O.compile_job(job))
    batch = O.ReadBatch(code, quality, offset)
    chain = [d for _, d in workload.chain_of(compiled)]
    ids = {0: chain[0]["undetermined"]["ID"]}
    ids.update({record["index"]: record["ID"] for record in chain[0]["codec"].values()})
    barcodes = [workload.barcode_matrix(d)[0] for d in chain]
    observed = [port.extract(k, batch) for k in range(2)]
    blocks = []
    for r in range(batch.n_reads):
        tags = {}
        sample = int(expected.index[r, 0])
        tags["RG"] = ids[sample]
        tags["BC"] = LETTER[observed[0][0][r]].tobytes().decode()
        tags["QT"] = (observed[0][1][r] + 33).astype(np.uint8).tobytes().decode()
        if 0 < expected.confidence[r, 0] < 1:
            tags["XB"] = 1.0 - expected.confidence[r, 0]
        cell = int(expected.index[r, 1])
        tags["CB"] = LETTER[barcodes[1][cell - 1]].tobytes().decode() if cell > 0 else "=" * barcodes[1].shape[1]
        tags["CR"] = LETTER[observed[1][0][r]].tobytes().decode()
        tags["CY"] = (observed[1][1][r] + 33).astype(np.uint8).tobytes().decode()
        if cell > 0 and 0 < expected.confidence[r, 1] < 1:
            tags["XC"] = 1.0 - expected.confidence[r, 1]
        blocks.append(tags)
    return blocks


def test_tags():
    rng = np.random.default_rng(43)
    job = {"sample": long_pamld(rng, (20, 20), 24), "cellular": [long_pamld(rng, (64,), 24)]}
    job["cellular"][0]["transform"]["token"] = ["2:0:64"]
    compiled = compile_job(job)
    n = 3000
    code, quality, offset, qcfail = synthesize(compiled, n, seed=47)
    chain = DecoderChain(compiled, device=0)
    aux, length, flags, results = chain.decode_raw_tags([(LETTER[c], (q.astype(np.int32) + 33).astype(np.uint8), o, 0) for c, q, o in zip(code, quality, offset)],
                                                        n, 33, qcfail, want_results=True)
    assert chain.kernel_description(0) == pamld_description(40) and chain.kernel_description(1) == pamld_description(64)
    checker = O.best_oracle(compiled, len(code))
    expected = checker.decode(O.ReadBatch(code, quality, offset, qcfail))
    check(chain, checker, results, flags, expected)
    blocks = expected_tags(job, compiled, code, quality, offset, expected)
    if O.ref_available():
        reference, reference_flags = O.RefOracle(copy.deepcopy(compiled), len(code)).tags(O.ReadBatch(code, quality, offset, qcfail))
        assert np.array_equal(flags, reference_flags)
        blocks = blocks + reference
    for i, want in enumerate(blocks):
        r = i % n
        got = parse_auxiliary(aux[r, :length[r]])
        assert list(got) == [t for t in ("RG", "BC", "QT", "XB", "CB", "CR", "CY", "XC") if t in want], r
        for tag, value in want.items():
            if tag in ("XB", "XC"):
                # 1 - confidence is formed in f64 (read.h:189), quantised at 2^-53 (the floor of test_gpu_tags.py)
                assert abs(float(got[tag]) - float(value)) <= 1e-6 * float(value) + 8 * 2.0 ** -53, (r, tag)
            else:
                assert got[tag] == value, (r, tag)
    chain.close()


def test_mixed_chain_and_report():
    """A <= 32 nt decoder and a long one in one chain: the oracle's results, the short decoder on the kernels it takes
    alone, and phq_report equal to the report of the oracle's tables."""
    rng = np.random.default_rng(53)
    short = helpers.random_job(rng, "pamld", (16,), 32)
    job = chain_job([short, long_pamld(rng, (48,), 40)])
    compiled = compile_job(job)
    alone = DecoderChain(compile_job({"sample": copy.deepcopy(job["sample"])}), device=0).kernel_description(0)
    code, quality, offset, qcfail = synthesize(compiled, 6000, seed=59, short=0.1)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    chain, checker = state[0], state[1]
    assert chain.kernel_description(0) == alone
    assert chain.kernel_description(1) == pamld_description(48)
    check(*state)
    tables = [checker.accumulators(k) for k in range(chain.n_decoders)]
    same_report(chain.report(), chain.encode_report(tables, checker.totals()))


def same_report(got, want, path="report"):
    """Equal keys, strings and integers; floats within the 1e-9 the f64 accumulators are held to."""
    assert type(got) is type(want) or {type(got), type(want)} <= {int, float}, path
    if isinstance(want, dict):
        assert sorted(got) == sorted(want), path
        for key in want:
            same_report(got[key], want[key], path + "." + key)
    elif isinstance(want, list):
        assert len(got) == len(want), path
        for i, (a, b) in enumerate(zip(got, want)):
            same_report(a, b, "%s[%d]" % (path, i))
    elif isinstance(want, float) or isinstance(got, float):
        assert got == pytest.approx(want, rel=1e-9, abs=1e-15), path
    else:
        assert got == want, path
