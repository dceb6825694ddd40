"""Every decode kernel across the whole quality byte range, against the oracle.

The synthetic workloads draw four Phred bins (Q37, Q23, Q12, Q2); here the same reads carry qualities from five
distributions instead:
  low      Q0..Q3 with many N bases: the q = 0 rows, mismatch ratios above 1 (Q1 ~3.9, Q2 ~1.7), the uniform factor
  full     uniform over 0..127
  high     42..93, and the last eighth of the reads Q93 at every base
  extreme  94..127: four mismatches take the f32 prefilter's products near or below the smallest normal float
  byte     uniform over 0..255, and the last eighth of the reads 0xFF at every base (a BAM record with QUAL '*'; a
           FASTQ decoded at too high an offset gives bytes 225..255). PAMLD scores a byte above 127 as q = 0, a base
           without information; MDD compares the byte with the masking threshold as it is.

Domain: the comparison needs the reference's p = B^sigma * prior to be a normal double (every p underflowing is out of
domain, DESIGN.md §5). B^sigma leaves the normal range near sigma = 3,070, and a prior of 10^-k lowers that by 10 k.
So PAMLD decoders longer than 16 nt draw at most Q93 (32 x 93 = 2,976), their priors stay at 10^-7 or above, and
the 94..255 ranges go to decoders of 16 nt or less. MDD does no arithmetic on qualities and takes every range at
every length.

The oracle restatement (oracle/pheniqs_oracle.c) defines a PAMLD byte above 127, where the reference indexes past
its table; the cases with such bytes compare with it rather than with the reference's own classes.

Bar as in test_gpu_parity.py. Every case asserts which kernels ran, so a change in kernel selection cannot empty it."""
import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import DecoderChain, compile_job, workload
from test_gpu_parity import check, run_both
from test_gpu_raw import to_fastq_bytes

DISTRIBUTIONS = ("low", "full", "high", "extreme", "byte")
SHORT_RANGES = ("low", "full", "high")          # what a PAMLD decoder longer than 16 nt may draw
LONGEST_FULL_RANGE = 16


def draw(rng, kind, size, ceiling=255):
    """`size` Phred bytes of distribution `kind`; `full` draws at most `ceiling`."""
    if kind == "low":
        return rng.integers(0, 4, size=size).astype(np.uint8)
    if kind == "full":
        return rng.integers(0, min(ceiling, 127) + 1, size=size).astype(np.uint8)
    if kind == "high":
        return rng.integers(42, 94, size=size).astype(np.uint8)
    assert ceiling >= 255, "the 94..255 ranges are for PAMLD decoders of at most 16 nt"
    if kind == "extreme":
        return rng.integers(94, 128, size=size).astype(np.uint8)
    return rng.integers(0, 256, size=size).astype(np.uint8)


def requalify(rng, kind, code, quality, offset, ceiling):
    """Replace the qualities of synthesized reads (in place) with draws from `kind`, ceiling[s] for input segment s,
    and add substitutions and N bases so that reads mismatch their barcode at a few positions, not only where the
    synthetic quality bins put errors."""
    n = offset[0].shape[0] - 1
    for s, c in enumerate(code):
        q = draw(rng, kind, c.shape[0], ceiling[s])
        tail = offset[s][n - n // 8]
        if kind == "high":
            q[tail:] = 93
        elif kind == "byte":
            q[tail:] = 255
        quality[s] = q
        called = (c == 1) | (c == 2) | (c == 4) | (c == 8)
        swap = called & (rng.random(c.shape) < 0.08)
        two_bit = np.log2(np.maximum(c, 1)).astype(np.int64)
        c[swap] = workload.BAM_OF_2BIT[(two_bit[swap] + rng.integers(1, 4, size=int(swap.sum()))) % 4]
        c[rng.random(c.shape) < (0.15 if kind == "low" else 0.02)] = 15


def chain_job(decoders):
    """The decoders as one chain (the first as the sample decoder, the rest cellular), each on input segments of its
    own: barcode segment i of a helpers.random_job decoder reads input segment i, shifted here past the earlier ones."""
    at = 0
    for d in decoders:
        tokens = d["transform"]["token"]
        d["transform"]["token"] = ["%d:%s" % (int(t.split(":")[0]) + at, t.split(":", 1)[1]) for t in tokens]
        at += len(tokens)
    job = {"sample": decoders[0]}
    if len(decoders) > 1:
        job["cellular"] = decoders[1:]
    return job


def reads(job, kind, n, seed, short_fraction=0.0):
    """(compiled job, code, quality, offset, qcfail) of n synthesized reads requalified with `kind`."""
    compiled = compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=seed, short_fraction=short_fraction)
    ceiling = [255] * len(code)
    for _, decoder in workload.chain_of(compiled):
        if decoder["algorithm"] == "pamld" and int(decoder["nucleotide cardinality"]) > LONGEST_FULL_RANGE:
            for t in decoder["transform"]["token"]:
                ceiling[int(t.split(":")[0])] = 93
    rng = np.random.default_rng(seed + 1)
    requalify(rng, kind, code, quality, offset, ceiling)
    qcfail = (rng.random(n) < 0.1).astype(np.uint8)
    return compiled, code, quality, offset, qcfail


def use_the_restatement(monkeypatch, kind):
    """Bytes above 127 are undefined in the reference's PAMLD; the restatement defines them (as q = 0)."""
    if kind == "byte":
        monkeypatch.setattr(O, "best_oracle", lambda compiled, input_segment_cardinality=0: O.PortOracle(compiled))


def uniform_priors(decoder):
    for record in decoder["codec"].values():
        record["concentration"] = 1.0
    return decoder


def prefilter_decoders(rng, kind, uniform):
    """Single segment PAMLD decoders of 4, 8, 16, 24 and 32 nt: 1, 2, 4, 6 and 8 quality words."""
    decoders = []
    for length in (4, 8, 16, 24, 32):
        if length > LONGEST_FULL_RANGE and kind not in SHORT_RANGES:
            continue
        extra = {"high quality threshold": 30, "high quality distance threshold": 2} if length == 8 else {}
        d = helpers.random_job(rng, "pamld", (length,), 12 if length == 4 else 32, minimum_distance=2 if length == 4 else 3, **extra)
        decoders.append(uniform_priors(d) if uniform else d)
    return decoders


@pytest.mark.gpu
@pytest.mark.parametrize("uniform", [False, True])
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_prefilter_scan(kind, uniform, monkeypatch):
    """pamld_fast_kernel, then the exact scan and the tie pass for the reads it leaves."""
    use_the_restatement(monkeypatch, kind)
    rng = np.random.default_rng(1000 + DISTRIBUTIONS.index(kind) * 2 + uniform)
    job = chain_job(prefilter_decoders(rng, kind, uniform))
    compiled, code, quality, offset, qcfail = reads(job, kind, 6000, seed=41)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    chain = state[0]
    for k, info in enumerate(chain.info):
        G = (info.nucleotide_cardinality + 3) // 4
        assert chain.kernel_description(k).startswith("pamld_fast_kernel<%d, %d> + pamld_kernel<%d>" % (G, int(uniform), G)), chain.kernel_description(k)
    check(*state)


@pytest.mark.gpu
@pytest.mark.parametrize("uniform", [False, True])
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_exact_scan_without_the_prefilter(kind, uniform, monkeypatch):
    """PHQ_DISABLE_FAST=1: the same decoders, every read through the f64 scan and the tie pass."""
    monkeypatch.setenv("PHQ_DISABLE_FAST", "1")
    use_the_restatement(monkeypatch, kind)
    rng = np.random.default_rng(1000 + DISTRIBUTIONS.index(kind) * 2 + uniform)
    job = chain_job(prefilter_decoders(rng, kind, uniform))
    compiled, code, quality, offset, qcfail = reads(job, kind, 6000, seed=43)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    chain = state[0]
    for k, info in enumerate(chain.info):
        G = (info.nucleotide_cardinality + 3) // 4
        assert chain.kernel_description(k) == "pamld_kernel<%d> + pamld_tie_kernel<%d>" % (G, G)
    check(*state)


# (first segment length, second segment length, distinct first words, distinct second words, fill, equal priors),
# and what pamld_grid_kernel's template and the prefilter in front of it look like for that form
GRIDS = {
    "separable": ((8, 8, 5, 8, 1.0, True), "pamld_fast_grid_kernel<8, 8, 0> + pamld_grid_kernel<8, 8, 2, 1, 1>"),
    "dense_8_8": ((8, 8, 7, 6, 1.0, False), "pamld_fast_grid_kernel<8, 8, 8> + pamld_grid_kernel<8, 8, 2, 8, 0>"),
    "dense_10_10": ((10, 10, 4, 16, 1.0, False), "pamld_fast_grid_kernel<10, 10, 16> + pamld_grid_kernel<10, 10, 2, 16, 0>"),
    "sparse": ((6, 6, 5, 7, 0.8, False), "pamld_grid_kernel<6, 6, 2, 0, 0>"),
}


def grid_job(form):
    (la, lb, ka, kb, fill, equal), _ = GRIDS[form]
    rng = np.random.default_rng(la * 100 + ka)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)

    def words(count, length):
        out = []
        while len(out) < count:
            w = rng.integers(0, 4, size=length)
            if all((w != v).sum() >= 3 for v in out):
                out.append(w)
        return [letters[w].tobytes().decode() for w in out]
    first, second = words(ka, la), words(kb, lb)
    codec = {}
    for i, a in enumerate(first):
        for j, b in enumerate(second):
            if rng.random() < fill:
                codec["@%02d_%02d" % (j, i)] = {"barcode": [a, b], "concentration": 1.0 if equal else float(rng.integers(1, 4))}
    return {"sample": {"algorithm": "pamld", "transform": {"token": ["0:0:%d" % la, "1:0:%d" % lb]}, "codec": codec, "noise": 0.04,
                       "confidence threshold": 0.9, "high quality threshold": 20, "high quality distance threshold": 2}}


@pytest.mark.gpu
@pytest.mark.parametrize("form, kind", [(f, k) for f in GRIDS for k in DISTRIBUTIONS if k in SHORT_RANGES or f != "dense_10_10"])
def test_combinatorial_grid(form, kind, monkeypatch):
    """Dual index codecs on the combinatorial scan: the separable form, dense 8 + 8 and 10 + 10 grids (20 nt: no
    qualities above 93), a sparse grid."""
    use_the_restatement(monkeypatch, kind)
    compiled, code, quality, offset, qcfail = reads(grid_job(form), kind, 6000, seed=47)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    description = state[0].kernel_description(0)
    assert description.startswith(GRIDS[form][1]), description
    if form == "sparse":
        assert "pamld_fast" not in description
    check(*state)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_whitelist_scan(kind, monkeypatch):
    """pamld_whitelist_kernel forced onto small codecs (its pruning bound folds the ratios above 1 of Q1 and Q2 in): a
    12 nt decoder with unequal priors and the high quality filter, a 16 nt one with flat priors and no noise."""
    monkeypatch.setenv("PHQ_WHITELIST_MINIMUM", "1")
    use_the_restatement(monkeypatch, kind)
    rng = np.random.default_rng(2000 + DISTRIBUTIONS.index(kind))
    first = helpers.random_job(rng, "pamld", (12,), 200, **{"high quality threshold": 30, "high quality distance threshold": 1})
    second = uniform_priors(helpers.random_job(rng, "pamld", (16,), 300, noise=0.0))
    compiled, code, quality, offset, qcfail = reads(chain_job([first, second]), kind, 6000, seed=53)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    assert all(state[0].kernel_description(k).startswith("pamld_whitelist_kernel") for k in range(2))
    check(*state)


def mdd_decoders(threshold):
    """By lookup (two 8 nt segments, tolerance 1 each: their Shannon bounds), and by scan: one 16 nt segment whose
    tolerance of 4 is more than the lookup enumerates, and five segments, more than the lookup keys."""
    rng = np.random.default_rng(3008)
    extra = {"quality masking threshold": threshold} if threshold else {}
    return [helpers.random_job(rng, "mdd", (8, 8), 16, minimum_distance=3, **extra),
            helpers.random_job(rng, "mdd", (16,), 20, minimum_distance=9, **extra),
            helpers.random_job(rng, "mdd", (4, 4, 4, 4, 4), 30, minimum_distance=3, **extra)]


@pytest.mark.gpu
@pytest.mark.parametrize("threshold", [0, 1, 128, 255])
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_mdd(kind, threshold):
    """mdd_table_kernel and, for the short reads it queues, mdd_kernel; mdd_kernel for every read of the scan decoders.
    A fifth of the reads are short: their absent positions must not count, while an observed base of quality 255 does."""
    compiled, code, quality, offset, qcfail = reads(chain_job(mdd_decoders(threshold)), kind, 8000, seed=59 + DISTRIBUTIONS.index(kind), short_fraction=0.2)
    chain_of = [d for _, d in workload.chain_of(compiled)]
    assert [d["quality masking threshold"] for d in chain_of] == [threshold] * 3
    assert [d["distance tolerance"] for d in chain_of] == [[1, 1], [4], [0] * 5]
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    chain = state[0]
    assert chain.kernel_description(0) == "mdd_table_kernel<2> + mdd_kernel<2> (short reads)"
    assert chain.kernel_description(1) == "mdd_kernel<1>"
    assert chain.kernel_description(2) == "mdd_kernel<0>"
    check(*state)


def forms_job(rng):
    """One PAMLD and one MDD decoder: what the input forms are checked on."""
    return chain_job([helpers.random_job(rng, "pamld", (12,), 32, **{"high quality threshold": 30, "high quality distance threshold": 2}),
                      helpers.random_job(rng, "mdd", (8, 8), 40, minimum_distance=3, **{"quality masking threshold": 20})])


def assert_forms_kernels(chain):
    assert chain.kernel_description(0).startswith("pamld_fast_kernel<3, 0>")
    assert chain.kernel_description(1).startswith("mdd_table_kernel<2>")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_device_resident_tiles(kind, monkeypatch):
    use_the_restatement(monkeypatch, kind)
    compiled, code, quality, offset, qcfail = reads(forms_job(np.random.default_rng(61)), kind, 6000, seed=61)
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled, device_path=True)
    assert_forms_kernels(state[0])
    check(*state)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", DISTRIBUTIONS)
def test_bam_segments(kind):
    """phq_decode_batch_bam: Phred bytes as the reference holds them, packed on the device."""
    compiled, code, quality, offset, qcfail = reads(forms_job(np.random.default_rng(67)), kind, 6000, seed=67)
    n = qcfail.shape[0]
    chain = DecoderChain(compiled, device=0)
    assert_forms_kernels(chain)
    results, flags = chain.decode_raw([(code[i], quality[i], offset[i], 0) for i in range(len(code))], n, 0, qcfail, bam=True)
    checker = O.PortOracle(compiled) if kind == "byte" else O.best_oracle(compiled, len(code))
    expected = checker.decode(O.ReadBatch(code, quality, offset, qcfail))
    check(chain, checker, results, flags, expected)


def assert_identical(chain, results, flags, tables, want, want_flags, want_tables):
    assert np.array_equal(flags, want_flags)
    for k in range(chain.n_decoders):
        for field in ("index", "distance"):
            assert np.array_equal(results[k][field], want[k][field]), (k, field)
        assert np.array_equal(results[k]["confidence"].view(np.uint64), want[k]["confidence"].view(np.uint64)), k
        assert np.array_equal(tables[k][0], want_tables[k][0]), k
        assert np.allclose(tables[k][1], want_tables[k][1], rtol=1e-9, atol=0), k


@pytest.mark.gpu
@pytest.mark.parametrize("bits, codebook", [(2, (0, 1, 127, 255)), (4, (0, 1, 2, 3, 37, 41, 42, 93, 94, 126, 127, 128, 200, 254, 255))])
def test_codebook_qualities(bits, codebook, monkeypatch):
    """Qualities travelling as 2-bit and 4-bit codebook indices, with 0, 1, 127 and 255 in the codebook, decode bit for
    bit as the byte form does, and the byte form as the oracle does."""
    use_the_restatement(monkeypatch, "byte")
    compiled, code, quality, offset, qcfail = reads(forms_job(np.random.default_rng(71)), "low", 6000, seed=71)
    rng = np.random.default_rng(bits)
    quality = [np.array(codebook, dtype=np.uint8)[rng.integers(0, len(codebook), size=q.shape)] for q in quality]
    n = qcfail.shape[0]
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    check(*state)
    chain, _, want, want_flags, _ = state
    assert_forms_kernels(chain)
    want_tables = [chain.accumulators(k) for k in range(chain.n_decoders)]
    chain.reset()
    small = DecoderChain(compiled, device=-1).pack(code, quality, offset, quality_bits=-1)
    assert all(t is None or t.quality_bits == bits for t in small)
    results, flags = chain.decode(small, n, qcfail)
    assert_identical(chain, results, flags, [chain.accumulators(k) for k in range(chain.n_decoders)], want, want_flags, want_tables)


@pytest.mark.gpu
@pytest.mark.parametrize("phred_offset", [33, 64])
def test_fastq_bytes(phred_offset, monkeypatch):
    """phq_decode_batch_raw from FASTQ quality bytes: at offset 33 every printable byte '!'..'~' (Q0..Q93); at offset
    64 the same bytes, those below '@' wrapping to 225..255 as the reference's char arithmetic does (fastq.h:73).
    Bit for bit what the host packer gives for the decoded bytes, and that as the oracle does."""
    use_the_restatement(monkeypatch, "byte")
    compiled, code, quality, offset, qcfail = reads(forms_job(np.random.default_rng(73)), "low", 6000, seed=73)
    rng = np.random.default_rng(phred_offset)
    printable = np.arange(33, 127, dtype=np.int64)
    quality = [((printable[rng.integers(0, printable.size, size=q.shape)] - phred_offset) % 256).astype(np.uint8) for q in quality]
    assert phred_offset == 33 or any(np.any(q >= 225) for q in quality)
    n = qcfail.shape[0]
    state = run_both(None, code, quality, offset, qcfail, compiled=compiled)
    check(*state)
    packed_chain, _, want, want_flags, _ = state
    sequence, ascii_quality = to_fastq_bytes(code, quality, phred_offset)
    assert all(np.all((a >= 33) & (a <= 126)) for a in ascii_quality)
    chain = DecoderChain(compiled, device=0)
    assert_forms_kernels(chain)
    results, flags = chain.decode_raw([(sequence[i], ascii_quality[i], offset[i], 0) for i in range(len(code))], n, phred_offset, qcfail)
    assert_identical(chain, results, flags, [chain.accumulators(k) for k in range(chain.n_decoders)],
                     want, want_flags, [packed_chain.accumulators(k) for k in range(chain.n_decoders)])


@pytest.mark.gpu
def test_ten_way_ties_at_high_quality():
    """The ten-way tie set of test_ties_between_sigmas_one_ulp_apart_keep_the_first_barcode at Q42..Q93: ten barcodes
    one mismatch away from every read, most reads with one quality at every position."""
    rng = np.random.default_rng(97)
    letters = "ACGT"
    base_word = "ACGTTGCAAC"
    codec = {}
    for i in range(10):
        w = list(base_word)
        w[i] = letters[(letters.index(w[i]) + 1) % 4]
        codec["@%02d" % i] = {"barcode": ["".join(w)], "concentration": 1.0}
    job = {"sample": {"algorithm": "pamld", "transform": {"token": ["0:0:10"]}, "codec": codec, "noise": 0.02, "confidence threshold": 0.05}}
    n = 6000
    lut = {c: v for c, v in zip("ACGT", (1, 2, 4, 8))}
    code = np.tile(np.array([lut[c] for c in base_word], dtype=np.uint8), (n, 1))
    quality = rng.integers(42, 94, size=(n, 10)).astype(np.uint8)
    same_quality = rng.random(n) < 0.7
    quality[same_quality] = quality[same_quality, :1]
    batch = O.ReadBatch.from_fixed([code], [quality])
    state = run_both(job, batch.code, batch.quality, batch.offset)
    assert state[0].kernel_description(0).startswith("pamld_fast_kernel<3, 1>")
    check(*state)
    assert state[0].statistics()["exact_path_reads"] > n // 2


def test_oracle_scores_bytes_above_127_as_no_information():
    """The restatement's rule for Phred bytes above 127, which the device follows: PAMLD scores such a base 0, exactly
    as q = 0 (oracle/pheniqs_oracle.c substitution_quality), and MDD compares the byte with the masking threshold as
    it is (sequence.h:321-332), here restated in numpy."""
    rng = np.random.default_rng(5)
    mdd = mdd_decoders(136)[0]                          # two 8 nt segments, tolerance 1 each
    compiled = O.compile_job(chain_job([helpers.random_job(rng, "pamld", (8,), 24), mdd]))
    n = 3000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=7)
    requalify(rng, "high", code, quality, offset, [255] * len(code))
    # the PAMLD segment: half the bases and every base of the last eighth of the reads above 127, the others Q42..Q93;
    # the MDD segments: every base above 127
    above = [(rng.random(q.shape) < 0.5) | (np.arange(q.shape[0]) >= o[n - n // 8]) for q, o in zip(quality, offset)]
    above[1:] = [np.ones(q.shape, dtype=bool) for q in quality[1:]]
    high = [np.where(a, rng.integers(128, 256, size=q.shape), q).astype(np.uint8) for q, a in zip(quality, above)]
    zero = [np.where(a, 0, q).astype(np.uint8) for q, a in zip(quality, above)]
    got = O.PortOracle(compiled).decode(O.ReadBatch(code, high, offset))
    zero = O.PortOracle(compiled).decode(O.ReadBatch(code, zero, offset))
    assert np.array_equal(got.index[:, 0], zero.index[:, 0])
    assert np.array_equal(got.distance[:, 0], zero.distance[:, 0])
    assert np.array_equal(got.confidence[:, 0].view(np.uint64), zero.confidence[:, 0].view(np.uint64))
    assert len(np.unique(got.index[:, 0])) > 10

    decoder = compiled["cellular"][0]
    barcodes, _ = workload.barcode_matrix(decoder)
    observed = np.concatenate([c.reshape(n, -1)[:, 2:10] for c in code[1:3]], axis=1)
    masked = np.concatenate([q.reshape(n, -1)[:, 2:10] for q in high[1:3]], axis=1) < 136
    error = (observed[:, None, :] != barcodes[None, :, :]) | masked[:, None, :]
    per_segment = np.stack([error[:, :, :8].sum(axis=2), error[:, :, 8:].sum(axis=2)], axis=2)
    within = np.all(per_segment <= np.array(decoder["distance tolerance"]), axis=2)
    exact = np.all(observed[:, None, :] == barcodes[None, :, :], axis=2)
    first = within.argmax(axis=1)
    want_index = np.where(exact.any(axis=1), exact.argmax(axis=1) + 1, np.where(within.any(axis=1), first + 1, 0))
    want_distance = np.where(exact.any(axis=1) | ~within.any(axis=1), 0, per_segment.sum(axis=2)[np.arange(n), first])
    assert np.array_equal(got.index[:, 1], want_index)
    assert np.array_equal(got.distance[:, 1], want_distance)
    assert np.count_nonzero(want_distance == 1) > 100 and np.count_nonzero(want_distance == 2) > 10
