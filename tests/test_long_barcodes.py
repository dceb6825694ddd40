"""Decoders of 33 to 64 nucleotides on the host side: configuration limits, decoder shapes and phq_pack's planes.
No GPU needed; the kernels are checked in test_gpu_long_barcodes.py."""
import os
import re

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import ConfigurationError, DecoderChain, binding, compile_job, workload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_binding_limit_equals_the_header():
    header = open(os.path.join(ROOT, "include", "pheniqs_b200.h")).read()
    assert binding.PHQ_MAX_NUCLEOTIDES == int(re.search(r"#define PHQ_MAX_NUCLEOTIDES (\d+)", header).group(1)) == 64


@pytest.mark.parametrize("segments", [(33,), (64,), (32, 32), (16, 16, 16, 16), (8,) * 8])
@pytest.mark.parametrize("algorithm", ["pamld", "mdd"])
def test_long_decoders_compile(algorithm, segments):
    rng = np.random.default_rng(sum(segments))
    compiled = compile_job({"sample": helpers.random_job(rng, algorithm, segments, 8, minimum_distance=3)})
    chain = DecoderChain(compiled, device=-1)
    info = chain.info[0]
    L = sum(segments)
    assert info.nucleotide_cardinality == L and info.segment_cardinality == len(segments)
    assert info.word_cardinality == (L + 15) // 16 and info.word_cardinality in (3, 4)
    assert info.quality_word_cardinality == (L + 3) // 4 and 9 <= info.quality_word_cardinality <= 16


@pytest.mark.parametrize("segments", [(65,), (33, 32)])
def test_more_than_64_nucleotides_are_refused(segments):
    rng = np.random.default_rng(65)
    with pytest.raises(ConfigurationError) as error:
        DecoderChain(compile_job({"sample": helpers.random_job(rng, "pamld", segments, 4)}), device=-1)
    assert "nucleotide cardinality 65 exceeds the 64 supported on this path" in str(error.value)


def numpy_planes(code, quality, absent):
    """The tile planes of BAM codes / Phred bytes [n, L] (include/pheniqs_b200.h phq_tile), absent positions marked."""
    n, L = code.shape
    two = np.select([code == 1, code == 2, code == 4, code == 8], [0, 1, 2, 3], -1)
    ambiguous = (two < 0) | absent
    lo = np.where(absent, 1, np.where(two < 0, 0, two & 1)).astype(np.uint64)
    hi = np.where(absent, 1, np.where(two < 0, 0, two >> 1)).astype(np.uint64)
    quality = np.where(absent, binding.PHQ_ABSENT_QUALITY, quality).astype(np.uint64)
    words = (L + 15) // 16
    bases = np.zeros((words, n), dtype=np.uint64)
    nmask = np.zeros((words, n), dtype=np.uint64)
    phred = np.zeros(((L + 3) // 4, n), dtype=np.uint64)
    for j in range(L):
        w, bit = divmod(j, 16)
        bases[w] |= (lo[:, j] << np.uint64(bit)) | (hi[:, j] << np.uint64(16 + bit))
        nmask[w] |= ambiguous[:, j].astype(np.uint64) << np.uint64(bit)
        phred[j // 4] |= quality[:, j] << np.uint64(8 * (j % 4))
    return bases.astype(np.uint32), nmask.astype(np.uint16), phred.astype(np.uint32)


def long_job(rng):
    """Long decoders with reverse complemented, knitted and short tokens: PAMLD 20 + 20 (one token reverse
    complemented), MDD 16 x 4 over two input segments, PAMLD 64 from two tokens."""
    first = helpers.random_job(rng, "pamld", (20, 20), 24, reverse=True)
    mdd = helpers.random_job(rng, "mdd", (16, 16, 16, 16), 24, minimum_distance=5)
    mdd["transform"] = {"token": ["0:0:16", "1:0:16", "0:20:36", "1:20:36"]}
    wide = helpers.random_job(rng, "pamld", (64,), 16, minimum_distance=10)
    wide["transform"] = {"token": ["0:4:36", "1:2:34"], "knit": ["0:1"]}
    return {"sample": first, "cellular": [mdd, wide]}


@pytest.mark.parametrize("short", [0.0, 0.3])
def test_pack_of_long_decoders_equals_numpy(short):
    """phq_pack of 33-64 nt decoders against the planes numpy packs from the oracle's Rule::apply: PAMLD tiles hold what a
    sequential reference thread's Observation holds (terminator and stale bytes), MDD tiles mark absent positions."""
    rng = np.random.default_rng(41)
    job = long_job(rng)
    compiled = compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], 1200, seed=5, short_fraction=short)
    chain = DecoderChain(compiled, device=-1)
    assert [info.nucleotide_cardinality for info in chain.info] == [40, 64, 64]
    tiles = chain.pack(code, quality, offset)
    port = O.PortOracle(O.compile_job(job))
    batch = O.ReadBatch(code, quality, offset)
    saw_short = False
    for k, info in enumerate(chain.info):
        L = info.nucleotide_cardinality
        want_code, want_quality, length = port.extract(k, batch)
        absent = np.zeros((batch.n_reads, L), dtype=bool)
        if info.algorithm == 1:
            starts = np.cumsum([0] + [info.segment_length[s] for s in range(info.segment_cardinality)])
            for s in range(info.segment_cardinality):
                absent[:, starts[s]:starts[s + 1]] = np.arange(info.segment_length[s])[None, :] >= length[:, s][:, None]
            saw_short = saw_short or bool(absent.any())
        bases, nmask, phred = numpy_planes(want_code, want_quality, absent)
        assert np.array_equal(tiles[k].bases[:, :batch.n_reads], bases), k
        assert np.array_equal(tiles[k].nmask[:, :batch.n_reads], nmask), k
        assert np.array_equal(tiles[k].quality[:, :batch.n_reads], phred), k
    assert saw_short == bool(short)


@pytest.mark.parametrize("bits, values", [(2, (0, 23, 37, 255)), (4, (0, 1, 2, 5, 9, 12, 17, 20, 23, 27, 30, 33, 37, 40, 41, 255))])
def test_codebook_forms_of_long_decoders(bits, values):
    """2- and 4-bit codebook indices over 16 quality words carry the Phred bytes of the byte form."""
    rng = np.random.default_rng(bits)
    job = long_job(rng)
    compiled = compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], 900, seed=7, short_fraction=0.2)
    quality = [np.array(values, dtype=np.uint8)[rng.integers(0, len(values), size=q.shape)] for q in quality]
    plain = DecoderChain(compiled, device=-1).pack(code, quality, offset)
    small = DecoderChain(compiled, device=-1).pack(code, quality, offset, quality_bits=-1)
    for k, info in enumerate(DecoderChain(compiled, device=-1).info):
        L = info.nucleotide_cardinality
        t = small[k]
        assert t.quality_bits == bits
        codebook = np.frombuffer(bytes(t.quality_codebook), dtype=np.uint8)
        per_word = 32 // bits
        index = np.stack([(t.quality[j // per_word] >> np.uint32(bits * (j % per_word))) & np.uint32((1 << bits) - 1) for j in range(L)], axis=1)
        decoded = codebook[index.astype(np.int64)]
        want = np.stack([(plain[k].quality[j // 4] >> np.uint32(8 * (j % 4))) & np.uint32(0xff) for j in range(L)], axis=1)
        assert np.array_equal(decoded, want.astype(np.uint8)), k
        assert np.array_equal(t.bases, plain[k].bases) and np.array_equal(t.nmask, plain[k].nmask)


def test_pamld_short_tokens_carry_over_calls():
    """Two phq_pack calls on one handle leave the same tiles as one call over both halves: the stale bytes of a short
    read come from the reads of the earlier call."""
    rng = np.random.default_rng(43)
    compiled = compile_job({"sample": helpers.random_job(rng, "pamld", (24, 24), 16)})
    code, quality, offset, _ = workload.synthesize(compiled, [0], 800, seed=9, short_fraction=0.4)
    whole = DecoderChain(compiled, device=-1).pack(code, quality, offset)[0]
    chain = DecoderChain(compiled, device=-1)
    half = 400
    parts = []
    for begin, end in ((0, half), (half, 800)):
        o = [x[begin:end + 1] - x[begin] for x in offset]
        c = [x[offset[i][begin]:offset[i][end]] for i, x in enumerate(code)]
        q = [x[offset[i][begin]:offset[i][end]] for i, x in enumerate(quality)]
        parts.append(chain.pack(c, q, o)[0])
    for plane in ("bases", "nmask", "quality"):
        joined = np.concatenate([getattr(p, plane)[:, :half] for p in parts], axis=1)
        assert np.array_equal(joined, getattr(whole, plane)[:, :800]), plane
