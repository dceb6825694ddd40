"""The C-ABI library: loads, exports every symbol include/pheniqs_b200.h declares, and fails loudly
(never silently falls back) where a GPU is needed. No compute calls here."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from pheniqs_b200 import ConfigurationError, DecoderChain, PheniqsError, binding, compile_job, workload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported():
    header = open(os.path.join(ROOT, "include", "pheniqs_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(phq_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations found"
    lib = C.CDLL(binding.LIBRARY_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), name + " is declared but not exported"
    assert declared == set(binding.EXPORTS)


def test_oracle_is_not_reachable_from_the_product():
    """The product path must not import, link or call anything under oracle/."""
    package = os.path.join(ROOT, "pheniqs_b200")
    for base, _, files in os.walk(package):
        for name in files:
            if name.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".cpp")):
                text = open(os.path.join(base, name)).read()
                assert "oracle" not in text.lower().replace("oracle/ (test", ""), os.path.join(base, name)


def test_compile_matches_the_restated_compile_and_the_reference_output():
    _, decoders, _ = helpers.bdggg()
    ours = compile_job(decoders)
    restated = O.compile_job(decoders)
    reference = helpers.golden("bdggg_compiled.json")
    for topic in ("sample", "cellular", "molecular"):
        a = ours[topic] if topic == "sample" else ours[topic][0]
        b = restated[topic] if topic == "sample" else restated[topic][0]
        c = reference[topic] if topic == "sample" else reference[topic][0]
        for key in ("algorithm", "index", "segment cardinality", "nucleotide cardinality", "barcode length", "noise", "confidence threshold",
                    "high quality threshold", "high quality distance threshold", "quality masking threshold", "corrected quality"):
            assert a[key] == b[key] == c[key], (topic, key)
        assert a["transform"] == c["transform"]
        assert a["undetermined"]["barcode"] == c["undetermined"]["barcode"]
        assert a["undetermined"]["concentration"] == c["undetermined"]["concentration"]
        if "codec" in c:
            assert a["random barcode probability"] == b["random barcode probability"]
            assert a["distance tolerance"] == c["distance tolerance"] == b["distance tolerance"]
            assert a["shannon bound"] == c["shannon bound"]
            assert a["barcode cardinality"] == c["barcode cardinality"]
            assert list(a["codec"].keys()) == sorted(c["codec"].keys())
            for key, record in c["codec"].items():
                assert a["codec"][key]["index"] == record["index"]
                assert a["codec"][key]["barcode"] == record["barcode"]
                assert a["codec"][key]["concentration"] == b["codec"][key]["concentration"]         # bit identical to the restatement
                assert a["codec"][key]["concentration"] == pytest.approx(record["concentration"], abs=1.1e-15)


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_compile_workloads(name):
    spec = workload.load(name)
    ours = compile_job(spec["job"])
    restated = O.compile_job(spec["job"])
    for (_, a), (_, b) in zip(workload.chain_of(ours), O.decoder_chain(restated)):
        assert a["nucleotide cardinality"] == b["nucleotide cardinality"]
        assert a["transform"]["knit"] == b["transform"]["knit"]
        if "codec" in b:
            assert a["distance tolerance"] == b["distance tolerance"]
            assert [r["concentration"] for r in a["codec"].values()] == [b["codec"][k]["concentration"] for k in a["codec"]]


def test_configuration_errors_carry_the_reference_error_code():
    rng = np.random.default_rng(0)
    good = helpers.random_job(rng, "mdd", (8,), 8, minimum_distance=3)
    cases = []
    bad = json.loads(json.dumps(good)); bad["distance tolerance"] = [3]; cases.append(bad)                      # above the Shannon bound
    bad = json.loads(json.dumps(good)); bad["transform"]["token"] = ["0:2:"]; cases.append(bad)                  # not fixed width
    bad = json.loads(json.dumps(good)); bad["noise"] = 1.5; cases.append(bad)
    bad = json.loads(json.dumps(good)); first = next(iter(bad["codec"])); bad["codec"]["dup"] = bad["codec"][first]; cases.append(bad)   # duplicate barcode
    bad = json.loads(json.dumps(good)); bad["codec"][first]["barcode"] = ["ACGT"]; cases.append(bad)              # wrong length
    bad = json.loads(json.dumps(good)); bad["algorithm"] = "bogus"; cases.append(bad)
    for decoder in cases:
        with pytest.raises(ConfigurationError) as error:
            compile_job({"sample": decoder})
        assert error.value.code == 3
    with pytest.raises(ConfigurationError):
        compile_job("{ not json")


def test_no_silent_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    compiled = compile_job(workload.load("c1")["job"])
    with pytest.raises(PheniqsError) as error:
        DecoderChain(compiled, device=0)
    assert error.value.code == 2 and "no CPU fallback" in str(error.value)
    host_only = DecoderChain(compiled, device=-1)
    tiles = host_only.allocate_tiles(4)
    with pytest.raises(PheniqsError) as error:
        host_only.decode(tiles, 4)
    assert "no CPU classification path" in str(error.value)
    # the feed-bytes and tag entry points refuse the same way; the record size is host arithmetic and still answers
    sequence = np.frombuffer(b"ACGTACGT" * 4, dtype=np.uint8)
    segments = [(sequence, sequence, None, 8), (sequence, sequence, None, 8)]
    calls = (lambda: host_only.decode_raw(segments, 4), lambda: host_only.decode_raw_tags(segments, 4),
             lambda: host_only.decode_raw(segments, 4, 0, bam=True), lambda: host_only.decode_raw(segments, 4, 0, compact=True, bam=True),
             lambda: host_only.decode_raw_tags(segments, 4, 0, bam=True), lambda: host_only.reference_power([1.0, 2.0]))
    for call in calls:
        with pytest.raises(PheniqsError) as error:
            call()
        assert "no CPU classification path" in str(error.value)
    # so does the collective (a null communicator is refused before anything else on a device handle; here the handle itself is)
    assert host_only.lib.phq_collect(host_only.handle, None, None) == binding.PHQ_INTERNAL_ERROR
    assert host_only.lib.phq_reset_accumulators_async(host_only.handle, None) == binding.PHQ_INTERNAL_ERROR
    assert host_only.tag_record_bytes() % 16 == 0 and host_only.tag_record_bytes() >= 3 + 16 + 1


@pytest.mark.parametrize("short", [0.0, 0.3])
def test_pack_reproduces_rule_apply(short):
    """phq_pack against the oracle's Rule::apply, including the short-token conventions (PAMLD: terminator +
    stale bytes of a sequential reference thread; MDD: absent positions)."""
    rng = np.random.default_rng(1)
    job = {"sample": helpers.random_job(rng, "pamld", (8, 9), 16, reverse=True),
           "molecular": [{"algorithm": "naive", "transform": {"token": ["0::4"]}}],
           "cellular": [helpers.random_job(rng, "mdd", (17,), 16, minimum_distance=3), helpers.random_job(rng, "pamld", (5,), 16, minimum_distance=2)]}
    job["cellular"][0]["transform"]["token"] = ["1:1:18"]
    compiled = compile_job(job)
    code, quality, offset, _ = workload.synthesize(compiled, [0], 1500, seed=3, short_fraction=short)
    chain = DecoderChain(compiled, device=-1)
    tiles = chain.pack(code, quality, offset)
    port = O.PortOracle(O.compile_job(job))
    batch = O.ReadBatch(code, quality, offset)
    saw_short = False
    for k, info in enumerate(chain.info):
        if not info.has_tile:
            assert tiles[k] is None
            continue
        L = info.nucleotide_cardinality
        got_code, got_quality = workload.unpack_tile(tiles[k].bases, tiles[k].nmask, tiles[k].quality, L)
        want_code, want_quality, length = port.extract(k, batch)
        offsets = np.cumsum([0] + [info.segment_length[s] for s in range(info.segment_cardinality)])
        position = np.arange(L)
        present = np.ones((batch.n_reads, L), dtype=bool)
        for s in range(info.segment_cardinality):
            inside = (position >= offsets[s]) & (position < offsets[s + 1])
            present[:, inside] = (position[inside][None, :] - offsets[s]) < length[:, s][:, None]
        if info.algorithm == 1:         # MDD: positions past the observed length are marked absent
            assert np.all(got_quality[~present] == binding.PHQ_ABSENT_QUALITY)
            assert np.array_equal(got_quality[present], want_quality[present])
            ambiguous = ~np.isin(want_code, (1, 2, 4, 8))
            assert np.array_equal(got_code[present & ~ambiguous], want_code[present & ~ambiguous])
            assert np.all(got_code[present & ambiguous] == 15)
        else:                           # PAMLD: exactly what the reference thread's scratch holds
            assert np.array_equal(got_quality, want_quality)
            ambiguous = ~np.isin(want_code, (1, 2, 4, 8))
            assert np.array_equal(got_code[~ambiguous], want_code[~ambiguous])
            assert np.all(got_code[ambiguous] == 15)
        saw_short = saw_short or bool((~present).any())
    assert saw_short == bool(short)
    # the codebook forms carry the same Phred values in fewer bytes
    smallest = DecoderChain(compiled, device=-1).pack(code, quality, offset, quality_bits=-1)
    for k, info in enumerate(chain.info):
        if not info.has_tile:
            continue
        L = info.nucleotide_cardinality
        a = workload.unpack_tile(tiles[k].bases, tiles[k].nmask, tiles[k].quality, L)
        b = workload.unpack_tile(smallest[k].bases, smallest[k].nmask, smallest[k].quality, L, smallest[k].quality_bits, smallest[k].quality_codebook)
        assert smallest[k].quality_bits in (2, 4) and smallest[k].packed_quality_words < tiles[k].packed_quality_words
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        copy = chain.pack(code, quality, offset)[k] if False else None
    with pytest.raises(ConfigurationError):
        noisy = [rng.integers(0, 40, size=q.shape).astype(np.uint8) for q in quality]
        DecoderChain(compiled, device=-1).pack(code, noisy, offset, quality_bits=2)


def test_job_file_with_import_and_base_compiles_like_the_reference(tmp_path):
    """SURVEY.md §8 f4: the reference's own test job (test/BDGGG/BDGGG_annotated.json, which imports
    BDGGG_interleave.json and inherits its decoders from the `decoder` repository through `base`) loaded with
    phq_load_job and compiled with phq_compile_job gives the decoder sections of the reference's own compile output
    (test/BDGGG/valid/compile_annotated.out -> tests/golden/bdggg_compiled.json): every key and value, barcode
    index, normalised concentration, read group ID / PU, Shannon bound and default tolerance. The keys of the
    multiplexer (output, TC, base output url: not on this path) are the only ones left out."""
    import json
    import os
    from pheniqs_b200 import compile_job, load_job
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    job = load_job(helpers.bdggg_import_documents(tmp_path))
    assert "import" not in job and job["flowcell id"] == "BDGGG" and "BDGGG_sample" in job["decoder"]
    compiled = compile_job(job)
    expected = json.load(open(os.path.join(golden, "bdggg_compiled.json")))
    outside = {"output", "TC", "base output url"}

    def same(mine, theirs, path):
        if isinstance(theirs, dict):
            assert isinstance(mine, dict), path
            assert set(mine) == set(theirs) - outside, "%s: %s" % (path, sorted(set(mine) ^ (set(theirs) - outside)))
            for key in mine:
                same(mine[key], theirs[key], path + "/" + key)
        elif isinstance(theirs, list):
            assert isinstance(mine, list) and len(mine) == len(theirs), path
            for i, (a, b) in enumerate(zip(mine, theirs)):
                same(a, b, "%s[%d]" % (path, i))
        elif isinstance(theirs, float):
            assert abs(mine - theirs) <= 1e-12 * max(1.0, abs(theirs)), path     # the golden is printed with 15 decimals
        else:
            assert mine == theirs, path
    same(compiled, expected, "")


def test_inheritance_errors():
    import pytest
    from pheniqs_b200 import ConfigurationError, compile_job
    with pytest.raises(ConfigurationError):
        compile_job({"sample": {"base": "nowhere", "transform": {"token": ["0::8"]}}, "decoder": {"a": {"noise": 0.1}}})
    with pytest.raises(ConfigurationError):
        compile_job({"decoder": {"a": {"base": "a"}}, "sample": {"base": "a", "transform": {"token": ["0::8"]}}})


def test_load_job_resolves_imports_relative_to_the_importing_file_and_visits_each_once(tmp_path):
    """Job::load_instruction_with_import (job.cpp:160-224): paths are relative to the importing document, the
    importing document wins over what it imports, later imports over earlier ones, and a document that is imported
    twice (here through a cycle) is read once."""
    import json
    from pheniqs_b200 import load_job
    (tmp_path / "lib").mkdir()
    (tmp_path / "lib" / "base.json").write_text(json.dumps({"import": ["../job.json"], "noise": 0.2, "PL": "ILLUMINA", "decoder": {"a": {"noise": 0.3}}}))
    (tmp_path / "lib" / "more.json").write_text(json.dumps({"noise": 0.4, "PM": "novaseq"}))
    (tmp_path / "job.json").write_text(json.dumps({"import": ["lib/base.json", "lib/more.json"], "decoder": {"b": {"base": "a"}}, "PL": "mine"}))
    job = load_job(str(tmp_path / "job.json"))
    assert "import" not in job
    assert job["PL"] == "mine" and job["PM"] == "novaseq" and job["noise"] == 0.4
    assert job["decoder"] == {"a": {"noise": 0.3}, "b": {"base": "a"}}


@pytest.mark.parametrize("short", [0.0, 0.01])
def test_threaded_pack_equals_the_sequential_one(short, monkeypatch):
    """phq_pack spreads large batches over threads on private Observations and falls back to the in-order pass when a
    short read makes tiles depend on earlier reads: either way the planes, the quality form and the state left behind
    are those of PHQ_PACK_THREADS=1."""
    rng = np.random.default_rng(3)
    job = {"sample": helpers.random_job(rng, "pamld", (8, 8), 24, reverse=True),
           "cellular": [helpers.random_job(rng, "mdd", (9,), 12, minimum_distance=3)]}
    job["cellular"][0]["transform"]["token"] = ["1:1:10"]
    compiled = compile_job(job)
    n = 70000
    code, quality, offset, _ = workload.synthesize(compiled, [0], n, seed=8, short_fraction=short)
    tail = [c[-400:] for c in code], [q[-400:] for q in quality]

    def run(threads):
        monkeypatch.setenv("PHQ_PACK_THREADS", str(threads))
        chain = DecoderChain(compiled, device=-1)
        first = chain.pack(code, quality, offset, quality_bits=-1)
        # a second, ragged batch packed by the same handle shows the state the first one left behind
        more_code, more_quality, more_offset, _ = workload.synthesize(compiled, [0], 500, seed=9, short_fraction=0.5)
        second = chain.pack(more_code, more_quality, more_offset)
        return first, second
    a, b = run(1), run(5)
    for x, y in zip(a[0] + a[1], b[0] + b[1]):
        if x is None:
            assert y is None
            continue
        assert x.quality_bits == y.quality_bits and bytes(x.quality_codebook) == bytes(y.quality_codebook)
        assert np.array_equal(x.bases, y.bases) and np.array_equal(x.nmask, y.nmask) and np.array_equal(x.quality, y.quality)


def test_host_entry_points_report_status_and_message():
    """The status and message of the entry points that need no device, read where phq_last_error finds them."""
    lib = binding.library()
    out = C.c_void_p(1)

    def global_error():
        return lib.phq_last_global_error().decode()

    assert lib.phq_compile_job(b"{ not json", C.byref(out)) == binding.PHQ_CONFIGURATION_ERROR
    assert global_error().startswith("Configuration error : ")
    assert lib.phq_compile_job(None, C.byref(out)) == binding.PHQ_INTERNAL_ERROR
    assert global_error() == "Internal error : null argument"

    job = json.dumps(compile_job(workload.load("c1")["job"])).encode()
    assert lib.phq_adjust_job(job, b"{ not json", 6, C.byref(out)) == binding.PHQ_CONFIGURATION_ERROR
    assert global_error().startswith("Configuration error : ")

    assert lib.phq_load_job(os.path.join(ROOT, "no", "such", "job.json").encode(), C.byref(out)) == binding.PHQ_CONFIGURATION_ERROR
    assert global_error().startswith("Configuration error : unable to read instruction file from ")
    assert out.value is None

    handle = C.c_void_p(1)
    assert lib.phq_create(b"{ not json", -1, C.byref(handle)) == binding.PHQ_CONFIGURATION_ERROR
    assert global_error().startswith("Configuration error : ")
    assert handle.value is None

    tiles = (binding.Tile * 1)()
    assert lib.phq_pack(None, 0, 0, None, None, None, tiles) == binding.PHQ_INTERNAL_ERROR
    assert global_error() == "Internal error : null handle"

    assert lib.phq_create(job, -1, C.byref(handle)) == binding.PHQ_OK
    try:
        assert lib.phq_tag_record_bytes(handle, None) == binding.PHQ_INTERNAL_ERROR
        assert lib.phq_last_error(handle).decode() == "Internal error : illegal argument"
    finally:
        lib.phq_destroy(handle)
