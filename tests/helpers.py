"""Shared test helpers: fixtures on disk, job builders, comparisons. Test infrastructure only."""
import json
import os

import numpy as np

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bdggg():
    z = np.load(os.path.join(GOLDEN, "bdggg_reads.npz"))
    batch = O.ReadBatch([z["code%d" % s] for s in range(3)], [z["quality%d" % s] for s in range(3)], [z["offset%d" % s] for s in range(3)], z["qcfail"])
    job = json.load(open(os.path.join(GOLDEN, "bdggg_job.json")))
    keep = np.ones(batch.n_reads, dtype=bool)
    for i in range(1, 3):                               # TranscodingThread::filter_input, transcode.h:193-200
        keep &= (batch.offset[i][1:] - batch.offset[i][:-1]) >= job["min input length"][i]
    expected = json.load(open(os.path.join(GOLDEN, "bdggg_expected.json")))
    names = list(z["name"][keep])
    assert names == [e["name"] for e in expected]
    decoders = {k: job[k] for k in ("sample", "molecular", "cellular")}
    return batch.select(keep), decoders, expected


def bdggg_import_documents(directory):
    """Write the job documents of the reference's annotated test (import + base inheritance) into `directory` under the
    file names their import list uses; returns the path of the top document."""
    documents = json.load(open(os.path.join(GOLDEN, "bdggg_import_documents.json")))
    for name, document in documents.items():
        with open(os.path.join(str(directory), name), "w") as f:
            json.dump(document, f)
    return os.path.join(str(directory), "BDGGG_annotated.json")


def golden(name):
    return json.load(open(os.path.join(GOLDEN, name)))


def error_tag(confidence):
    """Read::flush (read.h:187-199) + SAM float formatting (%g of a float32)."""
    if not (0 < confidence < 1):
        return None
    return "%g" % np.float32(1.0 - confidence)


def random_job(rng, algorithm="pamld", segments=(8,), n_barcodes=24, reverse=False, noise=0.05, threshold=0.9, minimum_distance=3, **extra):
    """A decoder over one input segment per barcode segment with a random codec of the given minimum distance."""
    total = sum(segments)
    words = []
    while len(words) < n_barcodes:
        w = rng.integers(0, 4, size=total)
        if all((w != v).sum() >= minimum_distance for v in words):
            words.append(w)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    codec = {}
    for i, w in enumerate(words):
        text = letters[w].tobytes().decode()
        parts, at = [], 0
        for n in segments:
            parts.append(text[at:at + n])
            at += n
        codec["@%03d" % i] = {"barcode": parts, "concentration": float(rng.integers(1, 5))}
    tokens = ["%d:%d:%d" % (i, 2, 2 + n) for i, n in enumerate(segments)]
    decoder = {"algorithm": algorithm, "transform": {"token": tokens}, "codec": codec, "noise": noise, "confidence threshold": threshold}
    if reverse:
        decoder["transform"]["knit"] = ["~%d" % i for i in range(len(segments))]
    decoder.update(extra)
    return decoder


def grid_job(la, lb, ka, kb, fill, equal):
    """A dual index PAMLD job: ka distinct first words of la nt times kb distinct second words of lb nt, each
    combination present with probability `fill`, under equal priors or priors of 1 to 3."""
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


def compare_pamld(got, expected_index, expected_distance, expected_confidence, label=""):
    assert np.array_equal(got["index"], expected_index), label + " barcode index"
    assert np.array_equal(got["distance"], expected_distance), label + " distance"
    ok = expected_confidence > 0
    assert np.array_equal(got["confidence"] > 0, ok), label + " confidence support"
    # posterior: |ln conf - ln conf_ref| <= 1e-6  (north_star tolerance, log space)
    assert np.all(np.abs(np.log(got["confidence"][ok]) - np.log(expected_confidence[ok])) <= 1e-6), label + " ln confidence"
    # error probability 1 - conf, where conf < 1: relative 1e-6, floored at 4 ulp of 1.0 because the
    # reference forms it as 1.0 - conf in f64 (read.h:189) and that difference is quantised at 2^-53
    e_got = 1.0 - got["confidence"][ok]
    e_ref = 1.0 - expected_confidence[ok]
    excess = np.abs(e_got - e_ref) - (1e-6 * e_ref + 4 * 2.0 ** -53)
    worst = int(np.argmax(excess)) if excess.size else 0
    assert np.all(excess <= 0), "%s error probability: %d reads out of tolerance, worst read %d: got %.17g expected %.17g (difference %.3g = %.2f x 2^-53)" % (
        label, int((excess > 0).sum()), int(np.nonzero(ok)[0][worst]), e_got[worst], e_ref[worst], e_got[worst] - e_ref[worst], (e_got[worst] - e_ref[worst]) * 2.0 ** 53)
