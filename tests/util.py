import hashlib
import json
import os
import re
from types import SimpleNamespace

import numpy as np

from julius_b200 import desc, refdump, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
# small_userlm: user-defined LM functions (-userlm) on top of the N-gram, tabulated by the exporter
CASES = ["tiny", "small_b100", "small_safe", "small_mp", "small_iwsp", "small_userlm"]
DNN_CASES = ["small_dnn", "small_dnn_iwsp"]
# pinned on the CPU only so far (the GPU suite does not run them yet)
ORACLE_ONLY_CASES = ["small_tr", "small_tm", "small_dfa"]

# jconf options beyond the golden cases above, pinned against the compiled reference in tests/golden/sweep
SWEEP = [
    ("small", ["-b", "80", "-iwcd1", "avg"]),
    ("small", ["-b", "80", "-iwcd1", "best", "5"]),
    ("small", ["-b", "120", "-lmp", "12.0", "-3.0"]),
    ("small", ["-b", "200", "-bs", "60"]),                       # score-envelope pruning (SCORE_PRUNING, beam.c:2718-2730)
    ("small", ["-multipath", "-b", "150", "-bs", "80"]),
    ("small_sp", ["-iwsp", "-b", "100", "-bs", "50", "-iwcd1", "avg"]),
    ("small", ["-gprune", "heuristic", "-tmix", "2", "-b", "90"]),
    ("small_tr", ["-multipath", "-b", "90"]),                    # transparent words on the multipath tree
    ("small_tm", ["-gprune", "none", "-b", "100"]),              # tied-mixture codebooks, calc_tied_mix.c:161-248
    ("small_tm", ["-gprune", "safe", "-tmix", "2", "-b", "80", "-multipath"]),
]
# grammar (DFA) mode on the "small" preset
GRAMMAR_SWEEP = [["-b", "100"], ["-b", "60", "-penalty1", "-2.5", "-iwcd1", "max"], ["-b", "150", "-multipath", "-penalty1", "1.5"]]
# how a sweep case was sampled: utterances, noise utterances, frames (make_golden.py runs the reference on exactly these)
SWEEP_UTTS, SWEEP_NOISE_UTTS, SWEEP_FRAMES, GRAMMAR_SWEEP_FRAMES = 2, 1, 150, 180


def digest(a: np.ndarray) -> str:
    """sha256 of an array's float32 bits: identical digests <=> bit-identical arrays"""
    return hashlib.sha256(np.ascontiguousarray(a, "<f4").tobytes()).hexdigest()


def sweep_dir(preset: str, extra: list, grammar: bool = False) -> str:
    name = re.sub(r"[^A-Za-z0-9.]+", "_", " ".join([preset] + list(extra)).replace("-", " ")).strip("_")
    return os.path.join(GOLDEN, "sweep", ("dfa_" if grammar else "") + name)


def load_pinned(d: str, feats=None):
    """meta.json and out.npz of a directory written by tests/golden/make_golden.py pin(): (meta, utterances), each
    utterance with the reference's trellis (atoms), words, status and score, and the digest of its state scores.  With
    feats given, every input must match the digest of the one the reference decoded."""
    meta = json.load(open(os.path.join(d, "meta.json")))
    out = np.load(os.path.join(d, "out.npz"))
    assert feats is None or len(feats) == len(meta["utts"]), "the inputs are not the ones the reference decoded"
    utts = []
    for i, u in enumerate(meta["utts"]):
        if feats is not None:
            assert digest(feats[i]) == u["feats_sha256"], f"input {i} differs from the one the reference decoded"
        utts.append(SimpleNamespace(atoms=out[f"u{i}"], words=u["words"], status=u["status"], score=np.float32(u["score"]),
                                    outprob_shape=tuple(u["outprob_shape"]), outprob_sha256=u["outprob_sha256"]))
    return meta, utts


class SweepGolden:
    """A sweep case as the compiled reference decoded it (written by tests/golden/make_golden.py).  To stay small on disk:
    the flattened model is kept as the entries that no committed golden model holds (meta "model" maps a golden case,
    or "" for model_delta.npz, to the entries taken from it); the inputs are regenerated from their seed and must match
    the recorded digests; the reference's state scores are kept as digests, its trellis and pass-1 result in full."""

    def __init__(self, preset: str, extra: list, grammar: bool = False):
        from oracle import fixtures
        d = sweep_dir(preset, extra, grammar)
        m = synth.SynthModel(synth.SynthConfig.preset(preset))
        self.feats = fixtures.sample_inputs(m, SWEEP_UTTS, GRAMMAR_SWEEP_FRAMES if grammar else SWEEP_FRAMES,
                                            noise_utts=SWEEP_NOISE_UTTS, grammar=grammar)
        self.meta, self.utts = load_pinned(d, self.feats)
        delta = np.load(os.path.join(d, "model_delta.npz"))
        self.blob = {}
        for src, keys in self.meta["model"].items():
            model = refdump.load_blob(os.path.join(GOLDEN, src, "model.jb2m")) if src else delta
            for key in keys.split():
                self.blob[key] = model[key]
        self.ds = desc.Descriptors(self.blob)


class Golden:
    def __init__(self, name):
        d = os.path.join(GOLDEN, name)
        self.dir = d
        self.blob = refdump.load_blob(os.path.join(d, "model.jb2m"))
        self.ds = desc.Descriptors(self.blob)
        self.utts = refdump.load_refdump(os.path.join(d, "out.jrf"))
        z = np.load(os.path.join(d, "feats.npz"))
        self.feats = [z[f"u{i}"] for i in range(len(self.utts))]
        self.meta = json.load(open(os.path.join(d, "meta.json")))


def atoms_equal(a, b):
    """bit-exact comparison of two structured atom arrays (wid, begin, end, backscore, lscore, last)."""
    if len(a) != len(b):
        return False, f"atom count {len(a)} != {len(b)}"
    for k in ("wid", "begin", "end", "last"):
        if not np.array_equal(a[k], b[k]):
            i = int(np.nonzero(a[k] != b[k])[0][0])
            return False, f"field {k} differs first at atom {i}: {a[i]} vs {b[i]}"
    for k in ("backscore", "lscore"):
        if not np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)):
            i = int(np.nonzero(a[k].view(np.uint32) != b[k].view(np.uint32))[0][0])
            return False, f"field {k} differs (bits) first at atom {i}: {a[i]} vs {b[i]}"
    return True, ""


def rel_err(a, b, floor=1.0):
    """|a-b| / max(|a|,|b|,floor): the relative criterion with an absolute floor (SURVEY 7, hard parts)."""
    return np.abs(a - b) / np.maximum(np.maximum(np.abs(a), np.abs(b)), floor)


def full_dnn_blob(seed=3, in_dim=528, hidden=2048, layers=7, n_out=3000):
    """A random-init DNN of the BASELINE configs[3] shape (528 = 48 x 11 inputs, 7 x 2048 logistic, n_out states) as a
    flattened-model blob dict, with the initialisation of julius_b200.synth.write_dnn (W ~ N(0, 1.5/sqrt(in)), output
    layer 3/sqrt(in), b ~ N(0, 0.1), Dirichlet priors stored as log10, calc_dnn.c:699-703)."""
    rng = np.random.default_rng(seed)
    dims = [in_dim] + [hidden] * layers + [n_out]
    b = {"dnn.n_layers": np.array([layers + 1], np.int32), "dnn.in_dim": np.array([in_dim], np.int32),
         "dnn.out_dim": np.array([n_out], np.int32), "gmm.n_states": np.array([n_out], np.int32)}
    for i in range(layers + 1):
        scale = (3.0 if i == layers else 1.5) / np.sqrt(dims[i])
        b[f"dnn.l{i}.in"] = np.array([dims[i]], np.int32)
        b[f"dnn.l{i}.out"] = np.array([dims[i + 1]], np.int32)
        b[f"dnn.l{i}.w"] = (rng.standard_normal((dims[i + 1], dims[i])) * scale).astype(np.float32).ravel()
        b[f"dnn.l{i}.b"] = (rng.standard_normal(dims[i + 1]) * 0.1).astype(np.float32)
    prior = rng.dirichlet(np.full(n_out, 5.0))
    b["dnn.state_prior"] = np.log10(prior).astype(np.float32)
    return b
