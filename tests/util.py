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
# tiny_d25 / tiny_d26: 25- and 26-dimensional features (MFCC_E_D_N_Z, MFCC_E_D_Z), 1..6 mixtures per state, NULL densities
CASES = ["tiny", "small_b100", "small_safe", "small_mp", "small_iwsp", "small_userlm", "tiny_d25", "tiny_d26"]
# tiny_dnn_odd: 117 -> 100 x 2 -> 60, widths that are not multiples of 8 (and an output width not a multiple of 4)
DNN_CASES = ["small_dnn", "small_dnn_iwsp", "tiny_dnn_odd"]
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


LOG_ZERO = np.float32(-1000000.0)


def gmm_blob(dim, counts, seed=0, null_states=(), null_gauss=(), gprune=(0, 0), cdsets=None, iwcd=(2, 3)):
    """A synthetic GMM acoustic model as a flattened-model blob dict (the layout the export plugin writes): state s has
    counts[s] mixture slots (0 allowed); every slot of the states in null_states, and the global slots in null_gauss,
    are NULL densities (valid 0, ln weight LOG_ZERO, as the reference reads an undefined <MIXTURE>,
    rdhmmdef_mpdf.c:170-193).  Means N(0,1), variances U(0.3,1.5), Dirichlet(2) weights, gconst = D ln 2pi + sum ln var.
    gprune = (method, -tmix); cdsets = list of state-id lists (pseudo-phone sets); iwcd = (method, N)."""
    rng = np.random.default_rng(seed)
    counts = np.asarray(counts, np.int64)
    S, G = len(counts), int(counts.sum())
    off = np.zeros(S + 1, np.int32)
    off[1:] = np.cumsum(counts)
    var = rng.uniform(0.3, 1.5, size=(G, dim))
    valid = np.ones(G, np.uint8)
    lnw = np.zeros(G, np.float32)
    for s in range(S):
        if counts[s]:
            lnw[off[s]:off[s + 1]] = np.log(rng.dirichlet(np.full(counts[s], 2.0)))
        if s in null_states:
            valid[off[s]:off[s + 1]] = 0
    valid[list(null_gauss)] = 0
    lnw[valid == 0] = LOG_ZERO
    b = {"gmm.n_states": np.array([S], np.int32), "gmm.dim": np.array([dim], np.int32),
         "gmm.n_gauss": np.array([G], np.int32), "gmm.max_mix": np.array([max(1, int(counts.max()))], np.int32),
         "gmm.gprune_method": np.array([gprune[0]], np.int32), "gmm.gprune_num": np.array([gprune[1]], np.int32),
         "gmm.state_off": off, "gmm.mean": rng.standard_normal((G, dim)).astype(np.float32).ravel(),
         "gmm.ivar": (1.0 / var).astype(np.float32).ravel(),
         "gmm.gconst": (dim * np.log(2 * np.pi) + np.log(var).sum(1)).astype(np.float32),
         "gmm.lnweight": lnw, "gmm.valid": valid,
         "am.iwcd_method": np.array([iwcd[0]], np.int32), "am.iwcd_nbest": np.array([iwcd[1]], np.int32)}
    if cdsets is not None:
        b["am.n_cdsets"] = np.array([len(cdsets)], np.int32)
        b["am.cd_off"] = np.concatenate([[0], np.cumsum([len(c) for c in cdsets])]).astype(np.int32)
        b["am.cd_states"] = np.concatenate([np.asarray(c, np.int32) for c in cdsets]).astype(np.int32)
        b["am.n_cdset_states"] = np.array([len(b["am.cd_states"])], np.int32)
    return b


def gmm_frames(blob, T, seed=1):
    """T feature vectors, each drawn around the mean of a random Gaussian of the model (so that every state scores over
    a wide range, near and far), with one in eight frames far from every mean."""
    rng = np.random.default_rng(seed)
    D = int(blob["gmm.dim"][0])
    mean = blob["gmm.mean"].reshape(-1, D)
    x = mean[rng.integers(len(mean), size=T)] + rng.normal(0.0, 0.7, size=(T, D))
    far = rng.random(T) < 0.125
    x[far] = rng.normal(0.0, 4.0, size=(int(far.sum()), D))
    return x.astype(np.float32)


def dnn_blob(in_dim, hidden, layers, out_dim, seed=7, w_scale=1.5):
    """A random-init DNN (full_dnn_blob's initialisation) with `layers` hidden layers of width `hidden`; layers == 0
    gives a one-layer network whose first layer is the output layer."""
    b = full_dnn_blob(seed=seed, in_dim=in_dim, hidden=hidden, layers=layers, n_out=out_dim)
    if w_scale != 1.5:
        for i in range(layers):
            b[f"dnn.l{i}.w"] = (b[f"dnn.l{i}.w"] * np.float32(w_scale / 1.5)).astype(np.float32)
    return b
