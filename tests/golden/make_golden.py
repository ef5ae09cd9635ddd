"""Regenerate the committed golden fixtures by running the UNMODIFIED compiled reference
(oracle/_ref/jref, built by oracle/Makefile from /root/reference) on seeded synthetic models.

    python tests/golden/make_golden.py [case ... | sweep | host]

Each fixture directory holds
    model.jb2m  the reference's loaded models, flattened by the export plugin
    out.jrf     reference outputs: [T x S] state scores, word trellis, pass-1 best
    feats.npz   the input feature matrices (u0, u1, ...)
    meta.json   the jconf-style options used

The sweep cases (tests/util.py SWEEP, GRAMMAR_SWEEP) go to sweep/<case>/ in the compact form tests/util.py SweepGolden
reads: model entries that no fixture above holds (model_delta.npz), trellis per utterance (out.npz), and in meta.json
the source of every model entry, digests of the inputs and of the state scores, and the pass-1 results.  host/ holds
what the stock host prints or decodes where the GPU boundary tests compare with it.
"""
import json
import os
import shutil
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from julius_b200 import refdump, synth  # noqa: E402
from oracle import ffi, fixtures  # noqa: E402
from util import (GRAMMAR_SWEEP, GRAMMAR_SWEEP_FRAMES, SWEEP, SWEEP_FRAMES, SWEEP_NOISE_UTTS, SWEEP_UTTS,  # noqa: E402
                  Golden, digest, sweep_dir)

HERE = os.path.dirname(os.path.abspath(__file__))

# grammar (DFA) mode cases: the LM is the synthetic finite-state grammar of julius_b200.synth.write_grammar
GRAMMAR_CASES = {"small_dfa"}

CASES = {
    # name: (preset, n_utts, n_frames, noise_utts, extra args)
    "tiny": ("tiny", 2, 150, 0, []),
    # the other MFCC sizes the GMM scorer is built for (25 = MFCC_E_D_N_Z, 26 = MFCC_E_D_Z), 1..6 mixtures per state and
    # a few NULL densities
    "tiny_d25": ("tiny_d25", 2, 150, 0, []),
    "tiny_d26": ("tiny_d26", 2, 150, 0, []),
    "small_b100": ("small", 2, 200, 1, ["-b", "100"]),
    "small_safe": ("small", 1, 150, 0, ["-gprune", "safe", "-tmix", "2", "-b", "60", "-iwcd1", "max"]),
    # multipath tree (non-emitting word-begin/word-end nodes), beam.c:2752-2828
    "small_mp": ("small", 2, 200, 1, ["-multipath", "-b", "120"]),
    # inter-word short pause (tee model => multipath by necessity), BASELINE configs[4] flavour
    "small_iwsp": ("small_sp", 2, 200, 1, ["-iwsp", "-iwcd1", "max", "-b", "150"]),
    # 40 transparent (filler) words: last_cword differs from the last word, beam.c:2300-2330
    "small_tr": ("small_tr", 2, 200, 1, ["-b", "100"]),
    # phonetic tied-mixture AM (<TMIX> codebooks, calc_tied_mix.c), flattened by the exporter; safe pruning
    "small_tm": ("small_tm", 2, 200, 1, ["-gprune", "safe", "-tmix", "4", "-b", "100"]),
    # grammar mode (category tree + category-pair constraint, beam.c:1669-1760, :2404-2455), BASELINE configs[0] flavour
    "small_dfa": ("small", 2, 200, 1, ["-b", "80", "-penalty1", "-1.0"]),
    # user-defined LM functions on top of the N-gram (-userlm, wchmm.h:274-276; registered by the driver, JREF_USERLM=1)
    "small_userlm": ("small", 2, 200, 1, ["-userlm", "-b", "100"]),
}
# cases that need something in the driver's environment
CASE_ENV = {"small_userlm": {"JREF_USERLM": "1"}}
# DNN-HMM: (preset, DnnConfig kwargs, n_utts, n_frames, extra args)
DNN_CASES = {
    "small_dnn": ("small", dict(in_dim=120, feature_len=40, context_len=3, hidden=128, layers=3), 2, 150, ["-b", "150"]),
    # configs[4] flavour: DNN-HMM on a multipath tree with -iwsp and a wide beam
    "small_dnn_iwsp": ("small_sp", dict(in_dim=120, feature_len=40, context_len=3, hidden=128, layers=3), 2, 150,
                       ["-iwsp", "-iwcd1", "max", "-b", "600"]),
    # widths off the GPU kernel's tiles: 112 inputs, 104 hidden (ends inside a 32-column epilogue chunk), 60 outputs (not a
    # multiple of 4).  Widths that are not multiples of 8 cannot be pinned here: the reference's x86 FMA GEMV
    # (calc_dnn_fma.c:18-95) runs over in/8 blocks of 8 and silently drops the remainder, its AVX and SSE variants refuse
    # such layers (calc_dnn.c:395-401).  tests/test_scoring_reference.py checks them against float64 instead.
    "tiny_dnn_odd": ("tiny", dict(in_dim=112, feature_len=28, context_len=4, hidden=104, layers=2), 2, 150, ["-b", "150"]),
}


def main():
    ffi.build()
    only = set(sys.argv[1:])
    for name, (preset, nu, nf, nn, extra) in CASES.items():
        if only and name not in only:
            continue
        tmp = tempfile.mkdtemp(prefix="jb200_golden_")
        m, files, dump, out = fixtures.make_fixture(preset, tmp, n_utts=nu, n_frames=nf, noise_utts=nn, extra_args=extra,
                                                    grammar=name in GRAMMAR_CASES, env_extra=CASE_ENV.get(name))
        dst = os.path.join(HERE, name)
        os.makedirs(dst, exist_ok=True)
        shutil.copy(os.path.join(tmp, "model.jb2m"), dst)
        shutil.copy(dump, os.path.join(dst, "out.jrf"))
        feats = {f"u{i}": synth.read_htk_param(fn)[0] for i, fn in enumerate(files)}
        np.savez_compressed(os.path.join(dst, "feats.npz"), **feats)
        with open(os.path.join(dst, "meta.json"), "w") as f:
            json.dump({"preset": preset, "extra_args": extra, "n_utts": len(files), "grammar": name in GRAMMAR_CASES, "env": CASE_ENV.get(name, {}),
                       "summary": out.strip().splitlines()[-1]}, f, indent=1)
        shutil.rmtree(tmp)
        print(name, "->", dst)
    for name, (preset, dkw, nu, nf, extra) in DNN_CASES.items():
        if only and name not in only:
            continue
        tmp = tempfile.mkdtemp(prefix="jb200_golden_")
        cfg = synth.SynthConfig.preset(preset)
        m = synth.SynthModel(cfg)
        m.write_all(tmp)
        dc = synth.DnnConfig(**dkw)
        synth.write_dnn(tmp, cfg.n_states, dc)
        rng = np.random.default_rng(17)
        files = []
        for u in range(nu):
            fn = os.path.join(tmp, f"u{u}.mfc")
            synth.write_htk_param(fn, synth.sample_dnn_input(rng, nf, dc.in_dim), parmkind=synth.PARMKIND_USER)
            files.append(fn)
        dump, out = ffi.run_ref(tmp, files, extra_args=["-dnnconf", "dnnconf"] + extra, export=os.path.join(tmp, "model.jb2m"))
        dst = os.path.join(HERE, name)
        os.makedirs(dst, exist_ok=True)
        shutil.copy(os.path.join(tmp, "model.jb2m"), dst)
        shutil.copy(dump, os.path.join(dst, "out.jrf"))
        np.savez_compressed(os.path.join(dst, "feats.npz"), **{f"u{i}": synth.read_htk_param(fn)[0] for i, fn in enumerate(files)})
        with open(os.path.join(dst, "meta.json"), "w") as f:
            json.dump({"preset": preset, "dnn": dkw, "extra_args": extra, "n_utts": len(files), "summary": out.strip().splitlines()[-1]}, f, indent=1)
        shutil.rmtree(tmp)
        print(name, "->", dst)
    if not only or "sweep" in only:
        for preset, extra in SWEEP:
            make_sweep_case(preset, extra, False)
        for extra in GRAMMAR_SWEEP:
            make_sweep_case("small", extra, True)
    if not only or "host" in only:
        make_host_cases()


def pin(dst, dump, feats=None, **meta):
    """The reference's pass-1 results in the compact form tests/util.py load_pinned reads: the trellis of every
    utterance (out.npz), and in meta.json digests of the state scores (and of the inputs), words, status and score."""
    os.makedirs(dst, exist_ok=True)
    utts = refdump.load_refdump(dump)
    np.savez_compressed(os.path.join(dst, "out.npz"), **{f"u{i}": u.atoms for i, u in enumerate(utts)})
    meta["utts"] = [dict(({"feats_sha256": digest(feats[i])} if feats is not None else {}), outprob_shape=list(u.outprob.shape),
                         outprob_sha256=digest(u.outprob), words=list(u.words), status=int(u.status), score=float(np.float32(u.score)))
                    for i, u in enumerate(utts)]
    with open(os.path.join(dst, "meta.json"), "w") as f:
        json.dump(meta, f, indent=1)


def host_inputs(case, d):
    """the model text files and input files of a golden case, for a run of the stock host (tests/test_gpu_host.py)"""
    g = Golden(case)
    synth.SynthModel(synth.SynthConfig.preset(g.meta["preset"])).write_all(d)
    files = []
    for i, x in enumerate(g.feats):
        files.append(os.path.join(d, f"u{i}.mfc"))
        synth.write_htk_param(files[-1], x)
    return g, files


def make_host_cases():
    """What the stock host prints or dumps where tests/test_gpu_host.py holds the host with the GPU code against it, and
    the reference's decode of the tri20k workload's probe utterance (tests/test_gpu_full.py)."""
    dst = os.path.join(HERE, "host")
    os.makedirs(dst, exist_ok=True)
    for case, extra, env, tag, prefix in (
            ("small_b100", [], {}, "two_pass", "JREF_RESULT"), ("small_iwsp", [], {}, "two_pass", "JREF_RESULT"),
            ("small_b100", ["-progout", "-proginterval", "100"], {"JREF_INTERIM": "1"}, "interim", "JREF_INTERIM"),
            ("small_mp", ["-progout", "-proginterval", "100"], {"JREF_INTERIM": "1"}, "interim", "JREF_INTERIM")):
        tmp = tempfile.mkdtemp(prefix="jb200_golden_")
        g, files = host_inputs(case, tmp)
        _, out = ffi.run_ref(tmp, files, extra_args=g.meta["extra_args"] + extra, two_pass=tag == "two_pass", env_extra=env)
        with open(os.path.join(dst, f"{case}_{tag}.txt"), "w") as f:
            f.write("".join(ln + "\n" for ln in out.splitlines() if ln.startswith(prefix)))
        shutil.rmtree(tmp)
    tmp = tempfile.mkdtemp(prefix="jb200_golden_")
    g, files = host_inputs("tiny", tmp)
    dump, _ = ffi.run_ref(tmp, files, extra_args=["-gprune", "none"])
    pin(os.path.join(dst, "tiny_gprune_none"), dump, g.feats, extra_args=["-gprune", "none"])
    shutil.rmtree(tmp)
    from julius_b200 import workload
    if not workload.ensure("tri20k"):
        raise RuntimeError("workloads/tri20k could not be built")
    x, _ = synth.read_htk_param(workload.path("tri20k", "probe.mfc"))
    pin(os.path.join(dst, "tri20k_probe"), workload.path("tri20k", "probe.jrf"), [x])
    print("host ->", dst)


def make_sweep_case(preset, extra, grammar):
    tmp = tempfile.mkdtemp(prefix="jb200_golden_")
    m, files, dump, out = fixtures.make_fixture(preset, tmp, n_utts=SWEEP_UTTS, noise_utts=SWEEP_NOISE_UTTS, extra_args=extra,
                                                n_frames=GRAMMAR_SWEEP_FRAMES if grammar else SWEEP_FRAMES, grammar=grammar)
    blob = refdump.load_blob(os.path.join(tmp, "model.jb2m"))
    # the committed fixtures, the one sharing the most entries with this model first
    fixed = {c: refdump.load_blob(os.path.join(HERE, c, "model.jb2m")) for c in sorted(CASES) + sorted(DNN_CASES)}

    def same(a, b):
        return b is not None and a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))
    order = sorted(fixed, key=lambda c: -sum(same(v, fixed[c].get(k)) for k, v in blob.items()))
    src = {}
    for k, v in blob.items():
        src.setdefault(next((c for c in order if same(v, fixed[c].get(k))), ""), []).append(k)
    dst = sweep_dir(preset, extra, grammar)
    os.makedirs(dst, exist_ok=True)
    np.savez_compressed(os.path.join(dst, "model_delta.npz"), **{k: blob[k] for k in src.get("", [])})
    feats = [synth.read_htk_param(fn)[0] for fn in files]
    assert all(np.array_equal(x, y) for x, y in zip(feats, fixtures.sample_inputs(
        m, SWEEP_UTTS, GRAMMAR_SWEEP_FRAMES if grammar else SWEEP_FRAMES, noise_utts=SWEEP_NOISE_UTTS, grammar=grammar)))
    pin(dst, dump, feats, preset=preset, extra_args=extra, grammar=grammar, summary=out.strip().splitlines()[-1],
        model={c: " ".join(keys) for c, keys in src.items()})
    shutil.rmtree(tmp)
    print(" ".join([preset] + extra), "->", dst)


if __name__ == "__main__":
    main()
