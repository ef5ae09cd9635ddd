"""Fixture generation through the compiled reference -- TEST INFRASTRUCTURE.

make_fixture() writes a synthetic model (julius_b200.synth), samples utterances, runs the
UNMODIFIED reference (oracle/_ref/jref) on them with the export plugin loaded, and leaves
  model.jb2m   flattened model (what the GPU path and the restatement consume)
  out.jrf      reference outputs (state scores, trellis, pass-1 best[, per-frame tokens])
  u*.mfc       HTK parameter files
in `outdir`.  Needs /root/reference only to have been compiled (oracle/_ref travels).
"""
from __future__ import annotations

import os

import numpy as np

from julius_b200 import synth
from . import ffi


def make_fixture(preset, outdir: str, n_utts: int = 2, n_frames: int = 200, seed: int = 11,
                 extra_args: list = (), tokens: bool = False, noise_utts: int = 0, model=None, grammar: bool = False,
                 env_extra: dict | None = None):
    """grammar=True: decode with the synthetic finite-state grammar (-dfa/-v) instead of the N-gram; the sampled
    utterances then follow sentences of that grammar."""
    cfg = synth.SynthConfig.preset(preset) if isinstance(preset, str) else preset
    m = model if model is not None else synth.SynthModel(cfg)
    if model is None or not os.path.exists(os.path.join(outdir, "hmmdefs")):
        m.write_all(outdir)
    files = []
    lm_args = None
    if grammar:
        g = m.write_grammar(outdir)
        lm_args = ["-dfa", os.path.basename(g["dfa"]), "-v", os.path.basename(g["dict"])]
    for u, x in enumerate(sample_inputs(m, n_utts, n_frames, seed, noise_utts, grammar)):
        fn = os.path.join(outdir, f"u{u}.mfc" if u < n_utts else f"n{u - n_utts}.mfc")
        synth.write_htk_param(fn, x)
        files.append(fn)
    with open(os.path.join(outdir, "list.txt"), "w") as f:
        f.write("\n".join(files) + "\n")
    dump, out = ffi.run_ref(outdir, files, extra_args=extra_args, export=os.path.join(outdir, "model.jb2m"),
                            tokens=tokens, lm_args=lm_args, env_extra=env_extra)
    return m, files, dump, out


def sample_inputs(m, n_utts: int, n_frames: int, seed: int = 11, noise_utts: int = 0, grammar: bool = False) -> list:
    """The feature matrices make_fixture() decodes: n_utts sampled utterances (sentences of the synthetic grammar when
    grammar=True), then noise_utts noise utterances, all drawn from one generator seeded with `seed`."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_utts):
        ws = m.sample_grammar_sentence(rng, max(2, n_frames // 45)) if grammar else None
        out.append(m.sample_utterance(rng, n_frames, word_seq=ws)[0])
    for _ in range(noise_utts):
        out.append(m.sample_noise(rng, n_frames))
    return out
