"""GPU: the CUDA path against the compiled reference across jconf options beyond the committed golden cases --
the device-side twin of tests/test_oracle_sweep.py.  Each case's inputs go through K1 + K3 and must give the state
scores (bit for bit) and the word trellis the compiled reference produced for them (tests/golden/sweep).  Covers
-iwcd1 avg / best N, -lmp, score-envelope pruning (-bs), -gprune heuristic, -iwsp, transparent words, flattened
tied-mixture codebooks and DFA grammars on the device."""
import numpy as np
import pytest

from julius_b200 import capi
from util import GRAMMAR_SWEEP, SWEEP, SweepGolden, atoms_equal, digest

pytestmark = pytest.mark.gpu


def _check(r, u):
    ok, why = atoms_equal(r["atoms"], u.atoms)
    assert ok, why
    assert r["words"] == u.words and r["status"] == u.status and r["overflow"] == 0
    assert np.float32(r["score"]) == u.score


def _check_case(g):
    am = capi.GmmScorer(g.ds, mode=capi.GMM_EXACT)
    for u, x in zip(g.utts, g.feats):
        sc = am.score(x)
        assert digest(sc) == u.outprob_sha256, "state scores differ from the reference"
    dec = capi.Decoder(g.ds, am, max_utts=4, max_frames=2048)
    for r, u in zip(dec.decode(g.feats), g.utts):
        _check(r, u)


@pytest.mark.parametrize("preset,extra", SWEEP, ids=[" ".join([p] + e) for p, e in SWEEP])
def test_gpu_path_equals_compiled_reference(preset, extra):
    _check_case(SweepGolden(preset, extra))


# the GPU beam takes grammars on normal trees only (creation refuses -multipath loudly, tested in test_gpu_beam.py)
@pytest.mark.parametrize("extra", [e for e in GRAMMAR_SWEEP if "-multipath" not in e], ids=lambda e: " ".join(e))
def test_gpu_grammar_mode_equals_compiled_reference(extra):
    _check_case(SweepGolden("small", extra, grammar=True))
