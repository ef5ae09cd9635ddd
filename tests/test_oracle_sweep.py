"""CPU: the restatement against the compiled reference across jconf options beyond the committed golden cases.  The
reference's state scores, word trellis and pass-1 result for each case are pinned in tests/golden/sweep (written by
tests/golden/make_golden.py from oracle/_ref/jref); the restatement must give bit-identical state scores and an
identical word trellis."""
import os

import numpy as np
import pytest

from util import GRAMMAR_SWEEP, ROOT, SWEEP, SweepGolden, atoms_equal, digest

JREF = os.path.join(ROOT, "oracle", "_ref", "jref")


def _check_scores_and_trellis(g, oracle_lib):
    for u, x in zip(g.utts, g.feats):
        sc = oracle_lib.gmm_score(g.ds, x)
        assert sc.shape == u.outprob_shape
        assert digest(sc) == u.outprob_sha256, "state scores differ from the reference"
        r = oracle_lib.beam_decode(g.ds, sc)           # bit-identical to the reference's own score matrix
        ok, why = atoms_equal(r["atoms"], u.atoms)
        assert ok, why
        assert r["words"] == u.words and r["status"] == u.status
        assert np.float32(r["score"]) == u.score


@pytest.mark.parametrize("extra", GRAMMAR_SWEEP, ids=[" ".join(e) for e in GRAMMAR_SWEEP])
def test_grammar_mode_restatement_equals_compiled_reference(extra, oracle_lib):
    """Grammar (DFA) recognition: category tree, category-pair constraint, insertion penalty, all sentence-initial
    words alive at frame 0, best atom of the last frame as the pass-1 result (beam.c:1669-1760, :2404-2455, :435-458)."""
    g = SweepGolden("small", extra, grammar=True)
    assert g.ds.tree.lm_type == 1 and g.ds.tree.n_shared == 0 and g.ds.tree.n_init >= 1
    _check_scores_and_trellis(g, oracle_lib)


@pytest.mark.skipif(not os.path.exists(JREF), reason="compiled reference (oracle/_ref/jref) not present")
def test_tied_mixture_with_history_dependent_pruning_is_refused(tmp_path):
    """-gprune beam (the default) on a tied-mixture AM seeds each codebook's pruning with the previous frame's best
    ids, so its scores depend on which frames the search evaluated; the exporter must refuse rather than approximate."""
    from oracle import fixtures
    with pytest.raises(RuntimeError):
        fixtures.make_fixture("small_tm", str(tmp_path), n_utts=1, n_frames=50, extra_args=["-b", "60"])


@pytest.mark.parametrize("preset,extra", SWEEP, ids=[" ".join([p] + e) for p, e in SWEEP])
def test_restatement_equals_compiled_reference(preset, extra, oracle_lib):
    _check_scores_and_trellis(SweepGolden(preset, extra), oracle_lib)
