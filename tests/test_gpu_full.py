"""GPU, BASELINE.json full size (3000 states x 16 mix x 39, 20k-word tree, beam 800): the CUDA path
vs the CPU restatement on the same seeded inputs, plus size-independent properties."""
import os

import numpy as np
import pytest

from julius_b200 import capi, desc, workload
from util import GOLDEN, atoms_equal, load_pinned

pytestmark = pytest.mark.gpu

NAME = "tri20k"


@pytest.fixture(scope="module")
def full():
    if not workload.ready(NAME):
        pytest.skip("workloads/tri20k not prepared (built by __graft_entry__.build())")
    blob = workload.load_model(NAME)
    ds = desc.Descriptors(blob)
    m = workload.synth_model(NAME)
    am = capi.GmmScorer(ds, mode=capi.GMM_EXACT)
    dec = capi.Decoder(ds, am, max_utts=16, max_frames=16 * 400)
    return dict(blob=blob, ds=ds, m=m, am=am, dec=dec)


def test_full_size_gmm_bit_exact_vs_oracle(full, oracle_lib):
    x = workload.sample_batch(full["m"], 1, 64, seed=7)[0]
    got = full["am"].score(x)
    want = oracle_lib.gmm_score(full["ds"], x)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_full_size_end_to_end_vs_oracle(full, oracle_lib):
    """host MFCC -> GPU scoring -> GPU beam == oracle scoring -> oracle beam, atom for atom."""
    feats = workload.sample_batch(full["m"], 3, 300, seed=21)
    feats.append(full["m"].sample_noise(np.random.default_rng(5), 120))      # worst-case beam
    res = full["dec"].decode(feats)
    for x, r in zip(feats, res):
        sc = oracle_lib.gmm_score(full["ds"], x)
        o = oracle_lib.beam_decode(full["ds"], sc)
        assert r["overflow"] == 0
        ok, why = atoms_equal(r["atoms"], o["atoms"])
        assert ok, why
        assert r["words"] == o["words"] and r["status"] == o["status"]


def test_probe_utterance_matches_compiled_reference(full):
    """workloads/tri20k/probe.mfc, as the compiled reference decoded it (tests/golden/host/tri20k_probe)."""
    from julius_b200 import synth
    x, _ = synth.read_htk_param(workload.path(NAME, "probe.mfc"))
    u = load_pinned(os.path.join(GOLDEN, "host", "tri20k_probe"), [x])[1][0]
    r = full["dec"].decode([x])[0]
    ok, why = atoms_equal(r["atoms"], u.atoms)
    assert ok, why
    assert r["words"] == u.words and np.float32(r["score"]) == np.float32(u.score)


def test_trellis_structure_properties_at_full_batch(full):
    """Size-independent invariants on a larger batch: times are ordered, back pointers point to
    earlier atoms whose end frame precedes the begin frame, atoms are frame-major / wid-sorted,
    the best path ends in </s> at the last frame and starts with <s>."""
    feats = workload.sample_batch(full["m"], 16, 400, seed=33)
    res = full["dec"].decode(feats)
    tail, head = full["ds"].tree.tail_silwid, full["ds"].tree.head_silwid
    for r in res:
        a = r["atoms"]
        assert r["status"] == 0 and r["overflow"] == 0 and len(a) > 0
        key = a["end"].astype(np.int64) * 100000 + a["wid"]
        assert np.all(np.diff(key) > 0)
        assert np.all(a["begin"] <= a["end"] + 1)
        has = a["last"] >= 0
        assert np.all(a["last"][has] < np.nonzero(has)[0])
        assert np.all(a["end"][a["last"][has]] + 1 == a["begin"][has])
        assert np.all(a["begin"][~has] == 0)
        assert r["words"][0] == head and r["words"][-1] == tail


def test_fast_mode_scores_within_tolerance_and_decodes(full):
    am = capi.GmmScorer(full["ds"], mode=capi.GMM_FAST)
    x = workload.sample_batch(full["m"], 1, 128, seed=9)[0]
    a, b = am.score(x), full["am"].score(x)
    rel = np.abs(a - b) / np.maximum(np.maximum(np.abs(a), np.abs(b)), 1.0)
    assert rel.max() <= 1e-4      # BASELINE.json north_star tolerance on float log-likelihoods


def test_full_size_heap_self_check(monkeypatch, oracle_lib):
    """beam 800 over ~2400 tokens per frame: fast vs plain sequential heap replay on every frame."""
    if not workload.ready(NAME):
        pytest.skip("workloads/tri20k not prepared")
    monkeypatch.setenv("JB200_CHECK_HEAP", "1")
    blob = workload.load_model(NAME)
    ds = desc.Descriptors(blob)
    am = capi.GmmScorer(ds, mode=capi.GMM_EXACT)
    dec = capi.Decoder(ds, am, max_utts=8, max_frames=8 * 600)
    m = workload.synth_model(NAME)
    feats = workload.sample_batch(m, 6, 600, seed=77) + [m.sample_noise(np.random.default_rng(8), 300)]
    res = dec.decode(feats)
    assert all(r["overflow"] == 0 and r["status"] == 0 for r in res[:6])
    assert res[6]["overflow"] == 0
    x = feats[0]
    o = oracle_lib.beam_decode(ds, oracle_lib.gmm_score(ds, x))
    ok, why = atoms_equal(res[0]["atoms"], o["atoms"])
    assert ok, why


@pytest.mark.parametrize("name,frames", [("mono100", 400), ("tri20k_gbeam", 250), ("tri20k_mp", 250)])
def test_other_baseline_configs_end_to_end_vs_oracle(name, frames, oracle_lib):
    """BASELINE.json configs[0] (monophone 16-mix, 100 words) and configs[2] (-gprune beam, which is the
    safe top-N algorithm for state-tied models), and configs[1] on the multipath tree (-multipath): GPU end to end == CPU restatement, atom for atom."""
    if not workload.ready(name):
        pytest.skip(f"workloads/{name} not prepared")
    blob = workload.load_model(name)
    ds = desc.Descriptors(blob)
    m = workload.synth_model(name)
    am = capi.GmmScorer(ds, mode=capi.GMM_EXACT)
    dec = capi.Decoder(ds, am, max_utts=4, max_frames=4 * frames)
    feats = workload.sample_batch(m, 2, frames, seed=55)
    res = dec.decode(feats)
    for x, r in zip(feats, res):
        sc = oracle_lib.gmm_score(ds, x)
        got = am.score(x)
        assert np.array_equal(got.view(np.uint32), sc.view(np.uint32))
        o = oracle_lib.beam_decode(ds, sc)
        assert r["overflow"] == 0
        ok, why = atoms_equal(r["atoms"], o["atoms"])
        assert ok, why
        assert r["words"] == o["words"] and r["status"] == o["status"]


@pytest.mark.parametrize("name", ["tri20k", "tri20k_mp"])
def test_wide_beam_4000_vs_oracle(name, oracle_lib):
    """BASELINE.json configs[4] flavour: -b 4000 on the 20k-word tree (normal and multipath).  The heap-select
    array alone is 140 KB of shared memory, one utterance per SM; ~9000 tokens are created per frame."""
    if not workload.ready(name):
        pytest.skip(f"workloads/{name} not prepared")
    blob = workload.load_model(name)
    ds = desc.Descriptors(blob)
    ds.tree.beam_width = 4000
    m = workload.synth_model(name)
    am = capi.GmmScorer(ds, mode=capi.GMM_EXACT)
    dec = capi.Decoder(ds, am, max_utts=2, max_frames=2 * 120)
    feats = workload.sample_batch(m, 2, 120, seed=91)
    res = dec.decode(feats)
    for x, r in zip(feats, res):
        o = oracle_lib.beam_decode(ds, oracle_lib.gmm_score(ds, x), trace=True)
        assert r["overflow"] == 0
        ok, why = atoms_equal(r["atoms"], o["atoms"])
        assert ok, why
        assert r["words"] == o["words"] and r["status"] == o["status"]
    assert max(c[1] for c in o["trace"]) > 800      # the wide beam was actually used


@pytest.mark.parametrize("name,frames", [("dnn20k", 200), ("dnn60k_mp", 150)])
def test_dnn_hmm_configs_vs_oracle(name, frames, oracle_lib):
    """BASELINE.json configs[3] (DNN-HMM 528 -> 7 x 2048 -> 3000 states, 20k words) and configs[4] (the same acoustic
    model on the 60k-word multipath tree with -iwsp -iwcd1 max -b 4000: one utterance per SM, ~4 x beam tokens a frame).
    K2's scores are within 1e-4 of the reference, not bit-identical, so the beam is checked twice: bit-exact on the
    CPU restatement's own score matrix (GPU beam == CPU beam, atom for atom), and end to end (K2 -> K3) by the
    pass-1 word sequence and score."""
    if not workload.ready(name):
        pytest.skip(f"workloads/{name} not prepared")
    ds = desc.Descriptors(workload.load_model(name))
    m = workload.synth_model(name)
    feats = workload.sample_inputs(name, m, 2, frames, seed=61)
    am = capi.GmmScorer(ds, gmm_desc=ds.cd_only_gmm())
    dec = capi.Decoder(ds, am, max_utts=2, max_frames=2 * frames)
    scores = [oracle_lib.dnn_score(ds, x) for x in feats]
    want = [oracle_lib.beam_decode(ds, sc, trace=True) for sc in scores]
    for r, o in zip(dec.decode_scores(scores), want):
        assert r["overflow"] == 0
        ok, why = atoms_equal(r["atoms"], o["atoms"])
        assert ok, why
        assert r["words"] == o["words"] and r["status"] == o["status"]
    if name == "dnn60k_mp":
        assert max(c[1] for c in want[0]["trace"]) > 2000      # the wide beam was actually used
    dnn = capi.DnnScorer(ds)
    for x, sc in zip(feats, scores):
        got = dnn.score(x)
        rel = np.abs(got - sc) / np.maximum(np.maximum(np.abs(got), np.abs(sc)), 1.0)
        assert rel.max() <= 1e-4
    dec.attach_dnn(dnn)
    for r, o in zip(dec.decode(feats), want):
        assert r["overflow"] == 0 and r["status"] == o["status"]
        assert r["words"] == o["words"]
        assert abs(r["score"] - o["score"]) <= 1e-4 * abs(o["score"]) + 0.05
