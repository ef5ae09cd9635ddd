"""GPU: the drop-in boundaries exercised through the UNMODIFIED reference host (oracle/_ref).

  * jref + jb200.jpi with JB200_ATTACH=1: Julius' own pass-1 beam consumes GPU scores written into
    HMMWork.outprob_cache at CALLBACK_EVENT_PASS1_BEGIN  -> dump must equal the stock run (golden).
  * jref_gpu: libjulius linked with jb200_beam_shim.o instead of beam.o -> the stock host drives the
    GPU scorer + GPU beam through get_back_trellis_init/_end/finalize_1st_pass -> same trellis.
"""
import os

import numpy as np
import pytest

from julius_b200 import refdump, synth
from util import GOLDEN, Golden, atoms_equal, digest, load_pinned

pytestmark = pytest.mark.gpu


def _prepare(case, tmp_path):
    from oracle import ffi
    if not (ffi.have_ref() and os.path.exists(ffi.JREF_GPU)):
        pytest.skip("oracle/_ref host binaries not built")
    g = Golden(case)
    d = str(tmp_path)
    m = synth.SynthModel(synth.SynthConfig.preset(g.meta["preset"]))
    m.write_all(d)
    files = []
    for i, x in enumerate(g.feats):
        fn = os.path.join(d, f"u{i}.mfc")
        synth.write_htk_param(fn, x)
        files.append(fn)
    return g, d, files


@pytest.mark.parametrize("case", ["tiny", "small_b100", "small_iwsp"])
def test_attached_gpu_scores_drive_the_stock_beam(case, tmp_path):
    from oracle import ffi
    g, d, files = _prepare(case, tmp_path)
    dump, out = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], env_extra={"JB200_ATTACH": "1"})
    utts = refdump.load_refdump(dump)
    assert len(utts) == len(g.utts)
    for u, ref in zip(utts, g.utts):
        assert np.array_equal(u.outprob.view(np.uint32), ref.outprob.view(np.uint32))
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.words == ref.words and np.float32(u.score) == np.float32(ref.score)


@pytest.mark.parametrize("case", ["tiny", "small_b100", "small_safe", "small_mp", "small_iwsp"])
def test_stock_host_with_gpu_beam_linked_in(case, tmp_path):
    from oracle import ffi
    g, d, files = _prepare(case, tmp_path)
    dump, out = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], binary=ffi.JREF_GPU)
    utts = refdump.load_refdump(dump)
    assert len(utts) == len(g.utts)
    for u, ref in zip(utts, g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.status == ref.status
        assert u.words == ref.words and np.float32(u.score) == np.float32(ref.score)


def _results(out):
    return [ln for ln in out.splitlines() if ln.startswith("JREF_RESULT")]


def _stock(name):
    """lines the stock host printed for the same run (tests/golden/make_golden.py)"""
    return open(os.path.join(GOLDEN, "host", name)).read().splitlines()


@pytest.mark.parametrize("case", ["small_b100", "small_iwsp"])
def test_full_two_pass_recognition_is_unchanged_by_either_boundary(case, tmp_path):
    """SURVEY 8(f).1: the stock host runs BOTH passes; pass 2 (stack decoding on the word trellis,
    re-reading the state scores through outprob_state) must produce the same sentences and scores when
    (a) the GPU fills the score cache, (b) the GPU beam builds the trellis, (c) both."""
    from oracle import ffi
    g, d, files = _prepare(case, tmp_path)
    want = _stock(f"{case}_two_pass.txt")
    assert len(want) == len(files) and all("sent0=" in w for w in want[:2])
    _, a = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], two_pass=True, dump="a.jrf", env_extra={"JB200_ATTACH": "1"})
    assert _results(a) == want
    # (b): pass 1 never touches the host's score cache, pass 2 evaluates the states it needs on the CPU
    _, b = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], two_pass=True, dump="b.jrf", binary=ffi.JREF_GPU,
                       outprobout=False)
    assert _results(b) == want
    _, c = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], two_pass=True, dump="c.jrf", binary=ffi.JREF_GPU,
                       env_extra={"JB200_ATTACH": "1"})
    assert _results(c) == want


def test_calcmix_hook_equals_gprune_none(tmp_path):
    """The jconf surface `-gprune jb200` (plugin calcmix hook set, plugin.c:336-354): the host keeps its own
    outprob_state -> calc_mix path and asks the plugin for the per-Gaussian scores of the current frame, which come
    from the GPU (jb200_gmm_gauss_host).  No pruning is applied, so the run must equal stock `-gprune none`."""
    from oracle import ffi
    g, d, files = _prepare("tiny", tmp_path)
    _, want = load_pinned(os.path.join(GOLDEN, "host", "tiny_gprune_none"), g.feats)      # the stock host, -gprune none
    dump1, out = ffi.run_ref(d, files, extra_args=["-gprune", "jb200"], dump="hook.jrf", env_extra={"JB200_ATTACH": "calcmix"})
    got = refdump.load_refdump(dump1)
    assert len(want) == len(got) == len(files)
    for u, v in zip(want, got):
        assert digest(v.outprob) == u.outprob_sha256
        ok, why = atoms_equal(v.atoms, u.atoms)
        assert ok, why
        assert u.words == v.words and np.float32(u.score) == np.float32(v.score)


def test_beam_shim_decode_ahead_over_a_file_list(tmp_path):
    """The stock host hands the shim one utterance at a time.  With JB200_FILELIST naming the same list the host reads,
    the shim decodes the next files in one GPU batch and answers the host's following utterances from that batch --
    only when the vectors the host presents hash to what was decoded.  Same trellis and pass-1 result as the stock
    host, every utterance after the first batch answered from the cache."""
    from oracle import ffi
    g, d, files = _prepare("small_b100", tmp_path)
    files = files + files                      # 2 x the golden utterances: a list longer than one batch
    lst = os.path.join(d, "files.lst")
    with open(lst, "w") as f:
        f.write("\n".join(files) + "\n")
    dump, out = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], binary=ffi.JREF_GPU,
                            env_extra={"JB200_FILELIST": lst, "JB200_AHEAD": "3", "JB200_SHIM_VERBOSE": "1"})
    utts = refdump.load_refdump(dump)
    assert len(utts) == len(files)
    for u, ref in zip(utts, g.utts + g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.status == ref.status and u.words == ref.words and np.float32(u.score) == np.float32(ref.score)
    assert out.count("from_cache") == len(files)
    assert out.count("JB200_SHIM batch") == (len(files) + 2) // 3
    # a list that does not match what the host reads is harmless: everything is decoded singly, same result
    bad = os.path.join(d, "bad.lst")
    with open(bad, "w") as f:
        f.write("\n".join(reversed(files)) + "\n")
    dump2, out2 = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], binary=ffi.JREF_GPU, dump="bad.jrf",
                              env_extra={"JB200_FILELIST": bad, "JB200_AHEAD": "3", "JB200_SHIM_VERBOSE": "1"})
    for u, ref in zip(refdump.load_refdump(dump2), g.utts + g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why


@pytest.mark.parametrize("case", ["small_b100", "small_mp"])
@pytest.mark.parametrize("frames", ["1", "7"])
def test_stock_host_drives_the_gpu_beam_frame_by_frame(case, frames, tmp_path):
    """Frame-synchronous mode of the beam shim (what real-time input and -progout select; forced here with
    JB200_STREAM=1): get_back_trellis_proceed(t) feeds the frames that have arrived to a device stream
    (jb200_stream_feed_host), get_back_trellis_end sends the rest with the end-of-utterance mark.  Same trellis and
    pass-1 result as the stock host, whatever the feed size."""
    from oracle import ffi
    g, d, files = _prepare(case, tmp_path)
    dump, out = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], binary=ffi.JREF_GPU,
                            env_extra={"JB200_STREAM": "1", "JB200_STREAM_FRAMES": frames})
    utts = refdump.load_refdump(dump)
    assert len(utts) == len(g.utts)
    for u, ref in zip(utts, g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.status == ref.status
        assert u.words == ref.words and np.float32(u.score) == np.float32(ref.score)


@pytest.mark.parametrize("case", ["small_b100", "small_mp"])
def test_progressive_output_matches_the_stock_host(case, tmp_path):
    """-progout: every -proginterval the host publishes the best word sequence so far (bt_current_max, beam.c:876-921,
    raised through have_interim / CALLBACK_RESULT_PASS1_INTERIM, pass1.c:306-314).  The GPU beam must hand the host the
    same interim sequences and scores, at the same frames, as the stock beam -- and the same final trellis."""
    from oracle import ffi
    g, d, files = _prepare(case, tmp_path)
    extra = g.meta["extra_args"] + ["-progout", "-proginterval", "100"]
    want = _stock(f"{case}_interim.txt")
    assert len(want) >= 10 * len(files) and any("words=0," in w for w in want)
    dump, out = ffi.run_ref(d, files, extra_args=extra, binary=ffi.JREF_GPU, env_extra={"JREF_INTERIM": "1"})
    got = [ln for ln in out.splitlines() if ln.startswith("JREF_INTERIM")]
    assert got == want
    for u, ref in zip(refdump.load_refdump(dump), g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.words == ref.words and np.float32(u.score) == np.float32(ref.score)


def test_user_defined_lm_through_the_gpu_beam(tmp_path):
    """-userlm (wchmm.h:274-276): the application registers LM functions (the driver does, JREF_USERLM=1, the way
    julius/main.c:153-161 does); pass 1 reads them through two host function pointers, which the export step tabulates
    for the device.  The stock host with the GPU beam linked in must produce the stock host's trellis."""
    from oracle import ffi
    g, d, files = _prepare("small_userlm", tmp_path)
    dump, out = ffi.run_ref(d, files, extra_args=g.meta["extra_args"], binary=ffi.JREF_GPU, env_extra=g.meta["env"])
    utts = refdump.load_refdump(dump)
    assert len(utts) == len(g.utts)
    for u, ref in zip(utts, g.utts):
        ok, why = atoms_equal(u.atoms, ref.atoms)
        assert ok, why
        assert u.status == ref.status and u.words == ref.words and np.float32(u.score) == np.float32(ref.score)
    # and the user LM really is in effect: the plain N-gram run of the same input scores differently
    plain = Golden("small_b100")
    assert np.float32(plain.utts[0].score) != np.float32(g.utts[0].score)
