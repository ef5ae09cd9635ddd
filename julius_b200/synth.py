"""Seeded synthetic model / input generator (SURVEY.md section 8d "Synthetic inputs").

The reference ships no models and no test vectors (SURVEY.md section 4), so every
fixture is synthesised: an HTK-format tied-state triphone GMM acoustic model,
an HMMList, a pronunciation dictionary, a forward 2-gram ARPA LM and HTK
parameter files whose frames are sampled *from the model* along
``<s> w .. </s>`` state paths (i.i.d. noise makes pass 1 fail, SURVEY 4.6).

File formats follow the reference's readers:
  hmmdefs   libsent/src/hmminfo/rdhmmdef_*.c          (HTK ASCII macros)
  hmmlist   libsent/src/hmminfo/rdhmmlist.c:27-43     ("logical physical")
  dict      libsent/src/voca/voca_load_htkdict.c:33-52
  ARPA      libsent/src/ngram/ngram_read_arpa.c       (2-gram order = 1-gram listing order, :452-479)
  features  libsent/src/anlz/rdparam.c:83-187         (big-endian HTK parameter file)

This module only writes files / returns numpy arrays; it never calls the
reference or the oracle.
"""
from __future__ import annotations

import dataclasses
import os
import struct

import numpy as np

SIL = "sil"
# HTK parameter kinds (libsent/include/sent/htk_param.h): base MFCC = 6, qualifiers _E 0x40, _N 0x80, _D 0x100,
# _A 0x200, _Z 0x800
PARMKIND_MFCC_E_D_A = 6 | 0x40 | 0x100 | 0x200
PARMKIND_USER = 9
# the usual MFCC layout of each feature size the GMM scorer is built for: (kind name in hmmdefs, parmKind code).
# 25 = 12 MFCC + 12 delta + delta energy (_N drops absolute energy), the Julius dictation-kit format
PARMKINDS = {
    25: ("MFCC_E_D_N_Z", 6 | 0x40 | 0x100 | 0x80 | 0x800),
    26: ("MFCC_E_D_Z", 6 | 0x40 | 0x100 | 0x800),
    38: ("MFCC_E_D_A_N_Z", 6 | 0x40 | 0x100 | 0x200 | 0x80 | 0x800),
    39: ("MFCC_E_D_A", PARMKIND_MFCC_E_D_A),
}


def parmkind_for_dim(dim: int):
    """(hmmdefs kind name, HTK parmKind code) of a feature vector of `dim` values; USER for any other size"""
    return PARMKINDS.get(dim, ("USER", PARMKIND_USER))


@dataclasses.dataclass
class SynthConfig:
    name: str = "tiny"
    seed: int = 1
    n_phones: int = 8          # including sil (index 0)
    n_states: int = 60         # tied-state pool size S
    n_mix: int = 4             # M
    dim: int = 39              # D
    phys_per_phone: int = 6    # physical HMMs per centre phone
    vocab: int = 50            # words excluding <s>, </s>
    n_bigrams: int = 300
    min_wlen: int = 2
    max_wlen: int = 5
    monophone: bool = False    # context-independent AM (config[0])
    one_phone_words: int = 0   # number of 1-phone words (exercise AS_LRSET)
    sp_model: bool = False     # add a 1-state tee model "sp" (skip transition) for -iwsp; forces multipath
    transparent_words: int = 0 # the first k words get a {..} output string: transparent to the LM context (fillers)
    tied_mixture: bool = False # phonetic tied-mixture AM: one Gaussian codebook per (phone, state position), per-state weights
    # irregular mixtures: state s has 1..n_mix mixture slots, and in a few states one slot is left out of the
    # definition (a NULL density, rdhmmdef_mpdf.c:170-193); drawn from their own generator so the rest is unchanged
    irregular_mix: bool = False

    @staticmethod
    def preset(name: str) -> "SynthConfig":
        if name == "tiny":
            return SynthConfig()
        if name in ("tiny_d25", "tiny_d26"):   # "tiny" at the other MFCC sizes, irregular mixture counts, NULL densities
            return SynthConfig(name=name, dim=int(name[-2:]), n_mix=6, irregular_mix=True)
        if name == "small":      # a few hundred words, used for CPU-side parity
            return SynthConfig(name="small", seed=2, n_phones=12, n_states=240, n_mix=8,
                               phys_per_phone=24, vocab=400, n_bigrams=4000,
                               min_wlen=2, max_wlen=6, one_phone_words=3)
        if name == "small_sp":   # "small" plus a short-pause tee model (-iwsp, multipath by necessity)
            c = SynthConfig.preset("small")
            return dataclasses.replace(c, name="small_sp", sp_model=True)
        if name == "small_tm":   # phonetic tied-mixture variant of "small" (<TMIX> codebooks, calc_tied_mix.c)
            c = SynthConfig.preset("small")
            return dataclasses.replace(c, name="small_tm", tied_mixture=True, n_mix=16)
        if name == "small_tr":   # "small" with 40 transparent (filler) words: exercises last_cword / -transp penalty
            c = SynthConfig.preset("small")
            return dataclasses.replace(c, name="small_tr", transparent_words=40)
        if name == "mono100":    # BASELINE config[0]: monophone 16-mix, 100 words
            return SynthConfig(name="mono100", seed=3, n_phones=40, n_states=120, n_mix=16,
                               phys_per_phone=1, vocab=100, n_bigrams=1500,
                               min_wlen=2, max_wlen=6, monophone=True)
        if name == "tri20k":     # BASELINE config[1]/[2]: 3k states x 16 mix, 20k words
            return SynthConfig(name="tri20k", seed=4, n_phones=36, n_states=3000, n_mix=16,
                               phys_per_phone=84, vocab=20000, n_bigrams=200000,
                               min_wlen=3, max_wlen=8, one_phone_words=0)
        if name == "tri60k":     # BASELINE config[4]: the same AM, 60k words, short-pause model for -iwsp
            c = SynthConfig.preset("tri20k")
            return dataclasses.replace(c, name="tri60k", vocab=60000, n_bigrams=600000, sp_model=True)
        raise KeyError(name)


class SynthModel:
    """Holds the generated AM/LM/dict as numpy arrays + writers for the HTK formats."""

    def __init__(self, cfg: SynthConfig):
        self.cfg = cfg
        rng = np.random.default_rng(cfg.seed)
        P, S, M, D = cfg.n_phones, cfg.n_states, cfg.n_mix, cfg.dim
        self.phones = [SIL] + [f"p{i:02d}" for i in range(1, P)]
        # ---- tied-state Gaussian pool (SURVEY 8d: centre N(0,1) + N(0,0.5), var U(0.3,1.5), w Dirichlet(2))
        centre = rng.normal(0.0, 1.0, size=(S, 1, D))
        self.mean = (centre + rng.normal(0.0, 0.5, size=(S, M, D))).astype(np.float32)
        self.var = rng.uniform(0.3, 1.5, size=(S, M, D)).astype(np.float32)
        self.weight = rng.dirichlet(np.full(M, 2.0), size=S).astype(np.float32)
        # ---- irregular mixtures: n_mix_of[s] slots, null[s, m] = slot left undefined (weights renormalised over the rest)
        self.n_mix_of = np.full(S, M, dtype=np.int64)
        self.null = np.zeros((S, M), dtype=bool)
        if cfg.irregular_mix:
            r2 = np.random.default_rng(cfg.seed + 1000)
            self.n_mix_of = r2.integers(1, M + 1, size=S)
            for s in r2.choice(S, size=S // 8, replace=False):
                if self.n_mix_of[s] > 1:
                    self.null[s, r2.integers(self.n_mix_of[s])] = True
            present = (np.arange(M)[None, :] < self.n_mix_of[:, None]) & ~self.null
            w = np.where(present, self.weight, 0.0).astype(np.float64)
            self.weight = (w / w.sum(1, keepdims=True)).astype(np.float32)
        # ---- state pool partition by (centre phone, position)
        part = [[[] for _ in range(3)] for _ in range(P)]
        order = rng.permutation(S)
        for i, s in enumerate(order):
            part[(i // 3) % P][i % 3].append(int(s))
        for c in range(P):
            for k in range(3):
                if not part[c][k]:
                    part[c][k].append(int(order[(c * 3 + k) % S]))
        # ---- tied mixture: the states of one (phone, position) cell share the cell's codebook (its first state's
        #      Gaussians); the mixture weights stay per state
        self.book_of = np.full(S, -1, dtype=np.int64)
        if cfg.tied_mixture:
            for c in range(P):
                for k in range(3):
                    first = part[c][k][0]
                    for st_id in part[c][k]:
                        self.book_of[st_id] = c * 3 + k
                        self.mean[st_id] = self.mean[first]
                        self.var[st_id] = self.var[first]
            self.book_first = {c * 3 + k: part[c][k][0] for c in range(P) for k in range(3)}
        # ---- physical models: (state triple, transition macro)
        self.trans_names = ["T1", "T2", "T3"]
        self.trans_self = [0.6, 0.5, 0.7]
        K = cfg.phys_per_phone
        self.phys = []           # list of (name, [s0,s1,s2], trans_idx)
        self.phys_of = {}        # (c, h) -> phys index
        for c in range(P):
            for h in range(K):
                st = [part[c][k][int(rng.integers(len(part[c][k])))] for k in range(3)]
                self.phys_of[(c, h)] = len(self.phys)
                self.phys.append((f"m{c:02d}_{h:03d}", st, int(rng.integers(3))))
        self._ctx_hash = rng.integers(0, 1 << 30, size=(P, P))
        # ---- vocabulary
        V = cfg.vocab
        self.words = []          # (name, [phone idx...])
        seen = set()
        n1 = cfg.one_phone_words
        while len(self.words) < V:
            if n1 > 0:
                L = 1
            else:
                L = int(rng.integers(cfg.min_wlen, cfg.max_wlen + 1))
            pr = tuple(int(x) for x in rng.integers(1, P, size=L))
            if pr in seen:
                continue
            seen.add(pr)
            if L == 1:
                n1 -= 1
            self.words.append((f"w{len(self.words):05d}", list(pr)))
        # ---- LM: Zipf unigrams, random bigrams
        rank = rng.permutation(V) + 1
        p = 1.0 / rank.astype(np.float64)
        p = 0.9 * p / p.sum()
        self.lm_vocab = ["<unk>", "<s>", "</s>"] + [w for w, _ in self.words]
        uni = np.concatenate([[1e-4, 0.01, 0.09], p])
        self.uni_logp = np.log10(uni).astype(np.float32)
        self.uni_bow = (-rng.uniform(0.05, 1.0, size=len(uni))).astype(np.float32)
        nv = len(self.lm_vocab)
        pairs = set()
        nb = min(cfg.n_bigrams, (nv - 2) * (nv - 2) // 2)
        while len(pairs) < nb:
            k = nb - len(pairs)
            w1 = rng.integers(1, nv, size=k * 2)
            # Zipf-biased successor choice so that frequent words get bigrams
            w2 = np.minimum(nv - 1, 2 + (rng.pareto(1.2, size=k * 2) * 20).astype(np.int64) % (nv - 2))
            for a, b in zip(w1, w2):
                if a == 2 or b == 1 or a == 0 or b == 0:   # no "</s> x", no "x <s>", no <unk>
                    continue
                pairs.add((int(a), int(b)))
                if len(pairs) >= nb:
                    break
        self.bigrams = sorted(pairs)     # listing order == index order
        self.bi_logp = (-rng.uniform(0.3, 4.0, size=len(self.bigrams))).astype(np.float32)
        self.rng_state = rng

    # ------------------------------------------------------------------ AM helpers
    def triphone_phys(self, l: int, c: int, r: int) -> int:
        if self.cfg.monophone:
            return self.phys_of[(c, 0)]
        h = int(self._ctx_hash[l, r]) % self.cfg.phys_per_phone
        return self.phys_of[(c, h)]

    def logical_name(self, l: int, c: int, r: int) -> str:
        return f"{self.phones[l]}-{self.phones[c]}+{self.phones[r]}"

    # ------------------------------------------------------------------ writers
    def write_hmmdefs(self, path: str) -> None:
        cfg = self.cfg
        D, M = cfg.dim, cfg.n_mix
        ln2pi = np.log(2.0 * np.pi)
        with open(path, "w") as f:
            f.write(f"~o\n<STREAMINFO> 1 {D}\n<VECSIZE> {D}<NULLD><{parmkind_for_dim(D)[0]}><DIAGC>\n")
            for name, a_self in zip(self.trans_names, self.trans_self):
                a = np.zeros((5, 5))
                a[0, 1] = 1.0
                for i in (1, 2, 3):
                    a[i, i] = a_self
                    a[i, i + 1] = 1.0 - a_self
                f.write(f'~t "{name}"\n<TRANSP> 5\n')
                for row in a:
                    f.write(" " + " ".join(f"{x:.6e}" for x in row) + "\n")
            if cfg.tied_mixture:
                # codebook "cbNNN_": densities ~m "cbNNN_1" .. "cbNNN_M" (rdhmmdef_tiedmix.c:75-100 builds the index
                # from name + number), states carry <TMIX> book weights (rdhmmdef_tiedmix.c:135-190)
                for bk, first in sorted(self.book_first.items()):
                    for m in range(M):
                        f.write(f'~m "cb{bk:03d}_{m + 1}"\n')
                        f.write(f"<MEAN> {D}\n " + " ".join(f"{x:.8e}" for x in self.mean[first, m]) + "\n")
                        f.write(f"<VARIANCE> {D}\n " + " ".join(f"{x:.8e}" for x in self.var[first, m]) + "\n")
                        g = D * ln2pi + float(np.sum(np.log(self.var[first, m].astype(np.float64))))
                        f.write(f"<GCONST> {g:.8e}\n")
                for s in range(cfg.n_states):
                    f.write(f'~s "st{s}"\n<NUMMIXES> {M}\n<TMIX> cb{int(self.book_of[s]):03d}_ ')
                    f.write(" ".join(f"{w:.8e}" for w in self.weight[s]) + "\n")
            for s in range(cfg.n_states if not cfg.tied_mixture else 0):
                f.write(f'~s "st{s}"\n<NUMMIXES> {self.n_mix_of[s]}\n')
                for m in range(self.n_mix_of[s]):
                    if self.null[s, m]:
                        continue
                    f.write(f"<MIXTURE> {m + 1} {self.weight[s, m]:.8e}\n")
                    f.write(f"<MEAN> {D}\n " + " ".join(f"{x:.8e}" for x in self.mean[s, m]) + "\n")
                    f.write(f"<VARIANCE> {D}\n " + " ".join(f"{x:.8e}" for x in self.var[s, m]) + "\n")
                    g = D * ln2pi + float(np.sum(np.log(self.var[s, m].astype(np.float64))))
                    f.write(f"<GCONST> {g:.8e}\n")
            for name, st, ti in self.phys:
                f.write(f'~h "{name}"\n<BEGINHMM>\n<NUMSTATES> 5\n')
                for k in range(3):
                    f.write(f'<STATE> {k + 2}\n~s "st{st[k]}"\n')
                f.write(f'~t "{self.trans_names[ti]}"\n<ENDHMM>\n')
            if cfg.sp_model:
                # short pause: one emitting state (the middle state of a silence model) that can be skipped
                st = self.phys[self.phys_of[(0, 0)]][1][1]
                f.write(f'~h "sp"\n<BEGINHMM>\n<NUMSTATES> 3\n<STATE> 2\n~s "st{st}"\n<TRANSP> 3\n')
                f.write(" 0.0 0.7 0.3\n 0.0 0.6 0.4\n 0.0 0.0 0.0\n<ENDHMM>\n")

    def write_hmmlist(self, path: str) -> None:
        P = self.cfg.n_phones
        with open(path, "w") as f:
            if self.cfg.sp_model:
                f.write("sp sp\n")
            if self.cfg.monophone:
                for c in range(P):
                    f.write(f"{self.phones[c]} {self.phys[self.phys_of[(c, 0)]][0]}\n")
                return
            for l in range(P):
                for c in range(P):
                    for r in range(P):
                        f.write(f"{self.logical_name(l, c, r)} {self.phys[self.triphone_phys(l, c, r)][0]}\n")

    def write_dict(self, path: str) -> None:
        with open(path, "w") as f:
            f.write(f"<s> [] {SIL}\n</s> [] {SIL}\n")
            for i, (w, pr) in enumerate(self.words):
                out = f"{{{w}}}" if i < self.cfg.transparent_words else f"[{w}]"
                f.write(f"{w} {out} " + " ".join(self.phones[p] for p in pr) + "\n")

    def write_arpa(self, path: str) -> None:
        with open(path, "w") as f:
            f.write("\n\\data\\\n")
            f.write(f"ngram 1={len(self.lm_vocab)}\nngram 2={len(self.bigrams)}\n\n\\1-grams:\n")
            for i, w in enumerate(self.lm_vocab):
                f.write(f"{self.uni_logp[i]:.6f} {w} {self.uni_bow[i]:.6f}\n")
            f.write("\n\\2-grams:\n")
            for (a, b), lp in zip(self.bigrams, self.bi_logp):
                f.write(f"{lp:.6f} {self.lm_vocab[a]} {self.lm_vocab[b]}\n")
            f.write("\n\\end\\\n")

    # ------------------------------------------------------------------ grammar (DFA) mode
    GRAMMAR_NEXT = {0: (2, 3), 2: (3, 4), 3: (4, 5), 4: (5, 2, 1), 5: (2, 1)}    # category -> categories that may follow

    def write_grammar(self, outdir: str, prefix: str = "g") -> dict:
        """A finite-state grammar over the same vocabulary in the reference's formats (-dfa/-v, or -gram prefix):
        category 0 = sentence-initial silence, 1 = sentence-final silence, words spread over categories 2..5;
        GRAMMAR_NEXT is the forward category-pair relation.  The .dfa file is the REVERSED automaton Julius expects
        (rddfa.c:125-200: `state category next_state accept-flag`, state 0 initial, it reads the sentence from its
        last word), the .dict file carries the category id in the first column."""
        os.makedirs(outdir, exist_ok=True)
        cats = sorted(set(self.GRAMMAR_NEXT) | {c for v in self.GRAMMAR_NEXT.values() for c in v})
        state_of = {c: i + 1 for i, c in enumerate(c for c in cats if c != 0)}     # "the category to the right is c"
        final = len(state_of) + 1
        lines = [f"0 1 {state_of[1]} 0 0"]
        for p_cat, nxt in sorted(self.GRAMMAR_NEXT.items()):
            for c in nxt:
                if p_cat == 0:
                    lines.append(f"{state_of[c]} 0 {final} 0 0")
                else:
                    lines.append(f"{state_of[c]} {p_cat} {state_of[p_cat]} 0 0")
        lines.append(f"{final} -1 -1 1 0")
        dfa = os.path.join(outdir, prefix + ".dfa")
        with open(dfa, "w") as f:
            f.write("\n".join(lines) + "\n")
        dic = os.path.join(outdir, prefix + ".dict")
        with open(dic, "w") as f:
            f.write(f"0 [<s>] {SIL}\n1 [</s>] {SIL}\n")
            for i, (w, pr) in enumerate(self.words):
                f.write(f"{2 + i % 4} [{w}] " + " ".join(self.phones[p] for p in pr) + "\n")
        return {"dfa": dfa, "dict": dic}

    def sample_grammar_sentence(self, rng: np.random.Generator, n_words: int):
        """word indices of a sentence the grammar accepts (without the silences)"""
        by_cat = {c: [i for i in range(len(self.words)) if 2 + i % 4 == c] for c in (2, 3, 4, 5)}
        out, cat = [], 0
        while True:
            nxt = [c for c in self.GRAMMAR_NEXT[cat] if c != 1]
            if len(out) >= n_words and 1 in self.GRAMMAR_NEXT[cat]:
                return out
            cat = int(rng.choice(nxt))
            out.append(int(rng.choice(by_cat[cat])))

    def write_all(self, outdir: str) -> dict:
        os.makedirs(outdir, exist_ok=True)
        paths = {k: os.path.join(outdir, k) for k in ("hmmdefs", "hmmlist", "dict", "lm.arpa")}
        self.write_hmmdefs(paths["hmmdefs"])
        self.write_hmmlist(paths["hmmlist"])
        self.write_dict(paths["dict"])
        self.write_arpa(paths["lm.arpa"])
        return paths

    # ------------------------------------------------------------------ features
    def sample_state_path(self, rng: np.random.Generator, n_frames: int, word_seq=None):
        """A random ``<s> w.. </s>`` path through the tied states: (state ids [n_frames] int64, word index list).
        Words are appended until the frame budget is reached and the tail is padded with trailing silence so
        every utterance ends inside ``</s>``."""
        cfg = self.cfg
        states = []
        words = []
        avg = 3 * 2.5
        budget = n_frames - int(6 * avg)

        def add_phone(l, c, r):
            ph = self.phys[self.triphone_phys(l, c, r)]
            a_self = self.trans_self[ph[2]]
            for s in ph[1]:
                d = int(rng.geometric(1.0 - a_self))
                states.extend([s] * d)

        # <s>
        seq = [[0]]
        if word_seq is not None:             # a given word sequence (e.g. a sentence of the grammar)
            for wi in word_seq:
                seq.append(self.words[wi][1])
                words.append(int(wi))
        while word_seq is None:
            wi = int(rng.integers(len(self.words)))
            seq.append(self.words[wi][1])
            words.append(wi)
            if sum(len(x) for x in seq) * avg >= budget:
                break
        seq.append([0])
        flat = [p for w in seq for p in w]
        for i, c in enumerate(flat):
            l = flat[i - 1] if i > 0 else 0
            r = flat[i + 1] if i + 1 < len(flat) else 0
            add_phone(l, c, r)
        sil_states = self.phys[self.triphone_phys(flat[-2] if len(flat) > 1 else 0, 0, 0)][1]
        if len(states) > n_frames:
            # cut inside the path but keep a silence tail of ~15 frames
            tail = [sil_states[0]] * 5 + [sil_states[1]] * 5 + [sil_states[2]] * 5
            states = states[: n_frames - len(tail)] + tail
        while len(states) < n_frames:
            states.append(sil_states[2])
        return np.asarray(states[:n_frames], dtype=np.int64), words

    def sample_utterance(self, rng: np.random.Generator, n_frames: int, noise: float = 1.0, word_seq=None):
        """Sample n_frames feature frames along a random ``<s> w.. </s>`` path (sample_state_path), each frame drawn
        from one Gaussian of its state.  Returns (feats [T, D] float32, word index list)."""
        cfg = self.cfg
        st, words = self.sample_state_path(rng, n_frames, word_seq)
        comp = np.array([rng.choice(cfg.n_mix, p=self.weight[s].astype(np.float64) / float(self.weight[s].astype(np.float64).sum())) for s in st])
        mu = self.mean[st, comp]
        sd = np.sqrt(self.var[st, comp])
        x = mu + noise * sd * rng.standard_normal(mu.shape).astype(np.float32)
        return x.astype(np.float32), words

    def sample_noise(self, rng: np.random.Generator, n_frames: int):
        return rng.normal(0.0, 1.2, size=(n_frames, self.cfg.dim)).astype(np.float32)


def write_htk_param(path: str, feats: np.ndarray, parmkind: int | None = None,
                    samp_period: int = 100000) -> None:
    """Big-endian HTK parameter file (libsent/src/anlz/rdparam.c:83-187).  parmkind None: the kind the synthetic
    hmmdefs of this feature size declare (parmkind_for_dim)."""
    feats = np.ascontiguousarray(feats, dtype=np.float32)
    T, D = feats.shape
    if parmkind is None:
        parmkind = parmkind_for_dim(D)[1]
    with open(path, "wb") as f:
        f.write(struct.pack(">IIHh", T, samp_period, D * 4, parmkind))
        f.write(feats.astype(">f4").tobytes())


def read_htk_param(path: str):
    with open(path, "rb") as f:
        T, period, size, kind = struct.unpack(">IIHh", f.read(12))
        D = size // 4
        data = np.frombuffer(f.read(T * D * 4), dtype=">f4").astype(np.float32).reshape(T, D)
    return data, kind


# ---------------------------------------------------------------------------------------- DNN-HMM
@dataclasses.dataclass
class DnnConfig:
    in_dim: int = 120          # feature_len * context_len (already spliced, SURVEY 4.8)
    feature_len: int = 40
    context_len: int = 3
    hidden: int = 64
    layers: int = 2
    seed: int = 5
    # Benchmark workloads ("prototype" output layer): a random-init logistic stack of this depth with the default
    # weight scale maps every input to (almost) the same hidden vector, so the posteriors do not depend on the frame
    # at all and the beam search degenerates.  With w_scale ~ 8 the hidden layers keep the inputs apart, and the output
    # layer is set, instead of drawn, to the nearest-prototype classifier  logit_s(h) = proto_gain * (h_s - hbar).(h - hbar)
    # over one prototype input per state -- the stand-in for a trained network: on the prototype of state s the
    # network is confident of s.  Utterances then emit the prototypes along an HMM state path.
    w_scale: float = 1.5
    prototype_output: bool = False
    proto_gain: float = 0.03
    cache_dir: str = ""        # where the (BLAS-order dependent) prototype output layer is kept so every reader sees the same bits


_DNN_CACHE = {}


def dnn_arrays(n_states: int, cfg: DnnConfig) -> dict:
    """The synthetic DNN of a config: W{i} (out,in) and B{i} (out,1) as '<f4', output layer Wo/Bo, Dirichlet state
    priors (and, for prototype_output, the per-state prototype inputs "proto").  One seeded draw order, shared by
    write_dnn (files for the reference) and dnn_blob_entries (flattened)."""
    key = (n_states, dataclasses.astuple(cfg))
    if key in _DNN_CACHE:
        return _DNN_CACHE[key]
    rng = np.random.default_rng(cfg.seed)
    dims = [cfg.in_dim] + [cfg.hidden] * cfg.layers
    arrays = {}
    for i in range(cfg.layers):
        arrays[f"W{i + 1}"] = (rng.standard_normal((dims[i + 1], dims[i])) * (cfg.w_scale / np.sqrt(dims[i]))).astype("<f4")
        arrays[f"B{i + 1}"] = (rng.standard_normal((dims[i + 1], 1)) * 0.1).astype("<f4")
        if cfg.prototype_output and i > 0:
            # logistic activations average 0.5: centre each unit's input on that (bias = -0.5 * sum of its weights),
            # or the common component saturates every unit the same way for all inputs and the layers collapse them
            arrays[f"B{i + 1}"] = (arrays[f"B{i + 1}"] - 0.5 * arrays[f"W{i + 1}"].astype(np.float64).sum(1, keepdims=True)).astype("<f4")
    arrays["Wo"] = (rng.standard_normal((n_states, cfg.hidden)) * (3.0 / np.sqrt(cfg.hidden))).astype("<f4")
    arrays["Bo"] = (rng.standard_normal((n_states, 1)) * 0.1).astype("<f4")
    arrays["prior"] = rng.dirichlet(np.full(n_states, 5.0))
    if cfg.prototype_output:
        fn = os.path.join(cfg.cache_dir, f"dnn_proto_s{n_states}_i{cfg.in_dim}_h{cfg.hidden}x{cfg.layers}_seed{cfg.seed}.npz") if cfg.cache_dir else ""
        if fn and os.path.exists(fn):
            z = np.load(fn)
            arrays["proto"], arrays["Wo"], arrays["Bo"] = z["proto"], z["Wo"], z["Bo"]
        else:
            proto = rng.standard_normal((n_states, cfg.in_dim)).astype(np.float32)
            h = proto.astype(np.float64)
            for i in range(cfg.layers):
                h = 1.0 / (1.0 + np.exp(-(h @ arrays[f"W{i + 1}"].astype(np.float64).T + arrays[f"B{i + 1}"].astype(np.float64).ravel())))
            hbar = h.mean(0)
            hc = h - hbar
            arrays["proto"] = proto
            arrays["Wo"] = (cfg.proto_gain * hc).astype("<f4")
            arrays["Bo"] = (-cfg.proto_gain * (hc @ hbar)).astype("<f4").reshape(-1, 1)
            if fn:
                try:
                    os.makedirs(cfg.cache_dir, exist_ok=True)
                    np.savez(fn, proto=arrays["proto"], Wo=arrays["Wo"], Bo=arrays["Bo"])
                except OSError:
                    pass
    _DNN_CACHE[key] = arrays
    return arrays


def dnn_blob_entries(n_states: int, cfg: DnnConfig) -> dict:
    """The same DNN as the flattened-model entries the export plugin produces from the reference's DNNData
    (julius_b200/plugin/jb200_export.c): layer shapes, row-major (out,in) weights, biases, and the state priors as the
    reference stores them after loading 'id %.8e' lines with fscanf("%e") and log10-nizing (calc_dnn.c:691-703)."""
    a = dnn_arrays(n_states, cfg)
    dims = [cfg.in_dim] + [cfg.hidden] * cfg.layers + [n_states]
    b = {"dnn.n_layers": np.array([cfg.layers + 1], np.int32), "dnn.in_dim": np.array([cfg.in_dim], np.int32),
         "dnn.out_dim": np.array([n_states], np.int32)}
    for i in range(cfg.layers + 1):
        w, bias = (a[f"W{i + 1}"], a[f"B{i + 1}"]) if i < cfg.layers else (a["Wo"], a["Bo"])
        b[f"dnn.l{i}.in"] = np.array([dims[i]], np.int32)
        b[f"dnn.l{i}.out"] = np.array([dims[i + 1]], np.int32)
        b[f"dnn.l{i}.w"] = np.ascontiguousarray(w, np.float32).ravel()
        b[f"dnn.l{i}.b"] = np.ascontiguousarray(bias, np.float32).ravel()
    val = np.array([float(f"{p:.8e}") for p in a["prior"]], np.float32) * np.float32(1.0)
    b["dnn.state_prior"] = np.log10(val.astype(np.float64)).astype(np.float32)
    return b


def write_dnn(outdir: str, n_states: int, cfg: DnnConfig) -> dict:
    """Random-init DNN in the reference's file formats (libsent/src/phmm/calc_dnn.c:225-336,
    libjulius/src/m_jconf.c:579-733): W as C-order (out,in) '<f4' .npy, biases (out,1), prior file
    'state_id prior', and the dnnconf tying them together.  Returns the arrays."""
    os.makedirs(outdir, exist_ok=True)
    arrays = dnn_arrays(n_states, cfg)
    lines = ["feature_type USER", "feature_options -notypecheck", f"feature_len {cfg.feature_len}",
             f"context_len {cfg.context_len}", f"input_nodes {cfg.in_dim}", f"output_nodes {n_states}",
             f"hidden_nodes {cfg.hidden}", f"hidden_layers {cfg.layers}"]
    for i in range(cfg.layers):
        np.save(os.path.join(outdir, f"W{i + 1}.npy"), arrays[f"W{i + 1}"])
        np.save(os.path.join(outdir, f"B{i + 1}.npy"), arrays[f"B{i + 1}"])
        lines += [f"W{i + 1} W{i + 1}.npy", f"B{i + 1} B{i + 1}.npy"]
    np.save(os.path.join(outdir, "Wo.npy"), arrays["Wo"])
    np.save(os.path.join(outdir, "Bo.npy"), arrays["Bo"])
    with open(os.path.join(outdir, "prior.txt"), "w") as f:
        for i, p in enumerate(arrays["prior"]):
            f.write(f"{i} {p:.8e}\n")
    lines += ["output_W Wo.npy", "output_B Bo.npy", "state_prior prior.txt", "state_prior_factor 1.0",
              "state_prior_log10nize yes", "batch_size 1", "num_threads 1"]
    with open(os.path.join(outdir, "dnnconf"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return arrays


def sample_dnn_input(rng: np.random.Generator, n_frames: int, in_dim: int) -> np.ndarray:
    """Smooth random trajectories (AR(1)) so that consecutive frames favour similar states."""
    x = np.empty((n_frames, in_dim), np.float32)
    v = rng.standard_normal(in_dim)
    for t in range(n_frames):
        v = 0.9 * v + 0.45 * rng.standard_normal(in_dim)
        x[t] = v
    return x


def sample_dnn_batch(rng: np.random.Generator, n_utts: int, n_frames: int, in_dim: int) -> list:
    """n_utts independent trajectories of the same process, advanced together (one numpy step per frame for the whole
    batch instead of one per utterance-frame; float32 noise drawn in blocks of frames)."""
    x = np.empty((n_utts, n_frames, in_dim), np.float32)
    v = rng.standard_normal((n_utts, in_dim), dtype=np.float32)
    blk = 50
    for t0 in range(0, n_frames, blk):
        nb = min(blk, n_frames - t0)
        noise = rng.standard_normal((nb, n_utts, in_dim), dtype=np.float32)
        for k in range(nb):
            v = np.float32(0.9) * v + np.float32(0.45) * noise[k]
            x[:, t0 + k, :] = v
    return [x[i] for i in range(n_utts)]
