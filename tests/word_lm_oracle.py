"""Plain-Python statement of the word-level LM contract (velocity_asr.WordNGramLM and the word-fused beam search),
a seeded synthetic word-ARPA writer and logits that spell a given word sequence.

TEST INFRASTRUCTURE ONLY.  Independent of the package: word scoring is lm_oracle.ArpaLM with the file's word list as
its "vocabulary"; spelling, the history of a prefix and the search are restated here, and the search offers every
token of every hypothesis.  include/vasr.h states the same rule."""
import numpy as np

import lm_oracle as LO
import velocity_oracle as O


def unigram_words(path):
    """The words of the 1-gram section, first occurrence first, <s> excluded: word id = index."""
    words, seen, in_uni = [], set(), False
    with open(path, encoding="utf-8") as f:
        for line in f:
            parts = line.split()
            if not parts:
                continue
            if in_uni and parts[0].startswith("\\"):
                break
            if parts[0] == "\\1-grams:":
                in_uni = True
            elif in_uni and len(parts) >= 2 and parts[1] != "<s>" and parts[1] not in seen:
                seen.add(parts[1])
                words.append(parts[1])
    return words


class WordLM:
    """Words spelled one token per character (the first vocabulary entry with that string, neither the blank nor
    the delimiter d); the lexicon = spellable unigram words other than <s>, </s>, <unk>.  A prefix splits at each d
    into runs; its non-empty runs before the last d are its words, the run after the last d is the pending run u;
    word(run) = the lexicon word it spells, else <unk>; lm(h, w) = ArpaLM over word ids with h = the words."""

    def __init__(self, path, vocabulary, blank_token=O.BLANK_TOKEN, word_delimiter=" ", lexicon_constrained=False):
        self.words = unigram_words(path)
        self.ids = {w: i for i, w in enumerate(self.words)}
        self.arpa = LO.ArpaLM.from_arpa(path, self.words)
        self.order = self.arpa.order
        self.blank, self.d = blank_token, vocabulary.index(word_delimiter)
        self.constrained = lexicon_constrained
        first = {}
        for i, v in enumerate(vocabulary):
            first.setdefault(v, i)
        self.lexicon = {}                              # spelling (token tuple) -> word id
        for w, i in self.ids.items():
            if w in ("<unk>", "</s>"):
                continue
            toks = [first.get(ch) for ch in w]
            if all(t is not None and t not in (blank_token, self.d) for t in toks):
                self.lexicon[tuple(toks)] = i
        self.prefixes = {sp[:n] for sp in self.lexicon for n in range(len(sp) + 1)}
        self.unk = self.ids.get("<unk>")
        self.eos = self.ids.get("</s>", self.unk)

    def word(self, run):
        return self.lexicon.get(tuple(run), self.unk)

    def lm(self, history, w):
        return self.arpa.lm(tuple(history), w)

    def log_prob(self, history, word):
        """lm(history, word) over strings; unknown strings are <unk>."""
        wid = lambda s: self.ids.get(s, self.unk)
        return self.lm([wid(s) for s in history], wid(word))

    def split(self, prefix):
        """(history word ids, pending run u) of a prefix"""
        runs, cur = [], []
        for t in prefix:
            if t == self.d:
                runs.append(cur)
                cur = []
            else:
                cur.append(t)
        return tuple(self.word(r) for r in runs if r), tuple(cur)


def ctc_beam_search(logits, beam_width, blank_token, lm, lm_weight, word_score):
    """The word-fused prefix beam search, per utterance a list of (tokens, score), best first.  Offers, fp64 sums in
    this order: blank and the repeat of `last` keep the prefix with score + lp; d extends with score + lp[d], plus
    lm_weight * lm(h, word(u)) and then word_score when u is non-empty (constrained: only if u is a lexicon word);
    any other token t extends with score + lp[t] (constrained: only if u + t is a prefix of a lexicon spelling).
    Max-merge, first offer wins a tie, the stable top beam_width.  End: close u (constrained: drop the beam when u
    is not a lexicon word), add lm_weight * lm(h, </s>), sort stably by that score."""
    d = lm.d
    out = []
    for lp_utt in O.log_softmax32(logits):
        hyps = [((), 0.0, None)]
        for lp in lp_utt:
            offers = {}

            def offer(prefix, sc, tok):
                cur = offers.get(prefix)
                if cur is None:
                    offers[prefix] = [sc, tok]
                elif cur[0] < sc:
                    cur[0], cur[1] = sc, tok
            for prefix, sc, last in hyps:
                offer(prefix, sc + float(lp[blank_token]), blank_token)
                hist, u = lm.split(prefix)
                for tok in range(lp.shape[0]):
                    if tok == blank_token:
                        continue
                    if tok == last:
                        offer(prefix, sc + float(lp[tok]), tok)
                    elif tok == d:
                        if not u:
                            offer(prefix + (d,), sc + float(lp[d]), d)
                        elif not lm.constrained or u in lm.lexicon:
                            offer(prefix + (d,), ((sc + float(lp[d])) + lm_weight * lm.lm(hist, lm.word(u)))
                                  + word_score, d)
                    elif not lm.constrained or u + (tok,) in lm.prefixes:
                        offer(prefix + (tok,), sc + float(lp[tok]), tok)
            ranked = sorted(offers.items(), key=lambda kv: -kv[1][0])[:beam_width]
            hyps = [(k, v[0], v[1]) for k, v in ranked]
        final = []
        for prefix, sc, _ in hyps:
            hist, u = lm.split(prefix)
            if u:
                if lm.constrained and u not in lm.lexicon:
                    continue
                sc = (sc + lm_weight * lm.lm(hist, lm.word(u))) + word_score
                hist = hist + (lm.word(u),)
            final.append((list(prefix), sc + lm_weight * lm.lm(hist, lm.eos)))
        out.append(sorted(final, key=lambda r: -r[1]))
    return out


def write_synthetic_word_arpa(path, letters, order, seed=0, n_words=40, per_order=200, unk=True):
    """A seeded random word-level ARPA LM: random words over `letters`, words with characters outside any default
    vocabulary (unspellable), <unk> (unless unk=False), <s>, </s>, n-grams over words missing from the unigrams,
    -99 entries and back-off weights of both signs.  Returns the spellable words."""
    rs = np.random.RandomState(seed)
    letters = list(letters)
    cap = sum(len(letters) ** n for n in range(1, 5))
    words = set()
    while len(words) < min(n_words, cap):
        words.add("".join(rs.choice(letters, size=rs.randint(1, 5))))
    words = sorted(words)
    unspellable = ["#" + w for w in words[:3]] + ["café", "x~y"]
    oov = [f"oov{i}" for i in range(4)]
    grams = [dict() for _ in range(order + 1)]
    for w in words + unspellable + (["<unk>"] if unk else []) + ["<s>", "</s>"]:
        grams[1][(w,)] = None
    pool = words + unspellable + oov + ["</s>"]
    for n in range(2, order + 1):
        for _ in range(per_order):
            g = [pool[i] for i in rs.randint(0, len(pool), size=n)]
            if rs.rand() < 0.2:
                g[0] = "<s>"
            grams[n][tuple(g)] = None
    lines = ["\\data\\"] + [f"ngram {n}={len(grams[n])}" for n in range(1, order + 1)]
    for n in range(1, order + 1):
        lines += ["", f"\\{n}-grams:"]
        for g in grams[n]:
            lp = -99.0 if (g == ("<s>",) or rs.rand() < 0.03) else rs.uniform(-3.0, -0.05)
            line = f"{lp:.4f}\t{' '.join(g)}"
            if n < order and rs.rand() < 0.7:
                line += f"\t{rs.uniform(-1.0, 0.3):.4f}"
            lines.append(line)
    lines += ["", "\\end\\", ""]
    with open(path, "w", encoding="utf-8") as f:
        f.write("\n".join(lines))
    return words


def spelled_logits(vocabulary, words, blank_token=0, delimiter=" ", frames=2, peak=4.0, noise=1.0, seed=0):
    """(L, V) fp32 logits whose peaks spell delimiter.join(words): each character held `frames` frames, a blank
    between repeated characters and at the end, Gaussian noise on every entry."""
    rs = np.random.RandomState(seed)
    toks = [vocabulary.index(ch) for ch in delimiter.join(words)]
    seq = []
    for i, t in enumerate(toks):
        if i and toks[i - 1] == t:
            seq.append(blank_token)
        seq += [t] * frames
    seq.append(blank_token)
    lg = rs.standard_normal((len(seq), len(vocabulary))) * noise
    lg[np.arange(len(seq)), seq] += peak
    return lg.astype(np.float32)
