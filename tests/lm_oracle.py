"""Plain-Python statement of the n-gram LM contract (velocity_asr.NGramLM and the fused beam search), and a
seeded synthetic ARPA writer shared by the LM tests and tools/beam_bench.py.

TEST INFRASTRUCTURE ONLY.  Independent of the package's loader: the ARPA file is read here line by line, the
back-off rule is the textbook recursion, and the beam search offers every token of every hypothesis.  It is a
restatement, not an optimised decoder.  The reference has no counterpart (its lm_scorer is a Python callback)."""
import math

import numpy as np

import velocity_oracle as O


class ArpaLM:
    """lm(prefix, tok) in natural log over token ids:
      values: log10 parsed as a Python float, times math.log(10), rounded once to fp32 (log-probs and bows);
      words: an ARPA word is the vocabulary entry with the same string (the first), "<space>" is " "; "<s>" is a
      context; n-grams with any other word outside the vocabulary are dropped;
      h = ("<s>",) + prefix cut to its last order-1 items; P(w | h) = p(h w) if listed, else bow(h) + P(w | h[1:]),
      bow = 0 when h is not listed; the unigram level falls back to <unk>; summed in fp64 from the listed entry
      found, back-off weights from the shortest backed-off context outward; the sum rounded to fp32."""

    def __init__(self, order, prob, bow, unk):
        self.order, self.prob, self.bow, self.unk = order, prob, bow, unk
        self._memo = {}

    @classmethod
    def from_arpa(cls, path, vocabulary, blank_token: int = O.BLANK_TOKEN):
        ids = {}
        for i, w in enumerate(vocabulary):
            ids.setdefault("<space>" if w == " " else w, i)
        ids["<s>"] = "<s>"
        to_ln = lambda s: float(np.float32(float(s) * math.log(10)))
        prob, bow, unk, order, n = {}, {}, None, 0, 0
        with open(path, encoding="utf-8") as f:
            for line in f:
                parts = line.split()
                if not parts:
                    continue
                if parts[0].startswith("ngram") and len(parts) == 2:
                    order = max(order, int(parts[1].split("=")[0]))
                elif parts[0].endswith("-grams:"):
                    n = int(parts[0][1:-len("-grams:")])
                elif parts[0] == "\\end\\":
                    break
                elif n > 0 and parts[0] != "\\data\\":
                    words = parts[1:1 + n]
                    if n == 1 and words[0] == "<unk>":
                        unk = to_ln(parts[0])
                    if any(w not in ids for w in words):
                        continue
                    key = tuple(ids[w] for w in words)
                    prob[key] = to_ln(parts[0])
                    if len(parts) == n + 2:
                        bow[key] = to_ln(parts[1 + n])
        return cls(order, prob, bow, unk)

    def lm(self, prefix, tok):
        h = (("<s>",) + tuple(prefix))[-(self.order - 1):] if self.order > 1 else ()
        key = (h, tok)
        if key not in self._memo:
            self._memo[key] = self._lm(h, tok)
        return self._memo[key]

    def _lm(self, h, tok):
        bows = []
        while True:
            if h + (tok,) in self.prob:
                base = self.prob[h + (tok,)]
                break
            if not h:
                base = self.unk if self.unk is not None else -math.inf
                break
            bows.append(self.bow.get(h, 0.0))
            h = h[1:]
        s = base
        for b in reversed(bows):                     # shortest backed-off context first
            s = s + b
        return float(np.float32(s))


def ctc_beam_search(logits, beam_width: int = 10, blank_token: int = O.BLANK_TOKEN, lm_scorer=None,
                    lm_weight: float = 0.0):
    """velocity_oracle.ctc_beam_search's rule with shallow fusion, per utterance a list of (tokens, score), best
    first.  One hypothesis per collapsed prefix; every hypothesis offers the blank (prefix kept), its own last token
    again (prefix kept) and every other token (prefix grown); with an ArpaLM and lm_weight > 0 a grown prefix scores
    (score + lp[tok]) + lm_weight * lm(prefix, tok); equal prefixes keep the better score, the earlier offer on a
    tie; the `beam_width` best survive, earlier offers first among equals.  fp64 sums of fp32 log-probs."""
    use_lm = lm_scorer is not None and lm_weight > 0
    out = []
    for lp_utt in O.log_softmax32(logits):
        hyps = [((), 0.0, None)]                       # (prefix, score, last token), ranked
        for lp in lp_utt:
            offers = {}                                # prefix -> [score, last]; dicts keep first-offer order

            def offer(prefix, sc, tok):
                cur = offers.get(prefix)
                if cur is None:
                    offers[prefix] = [sc, tok]
                elif cur[0] < sc:
                    cur[0], cur[1] = sc, tok
            for prefix, sc, last in hyps:
                offer(prefix, sc + float(lp[blank_token]), blank_token)
                for tok in range(lp.shape[0]):
                    if tok == blank_token:
                        continue
                    if tok == last:
                        offer(prefix, sc + float(lp[tok]), tok)
                    elif use_lm:
                        offer(prefix + (tok,), (sc + float(lp[tok])) + lm_weight * lm_scorer.lm(prefix, tok), tok)
                    else:
                        offer(prefix + (tok,), sc + float(lp[tok]), tok)
            ranked = sorted(offers.items(), key=lambda kv: -kv[1][0])[:beam_width]   # stable
            hyps = [(k, v[0], v[1]) for k, v in ranked]
        out.append([(list(k), sc) for k, sc, _ in hyps])
    return out


def write_synthetic_arpa(path, vocabulary, order: int, seed: int = 0, per_order: int = 200,
                         blank_token: int = 0) -> int:
    """A seeded random ARPA LM over `vocabulary`.  It has what a real file has and what the back-off rule must get
    right: about a tenth of the vocabulary without a unigram (they take <unk>), words outside the vocabulary,
    <s> / </s>, -99 entries, back-off weights of both signs, and higher-order n-grams whose contexts are not listed
    one level down.  Returns the number of n-grams."""
    rs = np.random.RandomState(seed)
    words = ["<space>" if w == " " else w for i, w in enumerate(vocabulary) if i != blank_token]
    oov = [f"oov{i}" for i in range(max(2, len(words) // 20))]
    grams = [dict() for _ in range(order + 1)]
    grams[1] = {(w,): None for w in words if rs.rand() > 0.1}
    for w in ["<unk>", "<s>", "</s>"] + oov[: len(oov) // 2]:
        grams[1][(w,)] = None
    pool = words + oov
    for n in range(2, order + 1):
        for _ in range(per_order):
            g = [pool[i] for i in rs.randint(0, len(pool), size=n)]
            if rs.rand() < 0.2:
                g[0] = "<s>"
            if rs.rand() < 0.05:
                g[-1] = "</s>"
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
    return sum(len(g) for g in grams)
