"""numpy restatement of the CTC forced-alignment and log-likelihood rule of include/vasr.h (vasr_ctc_align,
vasr_ctc_log_likelihood).  It shares no code with the package.

The lattice is the CTC expansion blank, y0, blank, y1, ..., blank (2U + 1 states).  Each frame is one vectorised
step: the candidates stay / s-1 / s-2 are stacked in that order, so np.argmax (the first maximum) is the rule's
"first candidate with the strictly greatest value" tie break.  Scores are fp64 sums of the given lp values in time
order; lp is read as it is given (fp32 for the device comparisons)."""
import numpy as np

NEG = -np.inf


def lattice(y, blank):
    """(labels (S,), skip allowed (S,)) of target y."""
    y = np.asarray(y, np.int64).reshape(-1)
    S = 2 * y.size + 1
    lab = np.full(S, blank, np.int64)
    lab[1::2] = y
    skip = np.zeros(S, bool)
    skip[3::2] = y[1:] != y[:-1]
    return lab, skip


def _candidates(delta, skip, out):
    out[0] = delta
    out[1, 0] = NEG
    out[1, 1:] = delta[:-1]
    out[2, :2] = NEG
    out[2, 2:] = np.where(skip[2:], delta[:-2], NEG)
    return out


def viterbi(lp, y, blank=0):
    """lp (T, V) log-probs of one utterance's frames, y its target.  Returns (frame labels (T,) int32, frame log-probs
    (T,) of lp's dtype, path score as a Python float)."""
    lp = np.asarray(lp)
    T = lp.shape[0]
    lab, skip = lattice(y, blank)
    S = lab.size
    U = (S - 1) // 2
    delta = np.full(S, NEG)
    delta[0] = 0.0
    Sp = (S + 3) // 4 * 4
    bp = np.zeros((T, Sp // 4), np.uint8)              # 2 bits per state, as the device keeps them
    cand = np.empty((3, S))
    arg = np.zeros(Sp, np.uint8)
    idx = np.arange(S)
    for t in range(T):
        _candidates(delta, skip, cand)
        a = np.argmax(cand, axis=0)
        delta = cand[a, idx] + lp[t, lab].astype(np.float64)
        arg[:S] = a
        bp[t] = arg[0::4] | (arg[1::4] << 2) | (arg[2::4] << 4) | (arg[3::4] << 6)
    fin = 2 * U
    if U > 0 and not delta[2 * U] > delta[2 * U - 1]:
        fin = 2 * U - 1
    score = float(delta[fin])
    labels = np.full(T, -1, np.int32)
    flp = np.zeros(T, lp.dtype)
    if score == NEG:
        return labels, flp, score
    s = fin
    for t in range(T - 1, -1, -1):
        labels[t] = lab[s]
        flp[t] = lp[t, lab[s]]
        s -= int(bp[t, s >> 2] >> (2 * (s & 3))) & 3
    return labels, flp, score


def log_likelihood(lp, y, blank=0):
    """log sum over every alignment of y, same lattice, log-add m + log sum exp(x - m) in fp64."""
    lp = np.asarray(lp)
    lab, skip = lattice(y, blank)
    S = lab.size
    U = (S - 1) // 2
    alpha = np.full(S, NEG)
    alpha[0] = 0.0
    cand = np.empty((3, S))
    with np.errstate(invalid="ignore", divide="ignore"):
        for t in range(lp.shape[0]):
            _candidates(alpha, skip, cand)
            m = cand.max(axis=0)
            fin = m != NEG
            ms = np.where(fin, m, 0.0)
            total = (np.exp(cand[0] - ms) + np.exp(cand[1] - ms)) + np.exp(cand[2] - ms)
            alpha = np.where(fin, (ms + np.log(total)) + lp[t, lab].astype(np.float64), NEG)
    last = alpha[2 * U - 1] if U > 0 else NEG
    tail = alpha[2 * U]
    m = max(last, tail)
    if m == NEG:
        return NEG
    return float(m + np.log(np.exp(last - m) + np.exp(tail - m)))


def spans(labels, blank=0):
    """[start, end) frame range of each token of a best path's frame labels."""
    x = np.asarray(labels)
    out, t = [], 0
    while t < x.size:
        if x[t] != blank and x[t] >= 0:
            e = t
            while e + 1 < x.size and x[e + 1] == x[t]:
                e += 1
            out.append((t, e + 1))
            t = e + 1
        else:
            t += 1
    return out
