"""Exact CTC in float64 (plain numpy): an independent semantic reference for the beam decoder.

When the beam is at least as wide as the number of labelings that can have non-zero probability,
the prefix beam search prunes nothing and must compute exact CTC:

  * log_probability of a returned path = log p(l|x), the CTC forward score of its labeling l;
  * the top-P paths = the P most probable labelings;
  * the alignment score sum_t log softmax(x_t)[a_t] = the Viterbi score of l;
  * with a scorer table, log_probability = log p(l|x) + S(l).

With pruning the decoder only loses probability mass, so log_probability <= log p(l|x) and the
alignment score <= log_probability hold at any beam width.

Labelings are tuples of class indices, blank excluded, BEFORE merge_repeated is applied to the
output (the prefix the beam keeps: (a, a) is "a, blank, a"). TEST INFRASTRUCTURE.
"""
import numpy as np

NEG_INF = -np.inf


def log_softmax(x):
    """[..., C] logits -> float64 log-probabilities. -inf logits (masked classes) stay -inf."""
    x = np.asarray(x, np.float64)
    m = np.max(x, axis=-1, keepdims=True)
    return x - (m + np.log(np.sum(np.exp(x - m), axis=-1, keepdims=True)))


def _extend(label, blank):
    """Blank-extended label sequence (blank, l1, blank, l2, ..., blank) and the mask of states that
    may be entered by skipping the blank before them (a label that differs from the one two back)."""
    L = len(label)
    ext = np.full(2 * L + 1, blank, np.int64)
    ext[1::2] = np.asarray(label, np.int64)
    skip = np.zeros(2 * L + 1, bool)
    if L > 1:
        lab = np.asarray(label, np.int64)
        skip[3::2] = lab[1:] != lab[:-1]
    return ext, skip


def _recursion(lp, label, blank, combine):
    lp = np.asarray(lp, np.float64)
    ext, skip = _extend(label, blank)
    S = len(ext)
    if lp.shape[0] == 0:
        return 0.0 if len(label) == 0 else NEG_INF
    a = np.full(S, NEG_INF)
    a[0] = lp[0, blank]
    if S > 1:
        a[1] = lp[0, ext[1]]
    for t in range(1, lp.shape[0]):
        prev1 = np.concatenate(([NEG_INF], a[:-1]))
        prev2 = np.where(skip, np.concatenate(([NEG_INF, NEG_INF], a[:-2]))[:S], NEG_INF)
        a = combine(combine(a, prev1), prev2) + lp[t, ext]
    return float(combine(a[-1], a[-2])) if S > 1 else float(a[-1])


def ctc_forward(lp, label, blank):
    """log p(label | x): the CTC forward recursion over the blank-extended sequence, vectorised over
    states. lp = [T, C] log-probabilities (log_softmax of the logits)."""
    return _recursion(lp, label, blank, np.logaddexp)


def ctc_viterbi(lp, label, blank):
    """Score of the best single frame path (alignment) that collapses to `label`."""
    return _recursion(lp, label, blank, np.maximum)


def alignment_score(lp, alignment, blank, blank_label):
    """sum_t lp[t, a_t] of a returned alignment (blank frames are reported as blank_label)."""
    lp = np.asarray(lp, np.float64)
    cls = [blank if a == blank_label else a for a in alignment]
    return float(sum(lp[t, c] for t, c in enumerate(cls)))


def collapse(alignment, blank_label):
    """CTC collapse of a frame path: merge runs, drop blanks -> the labeling (before merge_repeated)."""
    out, prev = [], None
    for a in alignment:
        if a != blank_label and a != prev:
            out.append(int(a))
        prev = a
    return tuple(out)


def merge_repeats(label):
    """What the decoder outputs for labeling `label` with merge_repeated=True."""
    return tuple(v for i, v in enumerate(label) if i == 0 or v != label[i - 1])


def enumerate_labelings(lp, blank, limit=1 << 16):
    """Every labeling with non-zero probability under lp = [T, C] and its exact (log p, Viterbi) pair,
    by an unpruned prefix search in float64. Only classes that are finite in a frame are expanded in
    it, so vocabularies of 65k classes with a few finite ones per frame stay cheap. Returns a dict
    labeling -> (log p, Viterbi score); raises if more than `limit` labelings exist."""
    lp = np.asarray(lp, np.float64)
    # prefix -> [sum ending in blank, sum ending in label, max ending in blank, max ending in label]
    beams = {(): [0.0, NEG_INF, 0.0, NEG_INF]}
    for t in range(lp.shape[0]):
        row = lp[t]
        pb = row[blank]
        finite = [int(c) for c in np.flatnonzero(np.isfinite(row)) if c != blank]
        nxt = {}

        def acc(key, k, v, comb):
            e = nxt.get(key)
            if e is None:
                e = nxt[key] = [NEG_INF, NEG_INF, NEG_INF, NEG_INF]
            e[k] = comb(e[k], v)

        for pre, (sb, sn, vb, vn) in beams.items():
            tot, vtot = np.logaddexp(sb, sn), max(vb, vn)
            if np.isfinite(pb):
                acc(pre, 0, tot + pb, np.logaddexp)
                acc(pre, 2, vtot + pb, max)
            if pre and np.isfinite(row[pre[-1]]):  # the last label continues
                acc(pre, 1, sn + row[pre[-1]], np.logaddexp)
                acc(pre, 3, vn + row[pre[-1]], max)
            for c in finite:
                ext = pre + (c,)
                if pre and c == pre[-1]:  # a repeat needs a blank in between
                    acc(ext, 1, sb + row[c], np.logaddexp)
                    acc(ext, 3, vb + row[c], max)
                else:
                    acc(ext, 1, tot + row[c], np.logaddexp)
                    acc(ext, 3, vtot + row[c], max)
        beams = {k: v for k, v in nxt.items() if np.isfinite(np.logaddexp(v[0], v[1]))}
        if len(beams) > limit:
            raise ValueError("more than %d labelings with non-zero probability" % limit)
    return {k: (float(np.logaddexp(v[0], v[1])), float(max(v[2], v[3]))) for k, v in beams.items()}


def scorer_term(table, label):
    """S(l) = sum_k table[l_{k-1} + 1][l_k] (row 0: the empty prefix) in float64: what the scorer
    extension point adds to log p(l|x)."""
    table = np.asarray(table, np.float64)
    s, prev = 0.0, -1
    for v in label:
        s += table[prev + 1, v]
        prev = v
    return s


def labeling_count(T, K):
    """Labelings over K non-blank classes that fit in T frames (a repeat needs a blank between):
    the beam width at which nothing can ever be pruned from a decode of T frames."""
    # h[n] = non-empty labelings that need exactly n frames: a new label costs one frame, a repeat two
    h = [0, K] + [0] * max(T - 1, 0)
    for n in range(2, T + 1):
        h[n] = (K - 1) * h[n - 1] + (h[n - 2] if n > 2 else 0)
    return 1 + sum(h[1:T + 1])


def float32_tolerance(T, exact, logits):
    """Largest float32 error allowed between a decoder's log-probability and the float64 value.
    Every frame rounds the normaliser (a sum at the scale of the largest logit) and 1-3 additions and
    LogSumExps at the scale of the running total, so allow 4 ulps (2^-23 relative) of
    (|total| + max |logit| + 1) per frame, over T frames."""
    x = np.asarray(logits, np.float64)
    fin = x[np.isfinite(x)]
    xmax = float(np.max(np.abs(fin))) if fin.size else 0.0
    return 4.0 * 2.0 ** -23 * max(T, 1) * (abs(exact) + xmax + 1.0)


def check_paths(paths, lp, blank, blank_label, merge, exact=False, table=None, tol=None, logits=None,
                labelings=None):
    """Checks the paths one decoder returned for ONE utterance against exact CTC.

    paths  [(decoded, alignment, log_probability)] best first, as returned
    lp     [T_b, C] float64 log-probabilities of the frames the utterance consumed
    exact  True when the beam cannot have pruned anything: the returned labelings must then be the
           most probable ones and every score must equal its exact value; False: the bounds only
    table  scorer table, or None
    Returns a list of failure strings (empty = every check held)."""
    T = lp.shape[0]
    bad = []
    seen = set()
    prev_lp = np.inf
    for p, (dec, ali, got) in enumerate(paths):
        got = float(got)
        lab = collapse(ali, blank_label)
        if len(ali) != T:
            bad.append("path %d: alignment has %d frames, not %d" % (p, len(ali), T))
            continue
        if tuple(dec) != (merge_repeats(lab) if merge else lab):
            bad.append("path %d: decoded %s is not the collapse %s of its alignment" % (p, list(dec), list(lab)))
        if lab in seen:
            bad.append("path %d: labeling %s returned twice" % (p, list(lab)))
        seen.add(lab)
        if got > prev_lp:
            bad.append("path %d: log-probability %r above the previous path's %r" % (p, got, prev_lp))
        prev_lp = got
        s = scorer_term(table, lab) if table is not None else 0.0
        if labelings is not None and lab in labelings:
            fwd, vit = labelings[lab]
        else:
            fwd, vit = ctc_forward(lp, lab, blank), ctc_viterbi(lp, lab, blank)
        want = fwd + s
        tl = tol if tol is not None else float32_tolerance(T, want, logits if logits is not None else lp)
        ascore = alignment_score(lp, ali, blank, blank_label)
        if not got <= want + tl:
            bad.append("path %d %s: log-probability %r above exact %r (+tol %.3g)" % (p, list(lab), got, want, tl))
        if not ascore + s <= got + tl:
            bad.append("path %d %s: alignment score %r above the log-probability %r" % (p, list(lab), ascore + s, got))
        if not ascore <= vit + 1e-9 * (1 + abs(vit)):
            bad.append("path %d %s: alignment score %r above Viterbi %r" % (p, list(lab), ascore, vit))
        if exact:
            if abs(got - want) > tl:
                bad.append("path %d %s: log-probability %r, exact %r (tol %.3g)" % (p, list(lab), got, want, tl))
            if ascore < vit - tl:
                bad.append("path %d %s: alignment score %r, Viterbi %r" % (p, list(lab), ascore, vit))
    if exact and labelings is not None:
        ranked = sorted(((v[0] + (scorer_term(table, l) if table is not None else 0.0)) for l, v in labelings.items()),
                        reverse=True)
        for p, (dec, ali, got) in enumerate(paths):
            lab = collapse(ali, blank_label)
            if lab not in labelings:
                bad.append("path %d: labeling %s has probability 0" % (p, list(lab)))
                continue
            v = labelings[lab][0] + (scorer_term(table, lab) if table is not None else 0.0)
            tl = tol if tol is not None else float32_tolerance(T, v, logits if logits is not None else lp)
            if p < len(ranked) and v < ranked[p] - 2 * tl:
                bad.append("path %d %s: exact %r but the %d-th best labeling has %r" % (p, list(lab), v, p + 1, ranked[p]))
    return bad


def masked_logits(T, B, C, blank, rng, k=(2, 3), span=40, dtype=np.float32):
    """[T, B, C] logits with every class masked (-inf) but the blank and 2-3 non-blank classes per
    frame, drawn from the `span` highest label ids: a large vocabulary whose labelings can still be
    enumerated (and whose label ids need more than a byte)."""
    x = np.full((T, B, C), -np.inf, np.float64)
    x[:, :, blank] = rng.standard_normal((T, B))
    top = np.array([c for c in range(C - 1, -1, -1) if c != blank][:span])
    for t in range(T):
        for b in range(B):
            n = int(rng.integers(k[0], k[1] + 1))
            x[t, b, rng.choice(top, n, replace=False)] = rng.standard_normal(n) * 2
    return x.astype(dtype)


def max_labelings(x, sl, blank):
    """The largest number of labelings with non-zero probability over the utterances of x = [T, B, C]:
    the smallest beam width that prunes nothing."""
    return max(len(enumerate_labelings(log_softmax(x[:sl[b], b]), blank)) for b in range(x.shape[1]))


def ctc_scores_many(lps, labels, blank):
    """[(log p, Viterbi)] of labels[i] under lps[i] ([T_i, C] log-probabilities): ctc_forward and
    ctc_viterbi for many (utterance, labeling) pairs at once, vectorised over pairs and states."""
    N = len(labels)
    if N == 0:
        return []
    Ts = np.array([lp.shape[0] for lp in lps])
    Ls = np.array([len(l) for l in labels])
    Smax, Tmax, C = 2 * int(Ls.max()) + 1, int(Ts.max()), lps[0].shape[1]
    ext = np.full((N, Smax), blank, np.int64)
    skip = np.zeros((N, Smax), bool)
    for i, l in enumerate(labels):
        e, s = _extend(l, blank)
        ext[i, :len(e)], skip[i, :len(s)] = e, s
    live = np.arange(Smax)[None, :] < (2 * Ls + 1)[:, None]
    LP = np.full((N, max(Tmax, 1), C), NEG_INF)
    for i, lp in enumerate(lps):
        LP[i, :lp.shape[0]] = lp
    rows = np.arange(N)[:, None]
    out = np.zeros((N, 2))
    out[Ts == 0, 0] = np.where(Ls[Ts == 0] == 0, 0.0, NEG_INF)
    out[Ts == 0, 1] = out[Ts == 0, 0]
    a = [None, None]
    for t in range(Tmax):
        e = np.where(live, LP[rows, t, ext], NEG_INF)
        for k, comb in enumerate((np.logaddexp, np.maximum)):
            if t == 0:
                v = np.full((N, Smax), NEG_INF)
                v[:, 0] = e[:, 0]
                v[:, 1:2] = e[:, 1:2] if Smax > 1 else v[:, 1:2]
            else:
                prev = a[k]
                p1 = np.concatenate([np.full((N, 1), NEG_INF), prev[:, :-1]], axis=1)
                p2 = np.where(skip, np.concatenate([np.full((N, 2), NEG_INF), prev[:, :-2]], axis=1)[:, :Smax], NEG_INF)
                v = comb(comb(prev, p1), p2) + e
            a[k] = v
            end = Ts == t + 1
            if end.any():
                last = 2 * Ls[end]
                fin = v[end, last]
                pre = np.where(last >= 1, v[end, np.maximum(last - 1, 0)], NEG_INF)
                out[end, k] = comb(fin, pre)
    return [(float(f), float(m)) for f, m in out]
