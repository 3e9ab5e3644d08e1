"""Corpus BLEU as the reference computes it in `compute_bleu` (vae/losses.py:128-134), restated over token ids.

    refs  = [cut(X)[1:-1]    for X in Xbatch]
    cands = [cut(pred)[1:-1] for pred in pred_batch]
    torchtext 0.6 bleu_score(cands, [[r] for r in refs])      # max_n = 4, weights 0.25 each

cut(row) = row up to and including its first EOS, or the whole row if it has none (vae/utils.py:225 tensor2text); [1:-1]
then drops SOS and EOS -- or, in a row without EOS, SOS and the row's last token.  Ids stand for words: the reference's
idx2word is injective, so comparing ids gives the same n-gram matches as comparing strings.
"""
import math
from collections import Counter

MAX_N = 4


def cut(row, eos):
    row = [int(t) for t in row]
    if eos in row:
        row = row[:row.index(eos) + 1]
    return row[1:-1]


def ngrams(tokens, n):
    return Counter(tuple(tokens[i:i + n]) for i in range(len(tokens) - n + 1))


def bleu_counts(refs, cands, eos):
    """[clipped_1..4, total_1..4, cand_len, ref_len] of one batch of (reference row, candidate row) pairs."""
    clipped, total = [0] * MAX_N, [0] * MAX_N
    c_len = r_len = 0
    for ref_row, cand_row in zip(refs, cands, strict=True):
        r, c = cut(ref_row, eos), cut(cand_row, eos)
        c_len += len(c)
        r_len += len(r)
        for n in range(1, MAX_N + 1):
            cg, rg = ngrams(c, n), ngrams(r, n)
            clipped[n - 1] += sum(min(k, rg[g]) for g, k in cg.items())
            total[n - 1] += sum(cg.values())
    return clipped + total + [c_len, r_len]


def bleu_from_counts(counts):
    clipped, total, c_len, r_len = counts[:MAX_N], counts[MAX_N:2 * MAX_N], counts[8], counts[9]
    if min(clipped) == 0:
        return 0.0
    log_p = 0.0
    for n in range(MAX_N):
        log_p += 0.25 * math.log(clipped[n] / total[n])
    return math.exp(min(1.0 - r_len / c_len, 0.0)) * math.exp(log_p)


def corpus_bleu(refs, cands, eos):
    return bleu_from_counts(bleu_counts(refs, cands, eos))
