"""The corpus-BLEU oracle (oracle/bleu.py: vae/losses.py compute_bleu = torchtext 0.6 bleu_score) on hand-worked cases.
Token ids: 2 = SOS, 3 = EOS, 0 = PAD; a..f = 5..10."""
import math

import pytest

from oracle import bleu as OB

SOS, EOS, PAD = 2, 3, 0
a, b, c, d, e, f = 5, 6, 7, 8, 9, 10


def row(*toks, T=None):
    r = [SOS, *toks, EOS]
    return r + [PAD] * ((T or len(r)) - len(r))


def test_cut_drops_sos_eos_and_the_last_token_of_a_row_without_eos():
    assert OB.cut(row(a, b, c, T=8), EOS) == [a, b, c]
    assert OB.cut([SOS, a, b, c, d], EOS) == [a, b, c]          # no EOS: [1:-1] removes the last real token
    assert OB.cut([SOS, EOS, a, EOS], EOS) == []                # cut at the FIRST EOS
    assert OB.cut([SOS], EOS) == [] and OB.cut([a, EOS], EOS) == []


def test_identical_corpus_scores_one():
    refs = [row(a, b, c, d, e, T=9), row(b, c, d, e, f, a)]
    assert OB.corpus_bleu(refs, refs, EOS) == 1.0


def test_repeated_unigrams_are_clipped_by_the_reference_count():
    counts = OB.bleu_counts([row(a, b)], [row(a, a, a, a)], EOS)
    assert counts == [1, 0, 0, 0, 4, 3, 2, 1, 4, 2]
    assert OB.bleu_from_counts(counts) == 0.0
    # clipped but all n-gram orders matched: p = 5/6, 4/5, 3/4, 2/3, no brevity penalty
    got = OB.corpus_bleu([row(a, b, c, d, e)], [row(a, a, b, c, d, e)], EOS)
    assert got == pytest.approx((1 / 3) ** 0.25, rel=1e-15)


def test_brevity_penalty_when_the_candidate_is_shorter():
    got = OB.corpus_bleu([row(a, b, c, d, e, f)], [row(a, b, c, d, e)], EOS)
    assert got == pytest.approx(math.exp(1 - 6 / 5), rel=1e-15)
    # a longer candidate is not penalised for length (only its precisions drop)
    assert OB.corpus_bleu([row(a, b, c, d, e)], [row(a, b, c, d, e, f)], EOS) == pytest.approx((5 / 6 * 4 / 5 * 3 / 4 * 2 / 3) ** 0.25)


def test_any_zero_ngram_precision_gives_zero():
    assert OB.corpus_bleu([row(a, b, c)], [row(a, b, c)], EOS) == 0.0           # no 4-grams in a 3-token corpus
    assert OB.corpus_bleu([row(a, b, c, d)], [row(d, c, b, a)], EOS) == 0.0     # unigrams match, bigrams do not
    assert OB.corpus_bleu([row(a, b, c, d)], [row()], EOS) == 0.0               # empty candidate


def test_row_without_eos_uses_the_last_token_quirk():
    ref_no_eos = [SOS, a, b, c, d, e]            # -> a b c d (e is dropped as if it were EOS)
    assert OB.corpus_bleu([ref_no_eos], [row(a, b, c, d)], EOS) == 1.0
    assert OB.corpus_bleu([ref_no_eos], [row(a, b, c, d, e)], EOS) == pytest.approx((4 / 5 * 3 / 4 * 2 / 3 * 1 / 2) ** 0.25)


def test_corpus_bleu_is_not_the_mean_of_sentence_bleus():
    refs, cands = [row(a, b, c, d), row(e, f, a)], [row(a, b, c, d), row(e, f, a)]
    sentence = [OB.corpus_bleu([r], [h], EOS) for r, h in zip(refs, cands)]
    assert sentence == [1.0, 0.0]
    assert OB.corpus_bleu(refs, cands, EOS) == 1.0      # the 3-token pair adds 1-3-grams, and the first pair the 4-gram


def test_counts_of_a_corpus_are_the_sum_of_its_batches():
    refs = [row(a, b, c, d, a, b), row(c, c, d), row(f, e, d, c, b)]
    cands = [row(a, b, a, b, c, d), row(c, d, c), row(f, e, d)]
    whole = OB.bleu_counts(refs, cands, EOS)
    parts = [OB.bleu_counts(refs[:1], cands[:1], EOS), OB.bleu_counts(refs[1:], cands[1:], EOS)]
    assert whole == [x + y for x, y in zip(*parts)]
