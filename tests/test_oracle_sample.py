"""CPU checks of the device-draw oracle (oracle/sample_oracle.py): its Philox4x32-10 against curand's header and the
Random123 known answers, the two sampling rules branch by branch, and a fixed-seed uniformity test of the draws."""
import numpy as np
import pytest
from scipy import stats

from helpers import golden
from oracle import frcnn_oracle as O
from oracle import sample_oracle as S


def test_philox_equals_curand_header_and_known_answers():
    g = golden("philox")
    assert len(g["out"]) > 4096
    assert np.array_equal(S.philox(g["ctr"], g["key"]), g["out"])
    kat = {0: [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8], 0xFFFFFFFF: [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]}
    for v, want in kat.items():
        got = S.philox(np.full((1, 4), v, np.uint32), np.full((1, 2), v, np.uint32))[0]
        assert got.tolist() == want


def test_words_layout():
    """word j = word j & 3 of counter (j >> 2, img_lo, img_hi, tag), key (seed_lo, seed_hi)"""
    seed, img = 0x1234567890ABCDEF, (7 << 32) + 11
    w = S.words(seed, img, 2, 10)
    ctr = np.array([[2, 11, 7, 2]], np.uint32)
    key = np.array([[0x90ABCDEF, 0x12345678]], np.uint32)
    assert w[8:10].tolist() == S.philox(ctr, key)[0, :2].tolist()
    assert not np.array_equal(S.words(seed, img, 0, 8), S.words(seed, img, 1, 8))


@pytest.mark.parametrize("n_pos,n_neg", [(0, 0), (0, 100), (5, 100), (128, 128), (129, 10), (300, 5000), (40, 200)])
def test_rpn_keep_counts_and_categories(n_pos, n_neg):
    rng = np.random.default_rng(n_pos * 7 + n_neg)
    n = 9 * 38 * 63
    where = rng.permutation(n)
    is_pos = np.zeros(n, bool)
    can_use = np.zeros(n, bool)
    is_pos[where[:n_pos]] = True
    can_use[where[:n_pos + n_neg]] = True
    is_pos[where[n_pos + n_neg:n_pos + n_neg + 50]] = True           # positives that are not usable stay out
    ip0 = is_pos.copy()
    out = S.rpn_keep(can_use, is_pos, seed=3, img=n_pos)
    assert np.array_equal(is_pos, ip0)
    keep_p = min(n_pos, 128)
    keep_q = min(n_neg, 256 - keep_p)
    assert int((out & is_pos).sum()) == keep_p and int((out & ~is_pos).sum()) == keep_q
    assert not (out & ~can_use).any()
    # the same counts as the reference's random.sample switch-off
    ref = O.sample_rpn(is_pos.astype(np.uint8), can_use.astype(np.uint8).copy())
    assert int(ref.sum()) == int(out.sum())


DET_P = [0, 1, 15, 16, 17, 200]
DET_Q = [0, 1, 47, 48, 49, 1900]


@pytest.mark.parametrize("n_pos", DET_P)
@pytest.mark.parametrize("n_neg", DET_Q)
def test_det_samples_branches(n_pos, n_neg):
    rng = np.random.default_rng(1000 * n_pos + n_neg)
    is_pos = np.zeros(n_pos + n_neg, bool)
    is_pos[rng.permutation(n_pos + n_neg)[:n_pos]] = True
    idx = S.det_samples(is_pos, seed=9, img=n_neg, num_rois=64)
    if n_pos + n_neg == 0:
        assert idx.tolist() == [-1] * 64
        return
    np.random.seed(0)
    ref = O.sample_det(is_pos, 64)
    assert len(idx) == len(ref) == 64
    pos_rows = np.where(is_pos)[0]
    n_chosen_pos = min(n_pos, 16)
    assert np.array_equal(is_pos[idx], is_pos[np.array(ref)])       # the reference's row categories, in its order
    head = idx[:n_chosen_pos]
    assert np.all(is_pos[head]) and np.all(np.diff(head) > 0)
    tail = idx[n_chosen_pos:]
    if n_neg >= 64 - n_chosen_pos:
        assert not is_pos[tail].any() and np.all(np.diff(tail) > 0)
    elif n_neg > 0:
        assert not is_pos[tail].any()
    else:
        assert np.array_equal(tail, np.tile(pos_rows, 64 // n_pos + 1)[:64 - n_chosen_pos])
        assert np.array_equal(tail, np.array(ref[n_chosen_pos:]))


def _chi2_inclusion_p(counts, trials, k):
    """p-value of per-element inclusion counts of a uniform k-subset of n elements drawn `trials` times: the
    counts' covariance is T p (1-p) n/(n-1) (I - J/n), so the scaled statistic is chi-square with n-1 dof."""
    n = len(counts)
    p = k / n
    stat = float(((counts - trials * p) ** 2).sum()) / (trials * p * (1 - p) * n / (n - 1))
    return stats.chi2.sf(stat, n - 1)


def test_uniform_inclusion_frequencies():
    trials = 4000
    # RPN: 40 usable positives (keep all) and 300 usable negatives (keep 216)
    n = 9 * 6 * 8
    is_pos = np.zeros(n, bool)
    can_use = np.zeros(n, bool)
    is_pos[:40] = can_use[:340] = True
    neg_counts = np.zeros(300)
    for t in range(trials):
        out = S.rpn_keep(can_use, is_pos, seed=77, img=t)
        assert out[:40].all()
        neg_counts += out[40:340]
    assert _chi2_inclusion_p(neg_counts, trials, 216) > 1e-3
    # detector: 40 positives (keep 16), 100 negatives (keep 48)
    is_pos = np.zeros(140, bool)
    is_pos[::140 // 40][:40] = True
    assert is_pos.sum() == 40
    counts = np.zeros(140)
    for t in range(trials):
        counts[S.det_samples(is_pos, seed=78, img=t)] += 1
    assert _chi2_inclusion_p(counts[is_pos], trials, 16) > 1e-3
    assert _chi2_inclusion_p(counts[~is_pos], trials, 48) > 1e-3
    # with replacement: 10 negatives, 48 draws each -> multinomial cell frequencies
    is_pos = np.zeros(30, bool)
    is_pos[:20] = True
    draws = np.zeros(30)
    for t in range(trials):
        np.add.at(draws, S.det_samples(is_pos, seed=79, img=t)[16:], 1)
    assert stats.chisquare(draws[20:]).pvalue > 1e-3
