"""Oracle of the device-side mini-batch draws (csrc/sample.cu, include/frcnn_b200.h "training mini-batch draws on the
device"): a vectorised numpy Philox4x32-10 and the two sampling rules stated literally.

    word(seed, img, tag, j) = word j & 3 of Philox4x32_10(ctr = (j >> 2, img_lo, img_hi, tag), key = (seed_lo, seed_hi))

tests/golden/philox.npz pins `philox` against curand's own header compiled for the host (make_golden_philox.py).
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
TAG_RPN, TAG_DET, TAG_DET_DRAW = 0, 1, 2
_LO = np.uint64(0xFFFFFFFF)


def philox(ctr, key):
    """ctr (..., 4) uint32, key (..., 2) uint32 -> (..., 4) uint32: ten rounds of Philox4x32 (Salmon et al., SC'11)."""
    c = [np.asarray(ctr, np.uint32)[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = (np.asarray(key, np.uint32)[..., i].copy() for i in range(2))
    for r in range(10):
        if r:
            k0, k1 = k0 + W0, k1 + W1                 # uint32 wrap-around
        p0, p1 = M0 * c[0], M1 * c[2]                 # exact 64-bit products of 32-bit operands
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0.astype(np.uint64), p1 & _LO,
             (p0 >> np.uint64(32)) ^ c[3] ^ k1.astype(np.uint64), p0 & _LO]
    return np.stack(c, axis=-1).astype(np.uint32)


def words(seed, img, tag, n):
    """the first n words of image `img`'s stream `tag` -> (n,) uint32"""
    seed, img = int(seed) & 0xFFFFFFFFFFFFFFFF, int(img) & 0xFFFFFFFFFFFFFFFF
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([g, np.full_like(g, img & 0xFFFFFFFF), np.full_like(g, img >> 32), np.full_like(g, tag)], axis=1)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint64), (len(g), 2))
    return philox(ctr.astype(np.uint32), key.astype(np.uint32)).reshape(-1)[:n]


def _smallest(idx, u, keep):
    """the `keep` entries of idx with the smallest (u, idx), in ascending idx order"""
    order = np.lexsort((idx, u[idx]))
    return np.sort(idx[order[:keep]])


def rpn_keep(can_use, is_pos, seed, img, max_pos=128, sample_size=256):
    """rpn_util.py:324-350 with the device RNG for one image's flat (own-map) anchors -> the new can_use (bool copy).
    keep_p = min(|P|, max_pos), keep_q = min(|Q|, sample_size - keep_p); the kept anchors of each category are those
    with the smallest (word(i, tag 0), i); is_pos is not an output."""
    cu, ip = np.asarray(can_use).astype(bool), np.asarray(is_pos).astype(bool)
    u = words(seed, img, TAG_RPN, len(cu))
    pos, neg = np.where(cu & ip)[0], np.where(cu & ~ip)[0]
    keep_p = min(len(pos), max_pos)
    keep_q = min(len(neg), sample_size - keep_p)
    out = np.zeros_like(cu)
    out[_smallest(pos, u, keep_p)] = True
    out[_smallest(neg, u, keep_q)] = True
    return out


def det_samples(is_pos, seed, img, num_rois=64):
    """det_util.py:260-306 with the device RNG for one image's label_rois rows (is_pos (m,)) -> (num_rois,) int32 row
    index, all -1 when m == 0."""
    is_pos = np.asarray(is_pos).astype(bool)
    m, s = len(is_pos), int(num_rois)
    if m == 0:
        return np.full(s, -1, np.int32)
    u = words(seed, img, TAG_DET, m)
    pos, neg = np.where(is_pos)[0], np.where(~is_pos)[0]
    want_pos = s // 4
    chosen_pos = pos if len(pos) < want_pos else _smallest(pos, u, want_pos)
    want_neg = s - len(chosen_pos)
    if len(neg) >= want_neg:
        chosen_neg = _smallest(neg, u, want_neg)
    elif len(neg) > 0:                                # with replacement; bias of each row <= |Q| / 2^32
        v = words(seed, img, TAG_DET_DRAW, want_neg).astype(np.uint64)
        chosen_neg = neg[(v * np.uint64(len(neg))) >> np.uint64(32)]
    else:
        chosen_neg = np.tile(pos, want_neg // len(pos) + 1)[:want_neg]
    return np.concatenate([chosen_pos, chosen_neg]).astype(np.int32)
