"""CPU: the oracle's restatement of the ray march's jitter stream (Philox4x32-10 -> [N, S] uniforms), pinned to the published
Random123 known-answer vectors and to the counter layout the kernel uses. tests/test_gpu_ray_march.py compares the kernel with it."""
import numpy as np
import pytest

from oracle import nof_oracle as O

# Random123 kat_vectors, philox4x32_10: counter, key, expected output
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize('ctr,key,want', KAT)
def test_philox_known_answers(ctr, key, want):
    got = O.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))
    assert got.dtype == np.uint32
    assert [int(w) for w in got] == list(want)


def test_philox_is_vectorised_over_counters():
    ctrs = np.array([k[0] for k in KAT], np.uint32)
    keys = np.array([k[1] for k in KAT], np.uint32)
    np.testing.assert_array_equal(O.philox4x32_10(ctrs, keys), np.array([k[2] for k in KAT], np.uint32))


def _unit(words):
    return np.array([(int(w) >> 8) * 2.0 ** -24 for w in words], np.float32)


def test_march_uniforms_range_and_grid():
    u = O.march_uniforms(300, 37, 0x5DEECE66D, 12345)
    assert u.shape == (300, 37) and u.dtype == np.float32
    assert u.min() >= 0.0 and u.max() <= 1.0 - 2.0 ** -24
    k = u.astype(np.float64) * 2.0 ** 24
    np.testing.assert_array_equal(k, np.round(k))          # multiples of 2^-24: the top 24 bits of one word
    assert 0.45 < u.mean() < 0.55 and len(np.unique(u)) > 0.99 * u.size


def test_march_uniforms_follow_the_counter_layout():
    seed, offset = 0x89ABCDEF_01234567, 0x00000005_FFFFFFFE
    N, S = 6, 11
    u = O.march_uniforms(N, S, seed, offset)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32)
    for r in range(N):
        for g in range((S + 3) // 4):
            w = O.philox4x32_10(np.array([r, g, offset & 0xFFFFFFFF, offset >> 32], np.uint32), key)
            n = min(4, S - 4 * g)
            np.testing.assert_array_equal(u[r, 4 * g:4 * g + n], _unit(w)[:n])
    # the words past S in the last group are dropped, not shifted into the next row
    np.testing.assert_array_equal(O.march_uniforms(N, 12, seed, offset)[:, :S], u)


@pytest.mark.parametrize('what', ['seed_hi', 'offset_hi', 'offset_lo', 'ray'])
def test_march_uniforms_depend_on_every_counter_and_key_word(what):
    seed, offset = 0x5DEECE66D, 7
    base = O.march_uniforms(4, 8, seed, offset)
    if what == 'seed_hi':
        other = O.march_uniforms(4, 8, seed + (1 << 32), offset)
    elif what == 'offset_hi':
        other = O.march_uniforms(4, 8, seed, offset + (1 << 32))
    elif what == 'offset_lo':
        other = O.march_uniforms(4, 8, seed, offset + 1)
    else:                                               # ray r of a batch is ray r + 1 of a batch that starts one row earlier
        other = O.march_uniforms(5, 8, seed, offset)[1:]
    assert (other != base).all()
