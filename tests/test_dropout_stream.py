"""Statistical properties of the host port of the kernels' dropout stream (oracle/dropout_stream.py).

The port is pinned bit for bit to the kernels by tests/test_gpu_dropout.py; these checks need no GPU.  Each rate is
checked within 5 standard deviations of its binomial expectation."""
import numpy as np
import pytest

from oracle import dropout_stream as ds

N = 1 << 20
SEED = (12345 * 0x9E3779B97F4A7C15 + 7) & 0xFFFFFFFFFFFFFFFF      # models.py's seed formula: high 32 bits set
OFFSET = 3


def _within_5_sigma(rate, expect, n):
    sigma = np.sqrt(expect * (1.0 - expect) / n)
    assert abs(rate - expect) <= 5.0 * sigma, (rate, expect, sigma)


def _agreement(a, b, p):
    """(a != 0) == (b != 0) at the rate p^2 + (1-p)^2 of two independent masks."""
    a, b = np.asarray(a).reshape(-1), np.asarray(b).reshape(-1)
    assert a.size == b.size
    _within_5_sigma(float(np.mean((a != 0) == (b != 0))), p * p + (1 - p) * (1 - p), a.size)


@pytest.mark.parametrize("p", [0.1, 0.5, 0.8])
def test_keep_fraction(p):
    m = ds.multipliers(np.arange(N, dtype=np.uint64), p, SEED, OFFSET)
    _within_5_sigma(float(np.mean(m != 0)), 1.0 - p, N)


@pytest.mark.parametrize("p", [0.1, 0.5, 0.8])
def test_multiplier_takes_exactly_two_values(p):
    m = ds.multipliers(np.arange(N, dtype=np.uint64), p, SEED, OFFSET)
    assert m.dtype == np.float32
    vals = set(np.unique(m).tolist())
    kept = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
    assert vals == {0.0, kept}
    assert abs(kept - 1.0 / (1.0 - p)) <= 1e-6 * kept


def test_fmix32_matches_murmur3_reference_values():
    # murmur3 fmix32: 0 -> 0, and these values worked out by hand with Python's unbounded integers
    def ref(h):
        h ^= h >> 16
        h = (h * 0x85EBCA6B) & 0xFFFFFFFF
        h ^= h >> 13
        h = (h * 0xC2B2AE35) & 0xFFFFFFFF
        return h ^ (h >> 16)
    xs = np.array([0, 1, 0x7F4A7C15, 0x9E3779B9, 0xFFFFFFFF, 123456789], dtype=np.uint32)
    assert ds.fmix32(xs).tolist() == [ref(int(v)) for v in xs]


def test_ids_with_high_bits_use_them():
    """The upper 32 bits of an id enter the hash: ids k and 2^32 + k draw independent multipliers."""
    lo = np.arange(N, dtype=np.uint64)
    _agreement(ds.multipliers(lo, 0.5, SEED, OFFSET), ds.multipliers(lo + np.uint64(1 << 32), 0.5, SEED, OFFSET), 0.5)


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_successive_offsets_are_independent(p):
    ids = np.arange(N, dtype=np.uint64)
    _agreement(ds.multipliers(ids, p, SEED, OFFSET), ds.multipliers(ids, p, SEED, OFFSET + 1), p)
    # offsets past 2^32 (the high word of the offset enters k1)
    big = (1 << 32) + 5
    _agreement(ds.multipliers(ids, p, SEED, big), ds.multipliers(ids, p, SEED, big - (1 << 32)), p)


def test_gru_sites_are_independent():
    B, L, H = 16, 128, 128          # 2^19 elements a site
    m0 = ds.gru_masks(B, L, H, 3, 0.5, SEED, OFFSET)
    _agreement(m0[0], m0[1], 0.5)


def test_head_site_independent_of_gru_site_0():
    B = N // ds.HEAD_HID
    head = ds.head_mask(B, 0.5, SEED, OFFSET)
    site0 = ds.multipliers(np.arange(B * ds.HEAD_HID, dtype=np.uint64), 0.5, SEED, OFFSET)
    _agreement(head, site0, 0.5)


def test_direction_halves_are_independent():
    B, L, H = 64, 128, 64
    m = ds.gru_masks(B, L, H, 2, 0.5, SEED, OFFSET)[0]
    _agreement(m[..., :H], m[..., H:], 0.5)


def test_data_parallel_rank_seeds_are_independent():
    """DataParallelTrainStep seeds rank r with model._rng_seed ^ (0x9E3779B9 * (r + 1)) (parallel.py)."""
    ids = np.arange(N, dtype=np.uint64)
    s0, s1 = ((SEED ^ (0x9E3779B9 * (r + 1))) & 0xFFFFFFFFFFFFFFFF for r in (0, 1))
    _agreement(ds.multipliers(ids, 0.5, s0, OFFSET), ds.multipliers(ids, 0.5, s1, OFFSET), 0.5)


def test_fused_step_seed_independent_of_autograd_seed():
    """FusedTrainStep seeds with model._rng_seed ^ 0x5DEECE66D (trainer.py), the autograd path with model._rng_seed."""
    ids = np.arange(N, dtype=np.uint64)
    _agreement(ds.multipliers(ids, 0.5, SEED, OFFSET), ds.multipliers(ids, 0.5, SEED ^ 0x5DEECE66D, OFFSET), 0.5)


def test_site_id_ranges_do_not_overlap_at_the_largest_shape():
    """At the longest window the kernels accept (T = 16384), the largest hidden size (128), B = 4096 windows and the
    deepest stack (8 layers), every site's id range is disjoint from every other's, and no id wraps past 2^64."""
    T, H, B, layers = 16384, 128, 4096, 8
    L = ds.gru_seq_len(T)
    assert L == 1024 and ds.gru_seq_len(3840) == 240 and ds.gru_seq_len(1004) == 63
    ranges = [(l * ds.LAYER_STRIDE, l * ds.LAYER_STRIDE + B * L * 2 * H) for l in range(layers - 1)]
    ranges.append((ds.HEAD_BASE, ds.HEAD_BASE + B * ds.HEAD_HID))
    ranges.sort()
    for (lo0, hi0), (lo1, hi1) in zip(ranges, ranges[1:]):
        assert hi0 <= lo1, ((lo0, hi0), (lo1, hi1))
    assert ranges[-1][1] < 1 << 64
    # the helpers produce exactly these ids
    assert int(ds.gru_site_ids(1, 2, 3, 32)[1, 2, 63]) == ds.LAYER_STRIDE + (1 * 3 + 2) * 64 + 63
    assert int(ds.head_site_ids(3)[2, 5]) == ds.HEAD_BASE + 2 * 64 + 5
