"""The exact BLAS-speed DBSCAN reference and the planted match tables of tests/test_gram_dbscan_gpu.py, on the CPU: the
fast reference against the oracle's DBSCAN (itself pinned to sklearn in test_oracle_golden.py), and the plant against
what it claims to contain."""
import numpy as np
import pytest

from oracle import keymask_oracle as ko
from tests.gram_dbscan_reference import dbscan_hamming_fast, expected_grouping, plant_census, planted_video

PARAMS = [(0.2, 5), (0.1, 5), (0.1, 3), (0.05, 5)]


def _random_problem(rng, it):
    n = 1 if it % 50 == 0 else int(rng.integers(1, 120))
    d = int(rng.choice([1, 2, 3, 7, 10, 31, 32, 33, 50, 51, 64, 100, 299, 300]))
    base = rng.random((int(rng.integers(1, 6)), d)) < rng.choice([0.05, 0.3, 0.5])
    X = base[rng.integers(0, len(base), n)] ^ (rng.random((n, d)) < rng.choice([0.0, 0.01, 0.03, 0.1]))
    if it % 3 == 0:
        X[rng.integers(0, n, max(1, n // 3))] = False              # all-zero rows
    return X


@pytest.mark.parametrize("eps,ms", PARAMS)
def test_fast_dbscan_equals_oracle_on_random_problems(eps, ms):
    """60 random problems per (eps, min_samples), 240 in all: n = 1, widths 1 to 300 across word edges, all-zero rows,
    clusters of near-copies at several noise levels."""
    rng = np.random.default_rng(int(eps * 1000) + ms)
    for it in range(60):
        X = _random_problem(rng, it)
        assert np.array_equal(dbscan_hamming_fast(X, eps, ms), ko.dbscan_hamming(X, eps, ms)), (it, X.shape)


@pytest.mark.parametrize("eps,ms", PARAMS)
@pytest.mark.parametrize("d", [10, 40, 61, 300])
def test_fast_dbscan_equals_oracle_at_the_distance_and_count_edges(eps, ms, d):
    """Pairs at exactly kmax and kmax + 1, a row with exactly min_samples - 1 neighbours next to one with exactly
    min_samples, a border row between two cores: the thresholds sit exactly where both implementations decide."""
    rng = np.random.default_rng(d * 7 + ms)
    k = ko.hamming_kmax(d, eps)
    rows = []
    for extra, nsp in ((0, ms - 1), (0, ms - 2), (1, ms - 1)):
        h = rng.random(d) < 0.5
        cols = rng.permutation(d)
        rows.append(h)
        for i in range(nsp):                                     # spokes at distance k (+ extra) from the hub
            x = h.copy()
            x[cols[i * (k + extra):(i + 1) * (k + extra)] if (i + 1) * (k + extra) <= d else cols[:k + extra]] ^= True
            rows.append(x)
    h = rng.random(d) < 0.5
    if 2 * k <= d and k > 0:
        D = rng.permutation(d)[:2 * k]
        hB = h.copy(); hB[D] ^= True
        for _ in range(ms):
            rows += [h.copy(), hB.copy()]
        mid = h.copy(); mid[D[:k]] ^= True
        rows.append(mid)
    rows.append(np.zeros(d, bool))
    X = np.asarray(rows)
    for perm in (np.arange(len(X)), rng.permutation(len(X))):
        Y = X[perm]
        assert np.array_equal(dbscan_hamming_fast(Y, eps, ms), ko.dbscan_hamming(Y, eps, ms))


def test_fast_dbscan_equals_oracle_on_golden_match_matrices(golden_case):
    """the cropped match matrix of every cluster of every golden video that reaches DBSCAN #2"""
    name, g, labels, tracks, vis = golden_case
    res = ko.discover(labels, tracks, vis, g["visibility_threshold"], g["matching_threshold"])
    md = res["queries"]
    if not md:
        pytest.skip("no DBSCAN #2 in this video")
    max_id = max([x for m in md for x in m["matches"]], default=-1)
    n = 0
    for cid in sorted(set(m["cluster_id"] for m in md)):
        mat = np.zeros((max_id + 1, max_id + 1), bool)
        for m in md:
            if m["cluster_id"] == cid and m["overall_mask_id"] <= max_id:
                mat[m["overall_mask_id"], m["matches"]] = True
        cm, _ = ko.crop_bbox(mat)
        if cm.size == 0:
            continue
        eps, ms = ko.dbscan2_params(cm.shape[1])
        assert np.array_equal(dbscan_hamming_fast(cm, eps, ms), ko.dbscan_hamming(cm, eps, ms)), (name, cid)
        n += 1
    assert n > 0 or g["status"] != 1                        # every video that ends with status 1 ran DBSCAN #2


def test_fast_dbscan_equals_oracle_at_1500_rows():
    rng = np.random.default_rng(1500)
    d = 400
    base = rng.random((12, d)) < 0.3
    X = base[rng.integers(0, 12, 1500)] ^ (rng.random((1500, d)) < 0.012)
    X[rng.integers(0, 1500, 200)] = False
    assert np.array_equal(dbscan_hamming_fast(X, 0.05, 5), ko.dbscan_hamming(X, 0.05, 5))


@pytest.mark.parametrize("Nm", [2047, 2048, 3600])
def test_planted_tables_discriminate(Nm):
    """the plant the GPU test runs holds what it is meant to hold, in the expected result: clusters of >= 3 groups, border
    rows (some reachable from two groups), noise, zero rows forced to -1, pairs at exactly kmax and kmax + 1, rows with
    exactly min_samples - 1 and min_samples neighbours, skipped rows above the largest matched id, all three (eps,
    min_samples) regimes, status 1"""
    pv = planted_video(Nm, Nm)
    exp = expected_grouping(pv)
    assert exp["status"] == 1
    cen = plant_census(pv, exp)
    for key in ("clusters_ge3_groups", "border", "border_two_groups", "noise", "zero_forced", "kmax_pairs", "kmax1_pairs",
                "ms_rows", "ms1_rows", "skipped"):
        assert cen[key] > 0, (key, cen)
    assert cen["regimes"] == {(0.05, 5), (0.1, 5), (0.1, 3)}
    assert pv["nclusters"] == 16
    # the crops reach past row 2048 of the problem (rows the Gram path serves from the upper part of G)
    if Nm > 2048:
        assert (exp["clinfo"][:, 1] - exp["clinfo"][:, 0] >= 2048).any()
