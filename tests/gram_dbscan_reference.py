"""Helpers of the DBSCAN #2 tests at the row counts of long videos (tests/test_gram_dbscan_model.py on the CPU,
tests/test_gram_dbscan_gpu.py on the device).

`dbscan_hamming_fast` is the oracle's DBSCAN (oracle/keymask_oracle.py: dbscan_hamming, pinned to sklearn) with the
pairwise distances taken from a float32 BLAS Gram matrix. That is exact: the operands are 0/1 and every sum stays below
2^24. The oracle's own int32 matmul does not use BLAS and needs minutes at 9 000 rows.

`planted_video` writes the match tables stage D's grouping reads (rowinfo, mbits, one2x and the vidinfo words) with a
known structure: hubs with spokes at exactly kmax, rows with exactly min_samples - 1 and min_samples neighbours, border
rows between two groups, noise, all-zero rows, rows above the largest matched id, non-candidate rows and clusters
interleaved in row order. Scenes of moving objects give one group per cluster at these sizes, so only a planted table can
tell a right DBSCAN #2 from a wrong one.
"""
from __future__ import annotations

import numpy as np
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

from oracle import keymask_oracle as ko


def hamming_gram(X: np.ndarray) -> np.ndarray:
    """Pairwise Hamming distances of the 0/1 rows of X as int64, from one float32 Gram matrix."""
    Xf = (np.asarray(X) != 0).astype(np.float32)
    G = Xf @ Xf.T
    pop = Xf.sum(axis=1, dtype=np.float32)
    return (pop[:, None] + pop[None, :] - 2 * G).astype(np.int64)


def dbscan_hamming_fast(X: np.ndarray, eps: float, min_samples: int) -> np.ndarray:
    """sklearn's DBSCAN(metric="hamming") labels as ko.dbscan_hamming states them: neighbours <=> distance <= kmax (the row
    itself included), core <=> at least min_samples neighbours, clusters = connected components of the core-core graph
    numbered by their lowest core index, border rows take the smallest label among their core neighbours, the rest is -1.

    Identical rows have the same neighbours, so the graph is built on the distinct rows, each weighted by its copies (a
    cropped match matrix is mostly all-zero rows of other clusters)."""
    X = np.asarray(X) != 0
    n, d = X.shape
    if n == 0:
        return np.zeros(0, np.int64)
    U, inv, cnt = np.unique(X, axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    first_row = np.full(len(U), n, np.int64)
    np.minimum.at(first_row, inv, np.arange(n))
    nb = hamming_gram(U) <= ko.hamming_kmax(d, eps)
    core = nb.astype(np.int64) @ cnt >= min_samples
    lab = np.full(len(U), -1, np.int64)
    ci = np.nonzero(core)[0]
    if len(ci):
        ncomp, comp = connected_components(csr_matrix(nb[np.ix_(ci, ci)]), directed=False)
        first = np.full(ncomp, n, np.int64)
        np.minimum.at(first, comp, first_row[ci])
        rank = np.empty(ncomp, np.int64)
        rank[np.argsort(first)] = np.arange(ncomp)
        lab[ci] = rank[comp]
        big = np.iinfo(np.int64).max
        border = np.nonzero(~core)[0]
        if len(border):
            m = np.where(nb[np.ix_(border, ci)], lab[ci][None, :], big).min(axis=1)
            lab[border] = np.where(m == big, -1, m)
    return lab[inv]


# ----------------------------------------------------------------------------- planted match tables
def _eps_ms(span):
    return ko.dbscan2_params(span)


class _Cluster:
    """Rows of one visibility cluster as bit patterns over its column span [a, a + S): every pattern sets both end
    columns, so the cropped matrix has exactly S columns, and flips only touch the interior."""

    def __init__(self, rng, a, S):
        self.rng, self.a, self.S = rng, a, S
        eps, self.ms = _eps_ms(S)
        self.k = ko.hamming_kmax(S, eps)
        self.rows = []                       # (bits over the span [S] bool, kind)

    def hub(self):
        h = self.rng.random(self.S) < 0.4
        h[0] = h[-1] = True
        return h

    def flip(self, h, cols):
        x = h.copy()
        x[np.asarray(cols, np.int64)] ^= True
        return x

    def interior(self, n, avoid=()):
        pool = np.setdiff1d(np.arange(1, self.S - 1), np.asarray(avoid, np.int64))
        return self.rng.permutation(pool)[:n] if n <= len(pool) else None

    def star(self, nspokes, kind):
        """a hub with `nspokes` spokes at distance exactly k on disjoint columns (spokes 2k apart): the hub has
        nspokes + 1 neighbours; one more row at k + 1 from the hub that is nobody's neighbour"""
        h = self.hub()
        k = self.k
        cols = self.interior(max(k, 1) * (nspokes + 1) + 1)
        if cols is None or k == 0:
            for _ in range(nspokes + 1):     # kmax 0: neighbours are copies
                self.rows.append((h.copy(), kind))
            return h
        self.rows.append((h, kind))
        for i in range(nspokes):
            self.rows.append((self.flip(h, cols[i * k:(i + 1) * k]), kind + "_spoke"))
        self.rows.append((self.flip(h, cols[nspokes * k:nspokes * k + k + 1]), "far"))
        return h

    def bridge(self):
        """two cores whose hubs are 2k apart and a row k from both hubs: a border row reachable from two groups"""
        k = self.k
        if k == 0:
            return
        hA = self.hub()
        D = self.interior(2 * k)
        if D is None:
            return
        hB = self.flip(hA, D)
        for h in (hA, hB):
            cols = self.interior(k * (self.ms - 1), avoid=D)
            if cols is None:
                return
            self.rows.append((h, "core"))
            for i in range(self.ms - 1):
                self.rows.append((self.flip(h, cols[i * k:(i + 1) * k]), "core_spoke"))
        self.rows.append((self.flip(hA, D[:k]), "bridge"))

    def copies(self, n):
        h = self.hub()
        for _ in range(n):
            self.rows.append((h.copy(), "copy"))


def planted_video(seed: int, Nm: int, nclusters: int = 16, spans=None):
    """Match tables of one video with Nm rows: dict with rowinfo [Nm, 4], mbits [Nm, NW] (uint32), one2x [Nm], nclusters,
    maxid (largest matched id of a candidate row) and the planted rows' kinds. Rows are interleaved across clusters, the
    last rows are candidates above the largest matched id, non-candidate rows carry garbage match bits (the grouping
    must ignore them), some rows belong to no cluster."""
    rng = np.random.default_rng(seed)
    NW = (Nm + 31) // 32
    top = Nm - 40                                             # matched ids stay below this: later rows are skipped
    if spans is None:
        spans = [6, 9, 10, 30, 50, 51, 300, 1200, 2000, 40, 120, 8, 25, 700, 64, 11]
    spans = [min(s, top) for s in spans[:nclusters]]
    K = len(spans)
    # row slots: ~6 % no cluster, ~6 % non-candidate rows, the rest are candidates of a cluster chosen per row
    cl = rng.integers(0, K, size=Nm)
    cl[rng.random(Nm) < 0.06] = -1
    cand = (cl >= 0) & (rng.random(Nm) >= 0.06)
    bits = np.zeros((Nm, Nm), bool)
    kinds = np.array([""] * Nm, dtype=object)
    for c in range(K):
        S = spans[c]
        a = int(rng.integers(0, top - S + 1))
        C = _Cluster(rng, a, S)
        slots = rng.permutation(np.nonzero(cand & (cl == c))[0])
        budget = len(slots)
        while len(C.rows) < budget:
            r = rng.random()
            if r < 0.30:
                C.star(C.ms - 1, "hub_ms")           # hub with exactly ms neighbours: core
            elif r < 0.45:
                C.star(C.ms - 2, "hub_ms1")          # hub with exactly ms - 1 neighbours: noise
            elif r < 0.60:
                C.bridge()
            elif r < 0.75:
                C.copies(int(rng.integers(C.ms, C.ms + 6)))
            elif r < 0.85:
                C.rows.append((np.zeros(S, bool), "zero"))
            else:
                C.rows.append((C.hub(), "noise"))
        for q, (x, kind) in zip(slots, C.rows[:budget]):
            bits[q, a:a + S] = x
            kinds[q] = kind
    # non-candidate rows of a cluster hold stray bits the grouping must not read
    junk = (cl >= 0) & ~cand
    bits[junk] = rng.random((int(junk.sum()), Nm)) < 0.02
    kinds[junk] = "noncand"
    kinds[cl < 0] = "nocluster"
    maxid = int(np.nonzero(bits[cand].any(axis=0))[0].max())
    rowinfo = np.stack([cl, np.where(cand, 0, -1), np.zeros(Nm), np.zeros(Nm)], axis=1).astype(np.int32)
    pad = np.zeros((Nm, NW * 32), bool)
    pad[:, :Nm] = bits
    mbits = np.packbits(pad.reshape(Nm, NW, 32), axis=-1, bitorder="little").view(np.uint32).reshape(Nm, NW)
    one2x = (rng.random(Nm) < 0.3).astype(np.int32) * cand
    return dict(Nm=Nm, NW=NW, rowinfo=rowinfo, mbits=mbits, bits=bits, one2x=one2x.astype(np.int32), nclusters=K,
                maxid=maxid, kinds=kinds)


def expected_grouping(pv):
    """What stage D's grouping must produce for a planted video, through ko.temporal_clustering with the fast DBSCAN:
    glabel per row, per cluster the groups, clusterinfo[5:15] and the per-group (count, one2x sum), and the status."""
    Nm, ri, bits, one2x = pv["Nm"], pv["rowinfo"], pv["bits"], pv["one2x"]
    cand = np.nonzero((ri[:, 1] >= 0) & (ri[:, 0] >= 0))[0]
    matches_data = [{"cluster_id": int(ri[q, 0]), "overall_mask_id": int(q), "matches": np.nonzero(bits[q])[0].tolist()}
                    for q in cand]
    saved = ko.dbscan_hamming
    ko.dbscan_hamming = dbscan_hamming_fast
    try:
        cids, groupings = ko.temporal_clustering(matches_data, np.arange(Nm), np.zeros(Nm, np.int64))
    finally:
        ko.dbscan_hamming = saved
    K = pv["nclusters"]
    out = dict(glabel=np.full(Nm, -1, np.int64), status=-1, clinfo=np.zeros((K, 10), np.int64), groups={}, grp={})
    if cids == -1:
        return out
    assert cids == list(range(K))
    out["status"] = 1
    maxid = max(g for m in matches_data for g in m["matches"])
    assert maxid == pv["maxid"]
    for c, g in zip(cids, groupings):
        mine = cand[ri[cand, 0] == c]
        rows = mine[(mine <= maxid) & bits[mine].any(axis=1)]          # the nonzero rows of the cluster's match matrix
        cols = np.nonzero(bits[rows].any(axis=0))[0]
        ro, co = int(rows.min()), int(cols.min())
        cm = np.empty((int(rows.max()) - ro + 1, int(cols.max()) - co + 1))   # crop_bbox's shape
        eps, ms = ko.dbscan2_params(cm.shape[1])
        lab = g["overall_mask_ids_per_label"]
        for l, fms in lab.items():
            qs = [f for f, _ in fms]
            out["glabel"][qs] = l
            out["grp"][(c, l)] = (len(qs), int(one2x[qs].sum()))
        out["groups"][c] = g["visibility_to_temporal_factor"]
        matched = sum(len(v) for v in lab.values())
        out["clinfo"][c] = [ro, ro + cm.shape[0] - 1, co, co + cm.shape[1] - 1, ko.hamming_kmax(cm.shape[1], eps), ms,
                            len(lab), matched, int(one2x[mine].sum()), len(mine)]
    return out


def plant_census(pv, exp):
    """How much of the plant the expected result actually exercises: per property the number of rows / pairs / clusters
    (the tests assert each is nonzero)."""
    ri, bits = pv["rowinfo"], pv["bits"]
    maxid = pv["maxid"]
    cen = dict(clusters_ge3_groups=0, border=0, border_two_groups=0, noise=0, zero_forced=0, kmax_pairs=0,
               kmax1_pairs=0, ms_rows=0, ms1_rows=0, skipped=0, regimes=set())
    cand = (ri[:, 1] >= 0) & (ri[:, 0] >= 0)
    cen["skipped"] = int((cand & (np.arange(pv["Nm"]) > maxid) & bits.any(axis=1)).sum())
    for c in range(pv["nclusters"]):
        if exp["groups"].get(c, 0) >= 3:
            cen["clusters_ge3_groups"] += 1
        rmin, rmax, cmin, cmax, kmax, ms = exp["clinfo"][c][:6]
        cen["regimes"].add(ko.dbscan2_params(int(cmax - cmin + 1)))
        rows = np.arange(rmin, rmax + 1)
        valid = cand[rows] & (ri[rows, 0] == c) & (rows <= maxid)
        nz = valid & bits[rows, cmin:cmax + 1].any(axis=1)
        cen["zero_forced"] += int((valid & ~nz).sum())
        vv = rows[nz]                                   # the crop's nonzero rows; every other row of it is all-zero
        X = bits[vv, cmin:cmax + 1]
        D = hamming_gram(X)
        nb = D <= kmax
        nzero = len(rows) - len(vv)
        cnt = nb.sum(axis=1) + nzero * (X.sum(axis=1) <= kmax)
        core = cnt >= ms
        lab = exp["glabel"][vv]
        cen["ms_rows"] += int((cnt == ms).sum())
        cen["ms1_rows"] += int((cnt == ms - 1).sum())
        cen["border"] += int((~core & (lab >= 0)).sum())
        cen["noise"] += int((lab < 0).sum())
        cen["kmax_pairs"] += int((np.triu(D == kmax, 1)).sum())
        cen["kmax1_pairs"] += int((np.triu(D == kmax + 1, 1)).sum())
        # border rows with core neighbours in two different groups
        labs_core = np.where(core, lab, -1)
        for i in np.nonzero(~core & (lab >= 0))[0]:
            if len(set(labs_core[nb[i] & core].tolist()) - {-1}) >= 2:
                cen["border_two_groups"] += 1
    return cen
