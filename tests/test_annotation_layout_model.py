"""Host model of the annotation layout (s2d_b200/csrc/annotations.cu), checked against the frozen Python assembly of
Batch.annotations() (tests/annotation_reference.py) on synthetic batches. Runs without a GPU.

The kernels give every grouped row of a candidate cluster one key - cluster rank | decimal-string key of the group
label | frame | label - and sort them per video; a change of (cluster, group) starts an annotation, the last key of a
frame is its member. The host (annotations_from_layout, tested here as it is) only slices the tables."""
import numpy as np
import pytest

from s2d_b200.pipeline import LAYOUT_TABLES, annotations_from_layout
from tests.annotation_reference import decode_subset, reference, setbits, synthetic_batch


def decimal_key(x: int) -> int:
    """al_decimal_key: the digits zero-padded on the right to 10, ties broken by length"""
    d = len(str(x))
    return x * 10 ** (10 - d) * 16 + d


def test_decimal_key_sorts_like_the_strings():
    cl = list(range(16))
    assert sorted(cl, key=decimal_key) == sorted(cl, key=lambda c: f"cluster_{c}")
    gr = list(range(9001))
    assert sorted(gr, key=decimal_key) == sorted(gr, key=lambda l: f"group_{l}")
    assert decimal_key(2 ** 31 - 1) < 2 ** 38 and len({decimal_key(x) for x in gr}) == len(gr)
    rng = np.random.default_rng(5)
    big = rng.integers(0, 2 ** 31, size=5000).tolist() + [0, 1, 10, 100, 10 ** 9, 2 ** 31 - 1]
    assert sorted(big, key=decimal_key) == sorted(big, key=str)


def model_layout(t):
    """What al_sort_kernel, al_scan_kernel and al_write_kernel write, computed the same way on the host."""
    counts, per_video = [], []
    for vi, d in enumerate(t.descs):
        T, Nm, TW, r0, f0 = d.T, d.Nm, d.TW, d.row0, d.frame0
        if t.vidinfo[vi, 3] != 1:
            counts.append((0, 0, 0, 0, 0))
            per_video.append(None)
            continue
        kc = max(0, min(int(t.vidinfo[vi, 0]), 16, Nm))
        row = lambda a, c: a[d.xbits_off + c * TW:d.xbits_off + (c + 1) * TW]
        nruns = [min(len(setbits(row(t.rsbits, c), T)), len(setbits(row(t.rebits, c), T))) for c in range(kc)]
        cand = [False] * kc
        for q in range(Nm):
            c, r = (int(x) for x in t.rowinfo[r0 + q, :2])
            if 0 <= c < kc and 0 <= r < nruns[c] and (int(row(t.winbits, q)[r >> 5]) >> (r & 31)) & 1:
                cand[c] = True
        ranked = sorted((c for c in range(kc) if cand[c]), key=decimal_key)
        rank = {c: i for i, c in enumerate(ranked)}
        keys = []
        for q in range(Nm):
            c, l = int(t.rowinfo[r0 + q, 0]), int(t.glabel[r0 + q])
            if 0 <= c < kc and cand[c] and l >= 0:
                keys.append(rank[c] << 56 | decimal_key(l) << 18 | int(t.qframe[r0 + q]) << 8 | int(t.qlabel[r0 + q]))
        keys.sort()
        anns, mems = [], []                    # (rank, row) of each annotation start; row of each member
        for j, k in enumerate(keys):
            f, m = (k >> 8) & 1023, k & 255
            g = int(t.gid_of[f0 + f, m])
            if j == 0 or keys[j - 1] >> 18 != k >> 18:
                anns.append((k >> 56, g, len(mems)))
            if j == len(keys) - 1 or keys[j + 1] >> 8 != k >> 8:
                mems.append((f, m, g))
        annotated = sorted({a[0] for a in anns})
        nchars = sum(int(t.str_off[r0 + g + 1] - t.str_off[r0 + g]) for _, _, g in mems)
        counts.append((len(anns), len(mems), nchars, len(annotated), sum(nruns[ranked[r]] for r in annotated)))
        per_video.append((ranked, nruns, anns, mems, annotated))
    first = np.cumsum([(0,) * 5] + counts, axis=0)[:-1]
    tabs = {"vann": [], "ann": [], "members": [], "member_off": [], "chars": [], "clusters": [], "pairs": []}
    for vi, d in enumerate(t.descs):
        tabs["vann"] += [counts[vi][0], int(first[vi][0])]
        if per_video[vi] is None:
            continue
        ranked, nruns, anns, mems, annotated = per_video[vi]
        T, Nm, r0, f0 = d.T, d.Nm, d.row0, d.frame0
        M0, C0, K0, P0 = (int(x) for x in first[vi][1:])
        assert (len(tabs["members"]) // 6, len(tabs["chars"]), len(tabs["pairs"]) // 2) == (M0, C0, P0)
        cl_index = {}
        for i, r in enumerate(annotated):
            c = ranked[r]
            cl_index[r] = K0 + i
            assert len(tabs["clusters"]) // 2 == K0 + i
            tabs["clusters"] += [len(tabs["pairs"]) // 2, nruns[c]]
            row = lambda a: a[d.xbits_off + c * d.TW:d.xbits_off + (c + 1) * d.TW]
            for s, e in list(zip(setbits(row(t.rsbits), T), setbits(row(t.rebits), T)))[:nruns[c]]:
                tabs["pairs"] += [s, e]
        for a, (r, g, m0) in enumerate(anns):
            c, l = ranked[r], int(t.glabel[r0 + g])
            m1 = anns[a + 1][2] if a + 1 < len(anns) else len(mems)
            slot = 16 * r0 + c * Nm + l
            tabs["ann"] += [c, l, int(t.grp_n[slot]), int(t.grp_one2x[slot]), cl_index[r], M0 + m0, m1 - m0]
        for f, m, g in mems:
            x0, y0, x1, y1 = (int(v) for v in t.bbox[r0 + g])
            tabs["members"] += [f, x0, y0, x1, y1, int(t.area[f0 + f, m])]
            tabs["member_off"].append(len(tabs["chars"]))
            tabs["chars"] += list(t.chars[t.str_off[r0 + g]:t.str_off[r0 + g + 1]].encode())
    sizes = [len(tabs[k]) // LAYOUT_TABLES[k][0] for k in ("ann", "members", "chars", "clusters", "pairs")]
    assert sizes == [int(x) for x in np.sum(counts, axis=0)]
    out = {k: np.asarray(v, np.uint8 if k == "chars" else np.int64 if k == "member_off" else np.int32)
           for k, v in tabs.items()}
    return out


@pytest.mark.parametrize("seed", range(12))
def test_model_layout_equals_frozen_assembly(seed):
    t = synthetic_batch(seed, nvideos=6)
    want = reference(t)
    got = annotations_from_layout(t.descs, t.vidinfo[:, 3], model_layout(t))
    assert got == want


def test_synthetic_batches_cover_the_rules():
    """ties, > 10 groups in a cluster, clusters without candidates and status other than 1 all occur"""
    seen = dict(tie=False, many_groups=False, no_cand=False, failed=False)
    for seed in range(12):
        t = synthetic_batch(seed, nvideos=6)
        ref = reference(t)
        seen["failed"] |= any(a is None for a in ref)
        for vi, d in enumerate(t.descs):
            if ref[vi] is None:
                continue
            r0, Nm = d.row0, d.Nm
            ri, gl, qf = t.rowinfo[r0:r0 + Nm], t.glabel[r0:r0 + Nm], t.qframe[r0:r0 + Nm]
            for c in range(int(t.vidinfo[vi, 0])):
                sel = (ri[:, 0] == c) & (gl >= 0)
                seen["many_groups"] |= len(set(gl[sel].tolist())) > 10
                pairs = list(zip(gl[sel].tolist(), qf[sel].tolist()))
                seen["tie"] |= len(pairs) != len(set(pairs))
        for r in decode_subset(t):
            seen["no_cand"] |= r["status"] == 1 and any(not any(x["candidates"] for x in cl["all_candidates"])
                                                       for cl in r["clusters"])
    assert all(seen.values()), seen
