"""Reference for the annotation layout (s2d_b200/csrc/annotations.cu): the Python assembly Batch.annotations() used
before the layout moved to the device, frozen here as it was, plus the part of Batch.decode() it read, and a generator
of synthetic device tables (rowinfo, glabel, qframe, qlabel, run and winner bits, group sums, stage-E tables) with the
cases real batches rarely reach: ties, more than 10 groups, clusters without candidates, status other than 1."""
from types import SimpleNamespace

import numpy as np

S2D_MAX_LABELS = 256


def setbits(words, limit):
    out = []
    for w, m in enumerate(np.asarray(words).tolist()):
        m &= 0xFFFFFFFF
        while m:
            b = (m & -m).bit_length() - 1
            m &= m - 1
            if w * 32 + b < limit:
                out.append(w * 32 + b)
    return out


def decode_subset(t):
    """What Batch.decode() gave the assembly: status, clusters (candidates, ranges), groupings and one2x."""
    res = []
    for vi, d in enumerate(t.descs):
        T, Nm, TW, r0 = d.T, d.Nm, d.TW, d.row0
        ri = t.rowinfo[r0:r0 + Nm]
        qf, ql, gl = t.qframe[r0:r0 + Nm], t.qlabel[r0:r0 + Nm], t.glabel[r0:r0 + Nm]
        lab1 = ri[:, 0]
        bits = lambda a: a[d.xbits_off:d.xbits_off + Nm * TW].reshape(Nm, TW)
        rs, re, wb = bits(t.rsbits), bits(t.rebits), bits(t.winbits)
        k = int(t.vidinfo[vi, 0])
        clusters = []
        for c in range(k):
            starts, ends = setbits(rs[c], T), setbits(re[c], T)
            rows = np.nonzero(lab1 == c)[0]
            all_cands = []
            for r, (s, e) in enumerate(zip(starts, ends)):
                cands = []
                for g in rows:
                    if (int(wb[g, r >> 5]) >> (r & 31)) & 1 and ri[g, 1] == r:
                        cands.append({"start_frame": s, "end_frame": e, "frame_id": int(qf[g]), "mask_id": int(ql[g])})
                all_cands.append({"range": [s, e], "candidates": cands})
            clusters.append({"cluster_id": c, "ranges": [[s, e] for s, e in zip(starts, ends)], "all_candidates": all_cands})
        r = {"status": int(t.vidinfo[vi, 3]), "clusters": clusters}
        if r["status"] == 1:
            groupings, one2x = [], {}
            for c in range(k):
                groups = {}
                for g in np.nonzero(ri[:, 0] == c)[0]:
                    if gl[g] >= 0:
                        groups.setdefault(int(gl[g]), []).append((int(qf[g]), int(ql[g])))
                groupings.append({"cluster_id": c, "overall_mask_ids_per_label": groups})
                od = {}
                base = 16 * r0 + c * Nm
                for lab in groups:
                    n_, s_ = int(t.grp_n[base + lab]), int(t.grp_one2x[base + lab])
                    avg = s_ / n_ if n_ else 0
                    od[f"group_{lab}"] = {"avg_one2x": avg, "one2x_counts": n_, "noisy": bool(avg > 0.5)}
                one2x[f"cluster_{c}"] = od
            r["groupings"], r["one2x"] = groupings, one2x
        res.append(r)
    return res


def frozen_annotations(res, tab, area, gid_of, descs):
    """Batch.annotations() before the device layout: decode()'s structures + rle_tables() -> annotation lists."""
    soff, chars, bbox = tab["str_off"], tab["chars"], tab["bbox"]
    out = []
    for vi, r in enumerate(res):
        if r["status"] != 1:
            out.append(None)
            continue
        d = descs[vi]
        T, H, W, f0, r0 = d.T, d.H, d.W, d.frame0, d.row0
        with_cands = [c for c, cl in enumerate(r["clusters"]) if any(x["candidates"] for x in cl["all_candidates"])]
        groups_of = {gr["cluster_id"]: gr["overall_mask_ids_per_label"] for gr in r["groupings"]}
        anns = []
        for c in sorted(with_cands, key=lambda c: f"cluster_{c}"):
            cname = f"cluster_{c}"
            if cname not in r["one2x"]:
                continue
            groups = groups_of.get(c, {})
            for lab in sorted(groups, key=lambda l: f"group_{l}"):
                segs, boxes, areas = [None] * T, [None] * T, [None] * T
                for f, m in sorted(groups[lab], key=lambda fm: fm[1]):      # tie rule: the largest label id wins
                    g = r0 + int(gid_of[f0 + f, m])
                    segs[f] = {"size": [H, W], "counts": chars[soff[g]:soff[g + 1]]}
                    x0, y0, x1, y1 = (int(v) for v in bbox[g])
                    boxes[f] = [float(x0), float(y0), float(x1 - x0 + 1), float(y1 - y0 + 1)]
                    areas[f] = int(area[f0 + f, m])
                anns.append({"video_id": 1, "iscrowd": 0, "height": H, "width": W, "length": T,
                             "segmentations": segs, "bboxes": boxes, "areas": areas, "category_id": 1,
                             "id": len(anns) + 1, "one2x": round(float(r["one2x"][cname][f"group_{lab}"]["avg_one2x"]), 2),
                             "visibility_ranges": [list(x) for x in r["clusters"][c]["ranges"]]})
        out.append(anns)
    return out


def _runs(rng, T):
    """start / end bits of a random majority pattern over T frames (packed like rsbits / rebits)"""
    maj = rng.random(T) < rng.uniform(0.2, 0.9)
    prev = np.concatenate(([False], maj[:-1]))
    nxt = np.concatenate((maj[1:], [False]))
    return maj & ~prev, maj & ~nxt


def _pack(flags):
    n = (len(flags) + 31) // 32
    w = np.zeros(n, np.uint32)
    for i in np.nonzero(flags)[0]:
        w[i >> 5] |= np.uint32(1 << (i & 31))
    return w.view(np.int32)


def synthetic_batch(seed, nvideos=5):
    """Device-shaped tables of a batch whose videos have random rows, clusters, runs, winners, candidates and groups."""
    rng = np.random.default_rng(seed)
    descs, rows = [], []
    xw = row0 = frame0 = 0
    vidinfo = np.zeros((nvideos, 8), np.int32)
    gid_of_l, area_l, rs_l, re_l, wb_l = [], [], [], [], []
    for vi in range(nvideos):
        T = int(rng.integers(1, 70))
        H, W = int(rng.integers(1, 50)), int(rng.integers(1, 50))
        gid = np.full((T, S2D_MAX_LABELS), -1, np.int32)
        qf, ql = [], []
        for f in range(T):
            labs = np.sort(rng.choice(np.arange(1, 256), size=int(rng.integers(0, 9)), replace=False))
            for l in labs:
                gid[f, l] = len(qf)
                qf.append(f)
                ql.append(int(l))
        if not qf:
            gid[0, 1] = 0
            qf, ql = [0], [1]
        Nm, TW = len(qf), (T + 31) // 32
        k = int(min(Nm, rng.integers(1, 14)))
        rs, re, wb = np.zeros((Nm, TW), np.int32), np.zeros((Nm, TW), np.int32), np.zeros((Nm, TW), np.int32)
        nruns = []
        for c in range(k):
            s, e = _runs(rng, T)
            rs[c], re[c] = _pack(s), _pack(e)
            nruns.append(int(s.sum()))
        nocand = set(rng.choice(k, size=int(rng.integers(0, k)), replace=False).tolist()) if k > 1 else set()
        ngroups = int(rng.integers(1, 16))                       # more than 10 groups in some clusters
        ri = np.full((Nm, 4), -1, np.int32)
        gl = np.full(Nm, -1, np.int32)
        for g in range(Nm):
            c = int(rng.integers(-1, k))
            ri[g, 0] = c
            if c < 0:
                continue
            if nruns[c]:
                w = _pack(rng.random(nruns[c]) < 0.5)
                wb[g, :len(w)] = w
                r = int(rng.integers(0, nruns[c] + 1))           # r == nruns: no such run
                if c not in nocand and rng.random() < 0.6:
                    ri[g, 1] = r
            ri[g, 2:] = sorted(rng.integers(0, T, size=2))
            gl[g] = min(Nm - 1, int(rng.integers(-1, ngroups))) if rng.random() < 0.9 else int(rng.integers(0, Nm))
        vidinfo[vi, 0] = k
        vidinfo[vi, 3] = 1 if rng.random() < 0.75 else -1
        d = SimpleNamespace(T=T, H=H, W=W, Nm=Nm, TW=TW, row0=row0, frame0=frame0, xbits_off=xw)
        descs.append(d)
        rows.append((ri, gl, np.asarray(qf, np.int32), np.asarray(ql, np.int32)))
        gid_of_l.append(gid)
        area_l.append(rng.integers(1, 10 ** 6, size=(T, S2D_MAX_LABELS)).astype(np.int32))
        rs_l.append(rs.reshape(-1)); re_l.append(re.reshape(-1)); wb_l.append(wb.reshape(-1))
        xw += Nm * TW
        row0 += Nm
        frame0 += T
    R = row0
    lens = rng.integers(0, 40, size=R)
    str_off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    chars = "".join(chr(48 + int(x)) for x in rng.integers(0, 64, size=int(str_off[-1])))
    x0, y0 = rng.integers(0, 50, size=R), rng.integers(0, 50, size=R)
    bbox = np.stack([x0, y0, x0 + rng.integers(0, 9, size=R), y0 + rng.integers(0, 9, size=R)], 1).astype(np.int32)
    return SimpleNamespace(
        descs=descs, vidinfo=vidinfo,
        rowinfo=np.concatenate([r[0] for r in rows]), glabel=np.concatenate([r[1] for r in rows]),
        qframe=np.concatenate([r[2] for r in rows]), qlabel=np.concatenate([r[3] for r in rows]),
        rsbits=np.concatenate(rs_l), rebits=np.concatenate(re_l), winbits=np.concatenate(wb_l),
        grp_n=rng.integers(0, 6, size=16 * R).astype(np.int32), grp_one2x=rng.integers(0, 6, size=16 * R).astype(np.int32),
        gid_of=np.concatenate(gid_of_l), area=np.concatenate(area_l), bbox=bbox, str_off=str_off, chars=chars,
        total_rows=R, total_frames=frame0)


def reference(t):
    """The frozen assembly applied to a synthetic batch."""
    tab = {"str_off": t.str_off, "chars": t.chars, "bbox": t.bbox}
    return frozen_annotations(decode_subset(t), tab, t.area, t.gid_of, t.descs)
