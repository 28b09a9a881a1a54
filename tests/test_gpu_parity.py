"""CUDA path vs reference goldens and vs the CPU oracle, through the C ABI (needs a B200)."""
import os

import numpy as np
import pytest
import torch

from oracle import keymask_oracle as ko
from oracle.compare import check_against_golden

pytestmark = pytest.mark.gpu


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _video(labels, tracks, vis, **kw):
    from s2d_b200.pipeline import VideoInput
    d = _dev()
    return VideoInput(torch.from_numpy(np.ascontiguousarray(labels)).to(d),
                      torch.from_numpy(np.ascontiguousarray(tracks)).to(d),
                      torch.from_numpy(np.ascontiguousarray(vis)).to(d), **kw)


def test_pipeline_matches_reference_golden(golden_case):
    from s2d_b200.pipeline import Params, discover_keymasks
    name, g, labels, tracks, vis = golden_case
    res = discover_keymasks([_video(labels, tracks, vis)],
                            Params(g["visibility_threshold"], g["matching_threshold"]))[0]
    check_against_golden(res, g)


def test_gram_dbscan_path_matches_reference_golden(golden_case):
    """DBSCAN #2 with the pairwise distances taken from the int8 Gram contraction of the match rows (the path videos with
    >= 2048 rows take: s2d_unpack_bits + s2d_overlap_i8 + s2d_group_gram), forced on for every golden video: same groups,
    coverages and one2x sums as the reference."""
    from s2d_b200.pipeline import Batch, Params
    name, g, labels, tracks, vis = golden_case
    b = Batch([_video(labels, tracks, vis)], gram_min_rows=1)
    assert b.gram is not None
    b.run(Params(g["visibility_threshold"], g["matching_threshold"]))
    torch.cuda.synchronize()
    check_against_golden(b.decode()[0], g)


def test_unpack_bits_is_the_inverse_of_pack_bits():
    from s2d_b200 import _lib
    rng = np.random.default_rng(9)
    d = _dev()
    for N, D in ((5, 33), (40, 128), (7, 300), (64, 1000)):
        stride = (D + 31) // 32
        ncols = stride * 32
        X = (rng.random((N, D)) < 0.3)
        Xp = np.zeros((N, ncols), np.uint8)
        Xp[:, :D] = X
        words = np.packbits(Xp, axis=1, bitorder="little").view(np.uint32).reshape(N, stride)
        bits = torch.from_numpy(words.view(np.int32).copy()).to(d)
        planes = torch.full((N, ncols), 7, dtype=torch.uint8, device=d)
        _lib.call("s2d_unpack_bits", bits.data_ptr(), N, stride, ncols, planes.data_ptr(), torch.cuda.current_stream(d).cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(planes.cpu().numpy(), Xp)


def test_batched_heterogeneous_videos_match_goldens():
    """all golden cases in ONE batch (different T/H/W/P/Nm per video)."""
    from tests.conftest import GOLDEN_CASES, load_golden
    from s2d_b200.pipeline import Params, discover_keymasks
    cases = [load_golden(n) for n in GOLDEN_CASES]
    groups = {}
    for n, c in zip(GOLDEN_CASES, cases):
        groups.setdefault((c[0]["visibility_threshold"], c[0]["matching_threshold"]), []).append((n, c))
    for (vt, mt), items in groups.items():
        res = discover_keymasks([_video(c[1], c[2], c[3]) for _, c in items], Params(vt, mt))
        for (n, c), r in zip(items, res):
            check_against_golden(r, c[0])


def test_point_votes_all_pairs_vs_oracle(golden_case):
    from s2d_b200.pipeline import Batch
    name, g, labels, tracks, vis = golden_case
    b = Batch([_video(labels, tracks, vis)])
    b.hits.fill_(-7); b.uniq.fill_(-7)
    b.votes_all()
    torch.cuda.synchronize()
    Nm, T, P, _ = tracks.shape
    L = b.host_descs[0].L
    hits = b.hits.cpu().numpy().reshape(Nm, T, L)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        h, u = ko.point_votes(tracks[q], labels, 0, T - 1, nbins=L)
        assert np.array_equal(u, uniq[q]), (name, q)
        assert np.array_equal(h, hits[q]), (name, q)


@pytest.fixture(params=[0, 1, 2, 3, 4], ids=["product", "bitmap", "cta_per_tile", "table_any_P", "warp_any_frame"])
def pv_variant(request, monkeypatch):
    """run a test once per point-votes kernel variant (include/s2d_b200.h: s2d_point_votes_variant); the superseded
    bitmap kernel (1) only exists in the experiments build (make exp), which the runs of variant 1 load instead - also in a
    debug run with S2D_B200_LIB pointing at the bounds-checked library, so those runs are not bounds-checked"""
    from s2d_b200 import _lib
    if request.param == 1:
        monkeypatch.setattr(_lib, "LIB_PATH", os.path.join(os.path.dirname(_lib.LIB_PATH), "libs2d_b200_exp.so"))
        monkeypatch.setattr(_lib, "_lib", None)
    _lib.call("s2d_point_votes_variant", request.param)
    yield request.param
    _lib.call("s2d_point_votes_variant", 0)


@pytest.mark.parametrize("P,H,W", [(1000, 480, 854), (4096, 720, 1280), (777, 33, 1900), (8192, 1080, 1920), (20000, 64, 64),
                                   (16384, 480, 854), (12002, 300, 500), (2048, 96, 1280)])
def test_point_votes_shapes_and_bands(P, H, W, pv_variant):
    """odd P (no 128-bit path), P above the register tile, bounding boxes that need several
    bitmap bands (points spread over the whole 1080p frame), heavy duplication (P >> H*W)."""
    from s2d_b200.pipeline import Batch
    rng = np.random.default_rng(P + H)
    T, Nm = 3, 4
    labels = rng.integers(0, 7, size=(T, H, W)).astype(np.uint8)
    labels[:, : H // 2] = 3
    tracks = np.empty((Nm, T, P, 2), np.float32)
    tracks[..., 0] = rng.uniform(-20, W + 20, size=(Nm, T, P))
    tracks[..., 1] = rng.uniform(-20, H + 20, size=(Nm, T, P))
    tracks[0, 0, : P // 2] = tracks[0, 0, P // 2: P // 2 + P // 2][: P // 2]   # duplicates
    tracks[1, 1, ::5, 0] = np.nan
    tracks[2, 2, ::7, 1] = np.inf
    tracks[3, :, :, :] = np.round(tracks[3]) + 0.5                            # all half-integers
    vis = rng.integers(0, 2, size=(Nm, T, P)).astype(np.uint8)
    b = Batch([_video(labels, tracks, vis, max_label=6)])
    b.votes_all()
    torch.cuda.synchronize()
    hits = b.hits.cpu().numpy().reshape(Nm, T, 7)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        h, u = ko.point_votes(tracks[q], labels, 0, T - 1, nbins=7)
        assert np.array_equal(u, uniq[q]) and np.array_equal(h, hits[q]), (q, u, uniq[q])
    # stage A on the same batch: visibility mean is float32(cnt)/float32(P)
    from s2d_b200 import _lib
    _lib.call("s2d_vis_reduce", b.descs.data_ptr(), 1, b.max_rows_x_T, b.cnt.data_ptr(), b.V.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(b.V.cpu().numpy().reshape(Nm, T), ko.visibility_mean(vis))


@pytest.mark.parametrize("H,W,P,M,lab255,off", [(480, 854, 1000, 10, False, 5), (720, 1280, 4096, 20, False, 5),
                                                (720, 1280, 4096, 20, False, 0), (1080, 1920, 2048, 6, False, 16),
                                                (480, 864, 1024, 12, False, 0), (97, 131, 512, 5, True, 5),
                                                (720, 1280, 16384, 4, False, 0), (480, 854, 12000, 6, False, 5),
                                                (480, 854, 4096, 20, True, 0)])
def test_point_votes_scene_geometry(H, W, P, M, lab255, off, pv_variant):
    """Object-shaped point clouds (compact bounding boxes: the label-table kernel's main path, one
    or several bands), widths that are not a multiple of 16, a label map that does not start on a
    16-byte boundary (off = 5: tables fetched row by row; off = 0 / 16 with W a multiple of 16: tables
    fetched as 2D TMA boxes), and label id 255 in use (the table kernel must take its bitmap fallback)."""
    from s2d_b200.pipeline import Batch, VideoInput
    from s2d_b200.synth import make_scene
    sc = make_scene(31 + H, 5, H, W, M, P, specials=True, dup_rate=0.05)
    labels = sc.labels.copy()
    maxlab = int(labels.max())
    if lab255:
        labels[labels == maxlab] = 255
        maxlab = 255
    d = _dev()
    raw = torch.zeros(labels.size + 64, dtype=torch.uint8, device=d)
    raw[off:off + labels.size] = torch.from_numpy(labels.reshape(-1)).to(d)
    lab_dev = raw[off:off + labels.size].view(labels.shape)
    vid = VideoInput(labels=lab_dev, tracks=torch.from_numpy(sc.tracks).to(d), vis=torch.from_numpy(sc.vis).to(d),
                     max_label=maxlab)
    b = Batch([vid])
    b.hits.fill_(-3); b.uniq.fill_(-3)
    b.votes_all()
    torch.cuda.synchronize()
    Nm, T = sc.tracks.shape[:2]
    L = maxlab + 1
    hits = b.hits.cpu().numpy().reshape(Nm, T, L)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        h, u = ko.point_votes(sc.tracks[q], labels, 0, T - 1, nbins=L)
        assert np.array_equal(u, uniq[q]), (q, u, uniq[q])
        assert np.array_equal(h, hits[q]), q


@pytest.mark.parametrize("H,W,P,nlab,spread", [(1080, 1920, 1024, 256, True), (1080, 1920, 256, 40, True), (480, 854, 1000, 256, False),
                                                (720, 1280, 1024, 21, False), (64, 64, 1024, 7, True), (33, 1900, 2, 5, True)])
def test_point_votes_sparse_tiles_warp_kernel(H, W, P, nlab, spread, pv_variant):
    """Tiles of <= 1024 points (one warp per tile in the product dispatch): boxes of many bitmap bands (points spread over
    a 1080p frame), every label id in use (255 included), heavy duplication (P >> pixels of the box), P = 2, ragged point
    counts; the same inputs through the other variants."""
    from s2d_b200.pipeline import Batch
    rng = np.random.default_rng(H + P + nlab)
    T, Nm = 3, 6
    labels = rng.integers(0, nlab, size=(T, H, W)).astype(np.uint8)
    labels[:, : H // 2, : W // 2] = nlab - 1
    tracks = np.empty((Nm, T, P, 2), np.float32)
    if spread:
        tracks[..., 0] = rng.uniform(-20, W + 20, size=(Nm, T, P))
        tracks[..., 1] = rng.uniform(-20, H + 20, size=(Nm, T, P))
    else:                                           # object-sized clouds around a centre per (query, frame)
        cx = rng.uniform(0.2 * W, 0.8 * W, size=(Nm, T, 1)); cy = rng.uniform(0.2 * H, 0.8 * H, size=(Nm, T, 1))
        tracks[..., 0] = cx + rng.normal(0, 0.06 * W, size=(Nm, T, P))
        tracks[..., 1] = cy + rng.normal(0, 0.07 * H, size=(Nm, T, P))
        tracks[..., 0].sort(axis=-1)
    tracks[1, 1, ::5, 0] = np.nan
    tracks[2, :, :, :] = np.round(tracks[2]) + 0.5
    tracks[3, 0] = tracks[3, 0, 0]                  # all points on one pixel
    tracks[4, 2, :, 1] = -7                         # nothing inside the frame
    vis = rng.integers(0, 2, size=(Nm, T, P)).astype(np.uint8)
    v = _video(labels, tracks, vis, max_label=nlab - 1)
    npts = np.asarray([P, P, P, P, P, max(P - 3, 0)], np.int32)
    v.npts = torch.from_numpy(npts).to(_dev())
    b = Batch([v])
    b.hits.fill_(-5); b.uniq.fill_(-5)
    b.votes_all()
    torch.cuda.synchronize()
    hits = b.hits.cpu().numpy().reshape(Nm, T, nlab)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        h, u = ko.point_votes(tracks[q][:, : int(npts[q])], labels, 0, T - 1, nbins=nlab)
        assert np.array_equal(u, uniq[q]) and np.array_equal(h, hits[q]), (q, u, uniq[q])


def test_ragged_npts(pv_variant):
    from s2d_b200.pipeline import Batch
    rng = np.random.default_rng(5)
    T, Nm, P, H, W = 4, 6, 512, 90, 120
    labels = rng.integers(0, 4, size=(T, H, W)).astype(np.uint8)
    tracks = rng.uniform(0, 100, size=(Nm, T, P, 2)).astype(np.float32)
    vis = rng.integers(0, 2, size=(Nm, T, P)).astype(np.uint8)
    npts = np.asarray([512, 1, 0, 33, 400, 511], np.int32)
    v = _video(labels, tracks, vis, max_label=3)
    v.npts = torch.from_numpy(npts).to(_dev())
    b = Batch([v])
    b.votes_all()
    from s2d_b200 import _lib
    _lib.call("s2d_vis_reduce", b.descs.data_ptr(), 1, b.max_rows_x_T, b.cnt.data_ptr(), b.V.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    hits = b.hits.cpu().numpy().reshape(Nm, T, 4)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    V = b.V.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        n = int(npts[q])
        h, u = ko.point_votes(tracks[q][:, :n], labels, 0, T - 1, nbins=4)
        assert np.array_equal(u, uniq[q]) and np.array_equal(h, hits[q]), q
        assert np.array_equal(V[q], ko.visibility_mean(vis[q][:, :n]), equal_nan=True), q


@pytest.mark.parametrize("P", [4096, 1000, 77, 32, 5])
def test_vis_reduce_bit_packed_flags(P):
    """S2D_DESC_VIS_BITS: the producer hands the visibility flags over bit-packed (1/8 of the bytes); counts and the
    float32 means are the ones of the byte flags = the oracle's torch.mean restatement, ragged point counts included."""
    from s2d_b200.pipeline import Batch, VideoInput, pack_vis_bits
    rng = np.random.default_rng(P)
    Nm, T = 7, 5
    vis = (rng.random((Nm, T, P)) < 0.6).astype(np.uint8)
    npts = rng.integers(0, P + 1, size=Nm).astype(np.int32)
    npts[0] = P
    d = _dev()
    dv = torch.from_numpy(vis).to(d)
    for use_npts in (False, True):
        kw = dict(npts=torch.from_numpy(npts).to(d)) if use_npts else {}
        res = []
        for v in (VideoInput(vis=dv, dims=dict(H=8, W=8), **kw),
                  VideoInput(vis=pack_vis_bits(dv), vis_bits=True, dims=dict(H=8, W=8, P=P), **kw)):
            b = Batch([v], stages="V")
            b.run()
            torch.cuda.synchronize()
            res.append((b.cnt.cpu().numpy().reshape(Nm, T), b.V.cpu().numpy().reshape(Nm, T)))
        assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1], equal_nan=True)
        if not use_npts:
            assert np.array_equal(res[1][1], ko.visibility_mean(vis))
        else:
            want = np.stack([vis[q, :, :npts[q]].sum(1) for q in range(Nm)])
            assert np.array_equal(res[1][0], want)


@pytest.mark.parametrize("eps,ms", [(0.2, 5), (0.1, 5), (0.1, 3), (0.05, 5)])
def test_hamming_dbscan_vs_oracle(eps, ms):
    import ctypes as C
    from s2d_b200 import _lib
    rng = np.random.default_rng(11)
    dev = _dev()
    for it in range(25):
        n = int(rng.integers(1, 400))
        d = int(rng.integers(1, 200))
        if it == 0:
            n, d = 3000, 2100          # several word chunks and many row tiles
        base = rng.random((int(rng.integers(1, 6)), d)) < 0.5
        X = base[rng.integers(0, len(base), n)] ^ (rng.random((n, d)) < rng.choice([0.0, 0.02, 0.08]))
        if it % 3 == 0:
            X[rng.integers(0, n, max(1, n // 4))] = False
        stride = (d + 31) // 32
        pad = np.zeros((n, stride * 32), bool)
        pad[:, :d] = X
        words = np.packbits(pad.reshape(n, stride, 32), axis=-1, bitorder="little").view(np.uint32).reshape(n, stride)
        bits = torch.from_numpy(words.view(np.int32).copy()).to(dev)
        nw = C.c_int64()
        _lib.call("s2d_dbscan_work_ints", n, 1, C.byref(nw))
        work = torch.empty(nw.value + 2, dtype=torch.int32, device=dev)
        out = torch.empty(n, dtype=torch.int32, device=dev)
        _lib.call("s2d_hamming_dbscan", bits.data_ptr(), n, stride, d, eps, ms, work.data_ptr(), out.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), ko.dbscan_hamming(X, eps, ms)), (it, n, d)


def test_overlap_bits_vs_oracle():
    from s2d_b200 import _lib
    rng = np.random.default_rng(3)
    dev = _dev()
    st = torch.cuda.current_stream().cuda_stream
    for (Na, Nb, H, W) in [(5, 7, 30, 50), (70, 20, 96, 128), (33, 65, 100, 333)]:
        A = (rng.random((Na, H, W)) < 0.05).astype(np.uint8) * 255
        Bm = (rng.random((Nb, H, W)) < 0.4).astype(np.uint8)
        npix = H * W
        nw = (npix + 31) // 32
        dA, dB = torch.from_numpy(A).to(dev), torch.from_numpy(Bm).to(dev)
        bA = torch.empty(Na * nw, dtype=torch.int32, device=dev)
        bB = torch.empty(Nb * nw, dtype=torch.int32, device=dev)
        _lib.call("s2d_pack_bits", dA.data_ptr(), Na, npix, bA.data_ptr(), st)
        _lib.call("s2d_pack_bits", dB.data_ptr(), Nb, npix, bB.data_ptr(), st)
        I = torch.empty(Na * Nb, dtype=torch.int32, device=dev)
        aA = torch.empty(Na, dtype=torch.int32, device=dev)
        aB = torch.empty(Nb, dtype=torch.int32, device=dev)
        _lib.call("s2d_overlap_bits", bA.data_ptr(), Na, bB.data_ptr(), Nb, nw, I.data_ptr(), aA.data_ptr(),
                  aB.data_ptr(), st)
        torch.cuda.synchronize()
        rI, rA, rB = ko.overlap_counts(A, Bm)
        assert np.array_equal(I.cpu().numpy().reshape(Na, Nb), rI)
        assert np.array_equal(aA.cpu().numpy(), rA) and np.array_equal(aB.cpu().numpy(), rB)


def test_dense_overlap_equals_sparse_votes(golden_case):
    """K1 on rasterised tracks x one-hot masks == K2's hits (SURVEY.md section 8, row a12)."""
    from s2d_b200 import _lib
    from s2d_b200.pipeline import Batch
    name, g, labels, tracks, vis = golden_case
    dev = _dev()
    st = torch.cuda.current_stream().cuda_stream
    T, H, W = labels.shape
    Nm, _, P, _ = tracks.shape
    b = Batch([_video(labels, tracks, vis)])
    b.votes_all()
    L = b.host_descs[0].L
    hits = b.hits.cpu().numpy().reshape(Nm, T, L)
    npix, nw = H * W, (H * W + 31) // 32
    nq = min(Nm, 6)
    planes = torch.empty((T, H, W), dtype=torch.uint8, device=dev)
    for q in range(nq):
        tq = torch.from_numpy(np.ascontiguousarray(tracks[q])).to(dev)
        _lib.call("s2d_rasterise_tracks", tq.data_ptr(), T, P, H, W, planes.data_ptr(), st)
        torch.cuda.synchronize()
        ref_planes = np.stack([ko.rasterise_tracks(tracks[q][t], H, W) for t in range(T)])
        assert np.array_equal(planes.cpu().numpy(), ref_planes)
        for t in range(0, T, max(1, T // 3)):
            labs = np.unique(labels[t])
            onehot = np.stack([(labels[t] == l) for l in labs]).astype(np.uint8)
            dB = torch.from_numpy(onehot).to(dev)
            bA = torch.empty(nw, dtype=torch.int32, device=dev)
            bB = torch.empty(len(labs) * nw, dtype=torch.int32, device=dev)
            _lib.call("s2d_pack_bits", planes[t].data_ptr(), 1, npix, bA.data_ptr(), st)
            _lib.call("s2d_pack_bits", dB.data_ptr(), len(labs), npix, bB.data_ptr(), st)
            I = torch.empty(len(labs), dtype=torch.int32, device=dev)
            _lib.call("s2d_overlap_bits", bA.data_ptr(), 1, bB.data_ptr(), len(labs), nw, I.data_ptr(), None, None, st)
            torch.cuda.synchronize()
            assert np.array_equal(I.cpu().numpy(), hits[q, t, labs]), (name, q, t)


@pytest.mark.parametrize("Na,Nb,H,W", [(5, 7, 32, 48), (200, 20, 96, 128), (130, 300, 64, 80), (64, 33, 480, 854)])
def test_overlap_i8_tensor_core_vs_oracle(Na, Nb, H, W):
    """tcgen05 kind::i8 contraction == numpy int64 contraction, bit-exact."""
    from s2d_b200 import _lib
    rng = np.random.default_rng(Na * 1000 + Nb)
    dev = _dev()
    st = torch.cuda.current_stream().cuda_stream
    A = (rng.random((Na, H, W)) < 0.03).astype(np.uint8)
    Bm = (rng.random((Nb, H, W)) < 0.5).astype(np.uint8)
    Bm[0] = 1
    dA, dB = torch.from_numpy(A).to(dev), torch.from_numpy(Bm).to(dev)
    I = torch.full((Na * Nb,), -1, dtype=torch.int32, device=dev)
    _lib.call("s2d_overlap_i8", dA.data_ptr(), Na, dB.data_ptr(), Nb, H * W, I.data_ptr(), st)
    torch.cuda.synchronize()
    rI, _, _ = ko.overlap_counts(A, Bm)
    assert np.array_equal(I.cpu().numpy().reshape(Na, Nb), rI)


@pytest.mark.parametrize("F,L,H,W", [(3, 4, 16, 32), (6, 21, 48, 64), (36, 21, 96, 128), (13, 30, 120, 160),
                                     (10, 21, 17, 48), (50, 25, 64, 96), (12, 22, 19, 80),
                                     # few labels per frame and more than 256 rows: the label ring of the 256 x 256
                                     # tiling does not fit, the entry point falls back to 128 x 256 / 128 x 128 tiles
                                     (24, 11, 48, 64), (24, 14, 48, 64), (48, 6, 32, 64), (100, 3, 16, 64), (30, 18, 32, 48)])
def test_gram_labels_tensor_core_vs_oracle(F, L, H, W):
    """one-hot Gram matrix synthesised on-chip + tcgen05 kind::i8 == numpy one-hot contraction."""
    from s2d_b200 import _lib
    rng = np.random.default_rng(F * 100 + L)
    dev = _dev()
    labels = rng.integers(0, L, size=(F, H, W)).astype(np.uint8)
    labels[:, : H // 3] = 0
    d = torch.from_numpy(labels).to(dev)
    R = F * L
    G = torch.full((R * R,), -1, dtype=torch.int32, device=dev)
    import ctypes as C
    n = C.c_int64()
    _lib.call("s2d_overlap_gram_work_ints", F, L, H * W, C.byref(n))
    work = torch.full((n.value,), -7, dtype=torch.int32, device=dev)
    _lib.call("s2d_overlap_gram_labels", d.data_ptr(), F, L, H * W, work.data_ptr(), G.data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    X = (labels.reshape(F, 1, -1) == np.arange(L, dtype=np.uint8)[None, :, None]).reshape(R, -1).astype(np.int64)
    assert np.array_equal(G.cpu().numpy().reshape(R, R), X @ X.T)


@pytest.mark.parametrize("F,L,H,W,band", [(40, 21, 48, 64, 5), (64, 30, 32, 64, 8), (30, 18, 32, 48, 0), (36, 21, 96, 128, 40), (50, 11, 32, 64, 3)])
def test_gram_labels_banded_vs_oracle(F, L, H, W, band):
    """north_star kernel 1, "all mask pairs within a frame window": the banded Gram form computes only the 256 x 256 blocks
    whose frames lie within `band` of each other and returns the band layout [R][(2 band + 1) L]; every entry against the
    oracle's dense contraction of the one-hot masks (pairs beyond the band are not part of the output at all)."""
    import ctypes as C
    from s2d_b200 import _lib
    rng = np.random.default_rng(F * L + band)
    blocks = rng.integers(0, L, size=(F, (H + 7) // 8, (W + 7) // 8)).astype(np.uint8)
    labels = np.repeat(np.repeat(blocks, 8, axis=1), 8, axis=2)[:, :H, :W].copy()
    labels[:, 0, :L] = np.arange(L, dtype=np.uint8)
    R, Wb = F * L, (2 * band + 1) * L
    d = _dev()
    nw = C.c_int64()
    _lib.call("s2d_overlap_gram_band_work_ints", F, L, H * W, band, C.byref(nw))
    work = torch.empty(nw.value, dtype=torch.int32, device=d)
    Gb = torch.full((R * Wb,), -1, dtype=torch.int32, device=d)
    dlab = torch.from_numpy(labels).to(d)
    _lib.call("s2d_overlap_gram_labels_banded", dlab.data_ptr(), F, L, H * W, band, work.data_ptr(), Gb.data_ptr(),
              torch.cuda.current_stream(d).cuda_stream)
    torch.cuda.synchronize()
    X = (labels.reshape(F, 1, -1) == np.arange(L, dtype=np.uint8)[None, :, None]).reshape(R, -1)
    full, _, _ = ko.overlap_counts(X, X)
    want = np.zeros((R, Wb), np.int64)
    for f in range(F):
        for dd in range(-band, band + 1):
            if 0 <= f + dd < F:
                want[f * L:(f + 1) * L, (dd + band) * L:(dd + band + 1) * L] = full[f * L:(f + 1) * L, (f + dd) * L:(f + dd + 1) * L]
    assert np.array_equal(Gb.cpu().numpy().reshape(R, Wb), want)


def test_color_to_labels_vs_host_rule():
    """f1: colour PNG frames -> label ids on the GPU == rank of the RGB tuple among the non-black colours."""
    from s2d_b200.keymask_ident import _engine
    from s2d_b200.keymask_ident.crw_utils import rgb_to_label_ids
    rng = np.random.default_rng(4)
    for (F, H, W, ncol, black) in [(3, 33, 47, 5, True), (2, 64, 96, 40, True), (2, 30, 50, 7, False), (1, 17, 19, 255, True)]:
        pal = rng.integers(0, 256, size=(ncol, 3)).astype(np.uint8)
        pal[pal.sum(1) == 0] = 1
        if ncol >= 3:
            pal[1] = pal[0]; pal[1, 2] ^= 1          # colours differing in the last channel only
            pal[2] = pal[0]; pal[2, 0] ^= 128        # ... and in the first
        idx = rng.integers(0, ncol, size=(F, H, W))
        idx = np.repeat(np.repeat(idx[:, ::4, ::4], 4, axis=1), 4, axis=2)[:, :H, :W]   # piecewise constant
        rgb = pal[idx]
        if black:
            rgb[:, : H // 3] = 0
        labels, ncols = _engine.color_frames_to_labels(rgb)
        got = labels.cpu().numpy()
        for f in range(F):
            ref = rgb_to_label_ids(rgb[f])
            assert np.array_equal(got[f], ref.astype(np.uint8)), (F, H, W, ncol, f)
            assert ncols[f] == len(np.unique(ref[ref > 0]))


def _assert_same_as_oracle(res, ref, min_queries):
    """every field of a pipeline result against the oracle's: visibility floats exact, clusters / windows / candidates,
    per query (cluster, frame, mask, one2x, matches, per-pair intersection and union counts), groups, coverages, one2x."""
    assert res["status"] == ref["status"] == 1
    assert np.array_equal(res["V"], ref["V"], equal_nan=True)
    assert np.array_equal(res["labels1"], ref["labels1"])
    assert json_eq(res["clusters"], ref["clusters"])
    assert len(res["queries"]) == len(ref["queries"]) > min_queries
    for a, b in zip(res["queries"], ref["queries"]):
        assert (a["cluster_id"], a["frame_id"], a["mask_id"], a["one2x"]) == (b["cluster_id"], b["frame_id"], b["mask_id"], b["one2x"])
        assert a["matches"] == b["matches"]
        assert tuple(a["v_range"]) == tuple(b["v_range"]) and a["grid_size"] == b["grid_size"]
        assert [c[:5] for c in a["comps"]] == [c[:5] for c in b["comps"]]
        assert all(abs(x[5] - y[5]) <= 1e-6 * abs(y[5]) for x, y in zip(a["comps"], b["comps"]))   # iou: 1e-6 relative (north_star)
    ga = [(g["cluster_id"], g["visibility_to_temporal_factor"], g["overall_mask_ids_per_label"]) for g in res["groupings"]]
    gb = [(g["cluster_id"], g["visibility_to_temporal_factor"], g["overall_mask_ids_per_label"]) for g in ref["groupings"]]
    assert ga == gb
    assert res["video_coverage"] == ref["video_coverage"] and res["cluster_coverages"] == ref["cluster_coverages"]
    assert res["one2x"] == ref["one2x"]


def test_c1_shape_full_pipeline_vs_oracle():
    """BASELINE.json configs[0]: one 24-frame 480x854 video, 10 masks/frame, 1000 tracks per query -
    the whole device pipeline against the CPU oracle (counts, windows, matches, groups bit-exact)."""
    from s2d_b200.pipeline import Params, discover_keymasks
    from s2d_b200.synth import make_scene
    sc = make_scene(1234, T=24, H=480, W=854, M=10, P=1000, specials=True)
    res = discover_keymasks([_video(sc.labels, sc.tracks, sc.vis, max_label=10)], Params())[0]
    ref = ko.discover(sc.labels, sc.tracks, sc.vis)
    _assert_same_as_oracle(res, ref, 200)


@pytest.mark.parametrize("order", ["raster", "random"])
def test_c2_shape_full_pipeline_vs_oracle(order):
    """BASELINE.json configs[1], the benchmarked shape: a 36-frame 720p video, 20 masks/frame, 4096 tracks per query
    (the generator, seed and point order of bench.py's video 0) through the whole device pipeline - two words per
    frame-bit row (T > 32), 23 words per match-bit row (Nm ~ 708), the 128-thread x 32-point label-table kernel with
    TMA boxes - against the CPU oracle, every field."""
    from s2d_b200.pipeline import Params, VideoInput, discover_keymasks
    from s2d_b200.synth import make_scene_device
    sc = make_scene_device(2024, 36, 720, 1280, 20, 4096, _dev(), point_order=order)
    res = discover_keymasks([VideoInput(sc["labels"], sc["tracks"], sc["vis"], max_label=20)], Params())[0]
    ref = ko.discover(sc["labels"].cpu().numpy(), sc["tracks"].cpu().numpy(), sc["vis"].cpu().numpy())
    _assert_same_as_oracle(res, ref, 600)
    assert sc["labels"].shape[0] > 32 and len(res["query_frame"]) > 640


def json_eq(a, b):
    import json
    return json.loads(json.dumps(a)) == json.loads(json.dumps(b))


def test_query_permutation_and_batch_invariance():
    """the result of a video does not depend on which other videos share its batch, and K2 does not
    depend on the order of a query's points (SURVEY.md section 4, property tests)."""
    from s2d_b200.pipeline import Batch, Params, discover_keymasks
    from s2d_b200.synth import make_scene
    a = make_scene(77, T=10, H=72, W=96, M=4, P=96, specials=True)
    b = make_scene(78, T=14, H=60, W=80, M=3, P=64)
    alone = discover_keymasks([_video(a.labels, a.tracks, a.vis)], Params())[0]
    both = discover_keymasks([_video(b.labels, b.tracks, b.vis), _video(a.labels, a.tracks, a.vis)], Params())[1]
    assert alone["status"] == both["status"]
    assert [q["matches"] for q in alone["queries"]] == [q["matches"] for q in both["queries"]]
    assert json_eq(alone["groupings"], both["groupings"]) and json_eq(alone["clusters"], both["clusters"])
    rng = np.random.default_rng(0)
    perm = rng.permutation(a.tracks.shape[2])
    b1 = Batch([_video(a.labels, a.tracks, a.vis)]); b1.votes_all()
    b2 = Batch([_video(a.labels, np.ascontiguousarray(a.tracks[:, :, perm]), np.ascontiguousarray(a.vis[:, :, perm]))]); b2.votes_all()
    torch.cuda.synchronize()
    assert torch.equal(b1.hits, b2.hits) and torch.equal(b1.uniq, b2.uniq)


@pytest.mark.parametrize("P", [64, 6000])
def test_windowed_track_storage(P):
    """long-video layout: only the frames of a query's window are stored ([Nm][Tw][P][2] + tstart);
    also exercises the P > 4096 kernel variant."""
    from s2d_b200.pipeline import Batch, VideoInput
    rng = np.random.default_rng(P)
    T, H, W, Nm, Tw = 20, 50, 70, 9, 6
    labels = rng.integers(0, 5, size=(T, H, W)).astype(np.uint8)
    full = rng.uniform(-3, 75, size=(Nm, T, P, 2)).astype(np.float32)
    v0 = rng.integers(0, T - Tw + 1, size=Nm)
    v1 = v0 + rng.integers(0, Tw, size=Nm)
    win = np.stack([full[q, v0[q]:v0[q] + Tw] for q in range(Nm)])
    d = _dev()
    vid = VideoInput(labels=torch.from_numpy(labels).to(d), tracks=torch.from_numpy(np.ascontiguousarray(win)).to(d),
                     tstart=torch.from_numpy(v0.astype(np.int32)).to(d), max_label=4)
    b = Batch([vid], stages="LD")
    rowinfo = np.stack([np.zeros(Nm), np.zeros(Nm), v0, v1], axis=1).astype(np.int32)
    rowinfo[3, 1] = -1                                   # not a candidate: untouched
    b.upload_stage_b(rowinfo, 1, 1)
    b.hits.fill_(-5); b.uniq.fill_(-5)
    b.run()
    torch.cuda.synchronize()
    hits = b.hits.cpu().numpy().reshape(Nm, T, 5)
    uniq = b.uniq.cpu().numpy().reshape(Nm, T)
    for q in range(Nm):
        inside = np.zeros(T, bool)
        if q != 3:
            inside[v0[q]:v1[q] + 1] = True
            h, u = ko.point_votes(full[q], labels, int(v0[q]), int(v1[q]), nbins=5)
            assert np.array_equal(uniq[q, inside], u) and np.array_equal(hits[q, inside], h), q
        assert (uniq[q, ~inside] == -5).all() and (hits[q, ~inside] == -5).all(), q


def test_windowed_track_storage_partial_cover():
    """a stored track window [tstart, tstart + Ttr) that covers only part of the device-computed [v0, v1]: the frames
    without tracks must count as "no point landed" (iou 0) in selection and grouping, whatever hits / uniq held
    before - identical to a full-length run whose missing frames are NaN."""
    from s2d_b200.pipeline import Batch, VideoInput
    from s2d_b200.synth import make_scene
    sc = make_scene(77, T=20, H=60, W=80, M=4, P=64, occlude=False)
    Nm, T, P, _ = sc.tracks.shape
    rng = np.random.default_rng(5)
    Tw = 9
    ts = rng.integers(0, T - Tw + 1, size=Nm)
    rowinfo = np.stack([np.zeros(Nm), np.zeros(Nm), np.full(Nm, 2), np.full(Nm, T - 3)], axis=1).astype(np.int32)
    d = _dev()
    lab = torch.from_numpy(sc.labels).to(d)
    win = np.ascontiguousarray(np.stack([sc.tracks[q, ts[q]:ts[q] + Tw] for q in range(Nm)]))
    full = np.full_like(sc.tracks, np.nan)
    for q in range(Nm):
        full[q, ts[q]:ts[q] + Tw] = sc.tracks[q, ts[q]:ts[q] + Tw]
    outs = []
    for vid, poison in ((VideoInput(labels=lab, tracks=torch.from_numpy(win).to(d), tstart=torch.from_numpy(ts.astype(np.int32)).to(d)), 12345),
                        (VideoInput(labels=lab, tracks=torch.from_numpy(full).to(d)), 0)):
        b = Batch([vid], stages="LD")
        b.upload_stage_b(rowinfo, 1, 1)
        b.hits.fill_(poison); b.uniq.fill_(max(poison, 1))
        b.run()
        torch.cuda.synchronize()
        outs.append({k: getattr(b, k).cpu().numpy().copy() for k in ("mbits", "one2x", "nmatch", "glabel", "vidinfo", "clusterinfo")})
    assert outs[1]["nmatch"].sum() > 0
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k


def test_appearance_events_vs_reference_golden():
    """K3d (appearance_events_kernel, boolean_visibility_kernel) through the drop-in functions of both
    modules against vectors produced by the unmodified reference (oracle/make_golden_events.py)."""
    import os
    from s2d_b200.keymask_ident import cotracker_matching as cm, cotracker_occlusions as co
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "events.npz"))
    for name in g["names"]:
        V = torch.from_numpy(g[f"{name}__V"])
        sw, th, k = g[f"{name}__params"]
        for mod in (co, cm):
            ev = mod.extract_appearance_events(V, smoothing_window=int(sw), thresh=float(th), min_run_length=int(k))
            npairs, pairs = g[f"{name}__npairs"], g[f"{name}__pairs"]
            assert [len(ev[i]) for i in range(V.shape[0])] == npairs.tolist(), name
            flat = [p for i in range(V.shape[0]) for p in ev[i]]
            assert np.array_equal(np.asarray(flat, np.int32).reshape(-1, 2), pairs), name
            assert np.array_equal(mod.boolean_visibility(V, threshold=float(th)).numpy(), g[f"{name}__bool"]), name
        ev_o, _ = ko.appearance_events(g[f"{name}__V"], int(sw), float(th), int(k))
        assert ev_o == ev, name
    with pytest.raises(RuntimeError):
        co.extract_appearance_events(torch.zeros(2, 1), min_run_length=4)      # torch: padding >= input size


@pytest.mark.parametrize("n1,n2,H,W", [(5, 7, 33, 47), (40, 130, 64, 80), (130, 70, 96, 128), (1, 1, 8, 8)])
def test_mask_iou_consumers_vs_reference_formulas(n1, n2, H, W):
    """f3: mask_iou_matrix / BatchIoU on the K1 kernels against the reference's own torch formulas
    (mask2former_video/engine/train_loop.py:378-388, cutler/tools/get_self_training_ann.py:80-89) on CPU."""
    from s2d_b200.mask_iou import BatchIoU, mask_iou_matrix
    rng = np.random.default_rng(n1 * 1000 + n2)
    x = torch.from_numpy((rng.random((n1, H, W)) < 0.3).astype(np.float32))
    y = torch.from_numpy((rng.random((n2, H, W)) < 0.4).astype(np.float32))
    y[0] = 0                                                   # empty mask: 0/0 -> nan like the reference
    xf, yf = x.reshape(n1, -1), y.reshape(n2, -1)
    inter = xf @ yf.t()
    sx, sy = xf.sum(1)[:, None].expand(n1, n2), yf.sum(1)[None, :].expand(n1, n2)
    for mode, want in (("iou", inter / (sx + sy - inter)), ("ioy", inter / sy)):
        got = mask_iou_matrix(x, y, mode=mode)
        assert got.dtype == torch.float32 and torch.equal(torch.isnan(got), torch.isnan(want))
        assert torch.equal(torch.nan_to_num(got), torch.nan_to_num(want)), mode
    p1, p2 = torch.from_numpy(rng.random((n1, H, W)).astype(np.float32)), torch.from_numpy(rng.random((n2, H, W)).astype(np.float32))
    m1, m2 = (p1 > 0.5), (p2 > 0.5)
    a, b = m1[:, None].expand(-1, n2, -1, -1), m2[None].expand(n1, -1, -1, -1)
    want = torch.sum(a * (a == b), dim=[-1, -2]).to(torch.float) / torch.sum(a + b, dim=[-1, -2])
    assert torch.equal(BatchIoU(p1, p2), want)


def test_cuda_graph_replay_matches_direct_run(golden_case):
    """Batch.capture / replay: the whole path recorded once as a CUDA graph gives the same result tables."""
    from s2d_b200.pipeline import Batch, Params
    name, g, labels, tracks, vis = golden_case
    par = Params(g["visibility_threshold"], g["matching_threshold"])
    b1 = Batch([_video(labels, tracks, vis)])
    b1.run(par)
    torch.cuda.synchronize()
    want = b1.fetch_summary()
    b2 = Batch([_video(labels, tracks, vis)])
    b2.capture(par)
    for _ in range(3):
        b2.replay()
    torch.cuda.synchronize()
    got = b2.fetch_summary()
    for k in want:
        assert np.array_equal(want[k], got[k]), (name, k)
    # (hits / uniq are only written for the voted tiles, the rest of those buffers is uninitialised: the result
    # tables above are what depends on them)


@pytest.mark.parametrize("seed,T,H,W,M,P,kw", [
    (11, 16, 120, 160, 5, 256, dict(specials=True)),
    (12, 20, 96, 128, 8, 130, dict(dup_rate=0.2)),
    (13, 14, 200, 320, 12, 512, dict(specials=True, noise=1.5)),
    (14, 30, 64, 80, 4, 64, dict(occlude=False)),
    (15, 12, 240, 426, 6, 1000, dict(full_cover_frames=(3, 4), specials=True)),
    (16, 18, 144, 256, 10, 300, dict(noise=0.0)),
])
def test_random_scenes_full_pipeline_vs_oracle(seed, T, H, W, M, P, kw):
    """Seeded scenes of different shapes (odd point counts, duplicates, NaN/inf/half-integer coordinates,
    frames without background, no occlusion): the whole device pipeline - whatever status the video ends with -
    against the CPU oracle restatement of the reference (itself pinned to the reference's goldens)."""
    from s2d_b200.pipeline import Params, discover_keymasks
    from s2d_b200.synth import make_scene
    sc = make_scene(seed, T=T, H=H, W=W, M=M, P=P, **kw)
    for mt in (0.5, 0.35):
        res = discover_keymasks([_video(sc.labels, sc.tracks, sc.vis, max_label=M)], Params(matching_threshold=mt))[0]
        ref = ko.discover(sc.labels, sc.tracks, sc.vis, matching_threshold=mt)
        assert res["status"] == ref["status"], (seed, mt)
        assert np.array_equal(res["V"], ref["V"], equal_nan=True)
        assert np.array_equal(res["labels1"], ref["labels1"])
        assert json_eq(res["clusters"], ref["clusters"])
        if ref["status"] != 1:
            continue
        assert len(res["queries"]) == len(ref["queries"])
        for a, b in zip(res["queries"], ref["queries"]):
            assert (a["cluster_id"], a["frame_id"], a["mask_id"], a["one2x"]) == (b["cluster_id"], b["frame_id"], b["mask_id"], b["one2x"])
            assert a["matches"] == b["matches"]
            assert [c[:5] for c in a["comps"]] == [c[:5] for c in b["comps"]]
        ga = [(g["cluster_id"], g["visibility_to_temporal_factor"], g["overall_mask_ids_per_label"]) for g in res["groupings"]]
        gb = [(g["cluster_id"], g["visibility_to_temporal_factor"], g["overall_mask_ids_per_label"]) for g in ref["groupings"]]
        assert ga == gb
        assert res["video_coverage"] == ref["video_coverage"] and res["cluster_coverages"] == ref["cluster_coverages"]
        assert res["one2x"] == ref["one2x"]
