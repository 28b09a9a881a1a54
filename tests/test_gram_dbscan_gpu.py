"""DBSCAN #2 on the Gram path at the row counts that take it (videos with >= 2048 query rows: every 300-frame video, the
long videos of a list): K1 on the unpacked match rows, the grouping on planted match tables against the oracle with an
exact BLAS-speed DBSCAN, two videos end to end, and stage B at the frame limit (needs a B200)."""
import numpy as np
import pytest
import torch

from oracle import keymask_oracle as ko
from s2d_b200 import _lib
from s2d_b200._lib import S2D_CLINFO_WORDS, S2D_MAX_CLUSTERS, S2D_VIDINFO_WORDS
from tests.gram_dbscan_reference import dbscan_hamming_fast, expected_grouping, plant_census, planted_video

pytestmark = pytest.mark.gpu


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _st():
    return torch.cuda.current_stream(_dev()).cuda_stream


def _pack(X):
    """[N, D] bool -> [N, ceil(D / 32)] int32 words, bit d % 32 of word d // 32 = X[:, d]"""
    N, D = X.shape
    NW = (D + 31) // 32
    pad = np.zeros((N, NW * 32), bool)
    pad[:, :D] = X
    return np.packbits(pad.reshape(N, NW, 32), axis=-1, bitorder="little").view(np.int32).reshape(N, NW)


def _gram_ref(A, B):
    """exact A B^T of 0/1 rows from float32 BLAS (sums stay below 2^24)"""
    return (A.astype(np.float32) @ B.astype(np.float32).T).astype(np.int64)


# ----------------------------------------------------------------------------- K1 at the Gram shapes
def _match_rows(rng, N, D):
    """empty rows, all-ones rows, rows one bit apart, sparse and dense random rows"""
    dens = rng.choice([0.0, 0.002, 0.03, 0.3, 0.85, 1.0], size=N, p=[0.1, 0.2, 0.3, 0.25, 0.1, 0.05])
    X = rng.random((N, D), dtype=np.float32) < dens[:, None].astype(np.float32)
    i = rng.choice(N - 1, size=N // 10, replace=False)
    X[i + 1] = X[i]
    X[i + 1, rng.integers(0, D, size=len(i))] ^= True
    X[0] = False
    X[-1] = True
    return X


@pytest.mark.parametrize("N", [2048, 2049, 2111, 2144, 3600, 9000])
def test_overlap_i8_gram_of_match_rows(N):
    """s2d_unpack_bits then s2d_overlap_i8 with A = B = the same planes, as stage D runs them for a video of N rows:
    K = 32 * ceil(N / 32) covers K mod 128 = 0, 32, 64 and 96, the last 128-row and 256-column tiles are partial. The whole
    N x N result against the exact float32 reference."""
    rng = np.random.default_rng(N)
    X = _match_rows(rng, N, N)
    words = _pack(X)
    NW = words.shape[1]
    K = NW * 32
    assert K % 128 == {2048: 0, 2049: 32, 2111: 64, 2144: 96, 3600: 32, 9000: 64}[N]
    d = _dev()
    bits = torch.from_numpy(words).to(d)
    planes = torch.full((N * K,), 7, dtype=torch.uint8, device=d)
    G = torch.full((N * N,), -1, dtype=torch.int32, device=d)
    _lib.call("s2d_unpack_bits", bits.data_ptr(), N, NW, K, planes.data_ptr(), _st())
    _lib.call("s2d_overlap_i8", planes.data_ptr(), N, planes.data_ptr(), N, K, G.data_ptr(), _st())
    torch.cuda.synchronize()
    pl = planes.view(N, K).cpu().numpy()
    assert np.array_equal(pl[:, :N], X) and not pl[:, N:].any()
    assert np.array_equal(G.view(N, N).cpu().numpy(), _gram_ref(X, X))


@pytest.mark.parametrize("Na,Nb,K", [(3000, 100, 4000), (2999, 257, 1040)])
def test_overlap_i8_mask_iou_shapes(Na, Nb, K):
    """non-square contractions of the mask-IoU kind: Nb = 100 (one 128-column tile), Nb = 257 (a 256-column tile and one
    column of the next), K a multiple of 16 but not of 128"""
    rng = np.random.default_rng(Na + Nb)
    A = _match_rows(rng, Na, K).astype(np.uint8)
    B = _match_rows(rng, Nb, K).astype(np.uint8)
    d = _dev()
    dA, dB = torch.from_numpy(A).to(d), torch.from_numpy(B).to(d)
    I = torch.full((Na * Nb,), -1, dtype=torch.int32, device=d)
    _lib.call("s2d_overlap_i8", dA.data_ptr(), Na, dB.data_ptr(), Nb, K, I.data_ptr(), _st())
    torch.cuda.synchronize()
    assert np.array_equal(I.view(Na, Nb).cpu().numpy(), _gram_ref(A, B))


# ----------------------------------------------------------------------------- grouping on planted match tables
def _planted_batch(pvs, gram_min_rows):
    """a stage-D batch of dims-only videos whose match tables (rowinfo, mbits, one2x, vidinfo) are the planted ones"""
    from s2d_b200.pipeline import Batch, VideoInput
    d = _dev()
    b = Batch([VideoInput(dims=dict(T=4, H=8, W=8, P=2, Nm=pv["Nm"])) for pv in pvs], device=d, stages="D",
              gram_min_rows=gram_min_rows)
    for vi, pv in enumerate(pvs):
        hd = b.host_descs[vi]
        Nm = pv["Nm"]
        assert hd.NW == pv["NW"]
        b.rowinfo[4 * hd.row0:4 * (hd.row0 + Nm)] = torch.from_numpy(pv["rowinfo"].reshape(-1)).to(d)
        b.mbits[hd.mbits_off:hd.mbits_off + Nm * hd.NW] = torch.from_numpy(pv["mbits"].view(np.int32).reshape(-1)).to(d)
        b.one2x[hd.row0:hd.row0 + Nm] = torch.from_numpy(pv["one2x"]).to(d)
        w = vi * S2D_VIDINFO_WORDS
        b.vidinfo[w:w + 4] = torch.tensor([pv["nclusters"], 1, pv["maxid"], 0], dtype=torch.int32, device=d)
    return b


def _check_grouping(b, pvs, exps, tag):
    torch.cuda.synchronize()
    glabel = b.glabel.cpu().numpy()
    clinfo = b.clusterinfo.cpu().numpy().reshape(b.nv, S2D_MAX_CLUSTERS, S2D_CLINFO_WORDS)
    grp_n, grp_o = b.grp_n.cpu().numpy(), b.grp_one2x.cpu().numpy()
    vidinfo = b.vidinfo.cpu().numpy().reshape(b.nv, S2D_VIDINFO_WORDS)
    for vi, (pv, exp) in enumerate(zip(pvs, exps)):
        hd = b.host_descs[vi]
        Nm, K = pv["Nm"], pv["nclusters"]
        assert vidinfo[vi, 3] == exp["status"] == 1, (tag, vi)
        got = glabel[hd.row0:hd.row0 + Nm]
        bad = np.nonzero(got != exp["glabel"])[0]
        assert len(bad) == 0, (tag, vi, len(bad), bad[:8], got[bad[:8]], exp["glabel"][bad[:8]], pv["kinds"][bad[:8]])
        assert np.array_equal(clinfo[vi, :K, 5:15], exp["clinfo"]), (tag, vi)
        for c in range(K):
            base = 16 * hd.row0 + c * Nm
            want_n, want_o = np.zeros(Nm, np.int64), np.zeros(Nm, np.int64)
            for (cc, l), (n, o) in exp["grp"].items():
                if cc == c:
                    want_n[l], want_o[l] = n, o
            assert np.array_equal(grp_n[base:base + Nm], want_n) and np.array_equal(grp_o[base:base + Nm], want_o), (tag, vi, c)


def _run_both_paths(pvs, gram_min_rows=1):
    exps = [expected_grouping(pv) for pv in pvs]
    b = _planted_batch(pvs, gram_min_rows)
    for gram in (True, False):
        b.clusterinfo.fill_(12345)
        b.group(gram=gram)
        _check_grouping(b, pvs, exps, "gram" if gram else "bits")
    return b, exps


@pytest.mark.parametrize("Nm", [2047, 2048, 3600, 9000])
def test_group_stage_on_planted_match_tables(Nm):
    """DBSCAN #2 and the grouping of one video whose match tables are planted (tests/gram_dbscan_reference.py): 16
    clusters interleaved in row order with column spans in all three (eps, min_samples) regimes, hubs with exactly
    min_samples and min_samples - 1 neighbours, spokes at exactly kmax, rows at kmax + 1, border rows between two cores,
    noise, all-zero rows, candidates above the largest matched id, non-candidate rows with stray bits. Once with the
    distances from the Gram matrix (unpack, overlap_i8, group_gram as run() enqueues them) and once from the bit rows:
    per row glabel, per cluster the crop, kmax, min_samples, groups, matched / one2x / candidate counts, per group the
    count and one2x sum, and the status, all as ko.temporal_clustering gives them."""
    pv = planted_video(Nm, Nm)
    b, (exp,) = _run_both_paths([pv])
    assert b.gram is not None
    cen = plant_census(pv, exp)
    for key in ("clusters_ge3_groups", "border", "border_two_groups", "noise", "zero_forced", "kmax_pairs", "kmax1_pairs",
                "ms_rows", "ms1_rows", "skipped"):
        assert cen[key] > 0, (key, cen)
    assert cen["regimes"] == {(0.05, 5), (0.1, 5), (0.1, 3)}


def test_group_stage_on_a_batch_of_big_and_small_videos():
    """a big video with an odd row count, a small one (bit path: no Gram matrix, gram_off -1) and a second big video, in
    one batch with the product's threshold: the second Gram matrix starts at the 16-byte aligned offset past the first"""
    pvs = [planted_video(71, 2061, nclusters=12), planted_video(72, 700, nclusters=5, spans=[6, 30, 51, 200, 10]),
           planted_video(73, 2300, nclusters=9)]
    b, exps = _run_both_paths(pvs, gram_min_rows=2048)
    offs = b.gram_off.cpu().tolist()
    pad = (-(2061 * 2061)) % 4
    assert pad and offs == [0, -1, 2061 * 2061 + pad]
    assert b.gram.numel() == 2061 * 2061 + pad + 2300 * 2300


# ----------------------------------------------------------------------------- end to end at real row counts
@pytest.fixture
def fast_oracle_dbscan(monkeypatch):
    monkeypatch.setattr(ko, "dbscan_hamming", dbscan_hamming_fast)


def _summaries_equal(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_c4_long_video_on_the_gram_path_vs_oracle(fast_oracle_dbscan):
    """A VIPSeg-like C4 video scaled down in pixels and points: 100 frames (4 words per frame-bit row), 30 objects,
    more than 2048 query rows, so DBSCAN #2 runs on the Gram path; every field against the oracle, and the same video in a
    batch that never takes the Gram path gives identical result tables. Scenes of moving objects give about one group per
    cluster at this size: this checks the plumbing of the path, the planted tables above check the grouping."""
    from s2d_b200.pipeline import Batch, Params, VideoInput
    from s2d_b200.synth import make_scene
    from tests.test_gpu_parity import _assert_same_as_oracle
    sc = make_scene(4101, T=100, H=72, W=128, M=30, P=64)
    Nm = sc.tracks.shape[0]
    assert Nm >= 2048 and sc.labels.shape[0] >= 97
    d = _dev()
    vid = VideoInput(torch.from_numpy(sc.labels).to(d), torch.from_numpy(sc.tracks).to(d), torch.from_numpy(sc.vis).to(d),
                     max_label=int(sc.labels.max()))
    summ = []
    for gmr in (2048, 10 ** 9):
        b = Batch([vid], gram_min_rows=gmr)
        assert (b.gram is not None) == (gmr == 2048)
        b.run(Params())
        torch.cuda.synchronize()
        summ.append(b.fetch_summary())
        if gmr == 2048:
            got = b.decode()[0]
    _summaries_equal(*summ)
    ref = ko.discover(sc.labels, sc.tracks, sc.vis)
    _assert_same_as_oracle(got, ref, 1000)


def test_c3_shaped_video_on_the_gram_path_vs_oracle(fast_oracle_dbscan):
    """test_workloads.py's windowed C3-shaped video (300 frames of 90 x 160, bit-packed flags, <= 64-frame track windows)
    with M = 8 instead of 6: 2243 query rows instead of about 1800, so DBSCAN #2 runs on the Gram path as it does for C3
    itself; every field against the oracle, and the grouping re-run from the bit rows gives identical tables. Like the
    C4 test, this checks plumbing: such scenes give about one group per cluster."""
    from s2d_b200 import workloads as wl
    from tests.test_gpu_parity import _assert_same_as_oracle
    dev = _dev()
    window = 64
    spec = wl.VideoSpec("c3gram", 31064, 300, 90, 160, 8, 64, window=window, vis_bits=True)
    res, st, (batch, scenes, vids) = wl.DeviceRunner(dev).run_list([spec], keep_batch=True)
    torch.cuda.synchronize()
    assert batch.gram is not None and batch.host_descs[0].Nm >= 2048
    got = batch.decode()[0]
    gram_summ = batch.fetch_summary()
    batch.group(gram=False)
    torch.cuda.synchronize()
    _summaries_equal(gram_summ, batch.fetch_summary())
    sc = scenes[0]
    Nm, Ttr, P, _ = sc["tracks"].shape
    ts = sc["tstart"].cpu().numpy()
    win = sc["tracks"].cpu().numpy()
    full = np.full((Nm, spec.T, P, 2), np.nan, np.float32)
    for q in range(Nm):
        full[q, ts[q]:ts[q] + window] = win[q]
    words = sc["vis"].cpu().numpy().view(np.uint32)
    vis = np.unpackbits(words.view(np.uint8).reshape(Nm, spec.T, -1), axis=2, bitorder="little")[:, :, :P]
    ref = ko.discover(sc["labels"].cpu().numpy(), full, vis)
    _assert_same_as_oracle(got, ref, 1000)


# ----------------------------------------------------------------------------- stage B at the frame limit
@pytest.mark.parametrize("T", [1024, 1000])
def test_stage_b_at_the_frame_limit_vs_oracle(T, fast_oracle_dbscan):
    """Stages A-B on videos of 1000 and 1024 frames (32 words per frame-bit row, the frame limit of s2d_label_stats and
    s2d_windows): visibility floats, DBSCAN #1 labels and the clusters' windows and candidates against the oracle."""
    from s2d_b200.pipeline import Batch, VideoInput
    from s2d_b200.synth import make_scene
    from tests.test_gpu_parity import json_eq
    sc = make_scene(77 + T, T=T, H=16, W=24, M=3, P=8)
    d = _dev()
    b = Batch([VideoInput(labels=torch.from_numpy(sc.labels).to(d), vis=torch.from_numpy(sc.vis).to(d), max_label=3)],
              stages="LVB")
    assert b.host_descs[0].TW == 32
    b.run()
    torch.cuda.synchronize()
    got = b.decode()[0]
    V = ko.visibility_mean(sc.vis)
    qf, ql, _ = ko.global_id_lookup(sc.labels)
    lab1, clusters = ko.visibility_windows(V, qf, ql)
    assert np.array_equal(got["V"], V, equal_nan=True)
    assert np.array_equal(got["labels1"], lab1)
    assert json_eq(got["clusters"], clusters) and len(clusters) >= 1


def test_frame_limit_is_refused_past_1024():
    """T = 1025 is refused by Batch, and s2d_label_stats refuses max_T = 1025 with a nonzero return"""
    from s2d_b200.pipeline import Batch, VideoInput
    d = _dev()
    with pytest.raises(AssertionError):
        Batch([VideoInput(labels=torch.zeros((1025, 4, 4), dtype=torch.uint8, device=d), dims=dict(Nm=1, P=1))], stages="L")
    b = Batch([VideoInput(labels=torch.zeros((1024, 4, 4), dtype=torch.uint8, device=d), dims=dict(Nm=1, P=1))], stages="L")
    p = lambda t: t.data_ptr()
    rc = _lib.load().s2d_label_stats(p(b.descs), 1, 1025, b.max_npix, b.total_frames, p(b.area), p(b.gid_of),
                                     p(b.frameinfo), p(b.qframe), p(b.qlabel), p(b.vidinfo), _st())
    assert rc != 0
