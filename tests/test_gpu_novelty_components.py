"""PCA novelty detection with more than one component (params.n_components > 1) on the GPU: the novelty kernel
against the oracle, rank 1 left as it was, K2's exact path, training, whole sequences against the CPU port, the
clip-resident driver, the dependent-launch chain and the error paths.  Needs a GPU: `pytest -m gpu`."""
import os
import subprocess
import sys

import cv2 as cv
import numpy as np
import pytest
import yaml

import pcm_oracle as orc
from helpers import PKG, GoldenSeq, polygons, sha1
from test_gpu_parity import _random_forest_arrays

pytestmark = pytest.mark.gpu

NOVELTY_RTOL = 1e-5


def _pca(rng, F, k):
    """Random mean and k orthonormal components (QR), scikit-learn's layout: components [k, F]."""
    q, _ = np.linalg.qr(rng.normal(size=(F, k)))
    return rng.random(F), np.ascontiguousarray(q.T)


def _features(features):
    n, spaces = orc.parse_features(features)
    return n, spaces, 3 * (1 + 8 * n) * len(spaces)


@pytest.mark.parametrize("features,shape", [("8 hsv_lab", (37, 70)), ("3 rgb_hsv_lab", (29, 45)), ("16 hsv", (41, 66)),
                                            ("2 rgb", (9, 13)), ("16 rgb_hsv_lab", (36, 40))])
@pytest.mark.parametrize("k", [2, 3, 5, 8])
def test_rank_k_novelty_error_matches_the_oracle(features, shape, k):
    """Synthetic PCAs of rank k (with k = 2 the second model is rank 1: a mixed blend), crops in two opposite corners of
    the frame, alone and blended: the novelty map within 1e-5 relative of the oracle, P(fg) still bit-equal."""
    from pcm import capi
    from pcm.providers import grid_segments
    rng = np.random.default_rng(100 * k + len(features) + shape[0])
    n, spaces, F = _features(features)
    hh, w = shape
    H, W = hh + 21, w + 33
    frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    t0, t1 = _random_forest_arrays(rng, 6, 5, F), _random_forest_arrays(rng, 4, 7, F)
    pcas = [_pca(rng, F, k), _pca(rng, F, 1 if k == 2 else k)]
    h = capi.Handle(0, debug=True)
    h.set_features(n, spaces)
    h.add_model_arrays(0, t0)
    h.add_model_arrays(5, t1)
    for m, (mean, comps) in enumerate(pcas):
        h.set_novelty(m, mean, comps)
    for rect in [(0, 0, w, hh), (W - w, H - hh, w, hh)]:
        crop = frame[rect[1]:rect[1] + hh, rect[0]:rect[0] + w]
        X = orc.get_features_int(orc.build_planes(crop, spaces), n)
        p = [orc.forest_p1(orc.forest_from_arrays(t, F), X) for t in (t0, t1)]
        e = [orc.novelty_error(X, mean, comps) for mean, comps in pcas]
        seg = grid_segments(crop, 5)
        S = int(seg.max()) + 1
        for blend, tau in [(False, 0.0), (True, 0.35)]:
            want_p = orc.blend(p[0], p[1], tau) if blend else p[0]
            want_e = orc.blend(e[0], e[1], tau) if blend else e[0]
            thr = float(np.median(want_e))
            prm = capi.Handle.make_params(0, 1 if blend else -1, 1 - tau, tau, novelty=True, dilation_kernel=3,
                                          outlier_threshold=thr)
            mask = np.zeros(frame.shape, np.uint8)
            h.update(frame, rect, seg, S, None, prm, mask)
            d = h.debug_last(hh, w, S)
            assert np.array_equal(d["p1"], want_p), (rect, blend)
            np.testing.assert_allclose(d["sa"], want_e, rtol=NOVELTY_RTOL, atol=0)
            scores, _ = orc.saliency_scores(want_p, want_e, seg, thr, np.full(S, -1, np.float32), 0.0)
            np.testing.assert_allclose(d["scores"], scores, rtol=NOVELTY_RTOL, atol=1e-6)
    h.close()


def test_rank_1_through_set_novelty_k_is_the_rank_1_path():
    """k = 1 handed over as a [1, F] array (pcm_set_novelty_k) leaves the state pcm_set_novelty leaves: the same bits for
    the novelty map, the scores and the mask, the same launches and no novelty-kernel launch.  A rank-3 model adds one
    novelty-kernel launch per frame (profile id 7)."""
    from pcm import capi
    from pcm.providers import voronoi_segments
    rng = np.random.default_rng(8)
    n, spaces, F = _features("8 hsv_lab")
    frame = rng.integers(0, 256, (140, 190, 3), dtype=np.uint8)
    rect = (11, 7, 160, 120)
    crop = frame[7:127, 11:171]
    seg = voronoi_segments(crop, 50, seed=2)
    S = int(seg.max()) + 1
    t0, t1 = _random_forest_arrays(rng, 8, 6, F), _random_forest_arrays(rng, 8, 6, F)
    pcas = [_pca(rng, F, 1), _pca(rng, F, 1)]
    prm = capi.Handle.make_params(0, 1, 0.6, 0.4, novelty=True, dilation_kernel=5, outlier_threshold=2.0)
    out = []
    for two_d in (False, True):
        h = capi.Handle(0, debug=True)
        h.set_features(n, spaces)
        h.add_model_arrays(0, t0)
        h.add_model_arrays(9, t1)
        for m, (mean, comps) in enumerate(pcas):
            h.set_novelty(m, mean, comps if two_d else comps[0])
        h.profile_enable(True)
        mask = np.zeros(frame.shape, np.uint8)
        before = h.launch_count
        h.update(frame, rect, seg, S, None, prm, mask)
        d = h.debug_last(120, 160, S)
        prof = h.profile_read(names=capi.ALL_KERNEL_NAMES)
        out.append((d["sa"].tobytes(), d["scores"].tobytes(), mask.tobytes(), h.launch_count - before, prof["novelty"][1]))
        h.close()
    assert out[0] == out[1]
    assert out[0][4] == 0
    h = capi.Handle(0, debug=True)
    h.set_features(n, spaces)
    h.add_model_arrays(0, t0)
    h.set_novelty(0, *_pca(rng, F, 3))
    h.profile_enable(True)
    before = h.launch_count
    h.update(frame, rect, seg, S, None, capi.Handle.make_params(0, novelty=True), np.zeros(frame.shape, np.uint8))
    prof = h.profile_read(names=capi.ALL_KERNEL_NAMES)
    assert prof["novelty"][1] == 1 and h.launch_count - before == out[0][3] + 1
    assert set(h.profile_read()) == set(capi.KERNEL_NAMES)
    h.close()


@pytest.mark.parametrize("keep_maps", [False, True])
def test_exact_path_reads_the_novelty_map(keep_maps):
    """Every label forced onto K2's exact path, two blended rank-3 models: scores and masks do not depend on whether the
    per-pixel maps are kept, and the scores are the reference's sequential float32 accumulation (to the novelty
    tolerance)."""
    from pcm import capi
    from pcm.providers import voronoi_segments
    rng = np.random.default_rng(31)
    hgt, wid, n, spaces = 75, 118, 3, ["lab", "rgb"]
    F = 3 * (1 + 8 * n) * len(spaces)
    frame = rng.integers(0, 256, (hgt + 9, wid + 14, 3), dtype=np.uint8)
    rect = (6, 4, wid, hgt)
    crop = frame[4:4 + hgt, 6:6 + wid]
    t0, t1 = _random_forest_arrays(rng, 7, 6, F), _random_forest_arrays(rng, 50, 3, F)
    pcas = [_pca(rng, F, 3), _pca(rng, F, 3)]
    X = orc.get_features_int(orc.build_planes(crop, spaces), n)
    tau = 0.7
    sa = orc.blend(orc.novelty_error(X, *pcas[0]), orc.novelty_error(X, *pcas[1]), tau)
    thr = float(np.percentile(sa, 40))
    seg = voronoi_segments(crop, 45, seed=5)
    S = int(seg.max()) + 1
    prm = capi.Handle.make_params(0, 1, 1 - tau, tau, novelty=True, dilation_kernel=3, outlier_threshold=thr)
    res = {}
    for keep in (keep_maps, not keep_maps):
        h = capi.Handle(0)
        h.set_debug(keep, force_exact=True)
        h.set_features(n, spaces)
        h.add_model_arrays(0, t0)
        h.add_model_arrays(1, t1)
        for m, (mean, comps) in enumerate(pcas):
            h.set_novelty(m, mean, comps)
        mask = np.zeros(frame.shape, np.uint8)
        h.update(frame, rect, seg, S, None, prm, mask)
        res[keep] = (h.debug_scores(S), mask)
        h.close()
    d, mask = res[keep_maps]
    p1 = orc.blend(orc.forest_p1(orc.forest_from_arrays(t0, F), X), orc.forest_p1(orc.forest_from_arrays(t1, F), X), tau)
    scores, areas = orc.saliency_scores(p1, sa, seg, thr, np.full(S, -1, np.float32), 0.0)
    assert d["n_exact"] == S and np.array_equal(d["areas"], areas)
    np.testing.assert_allclose(d["scores"], scores, rtol=NOVELTY_RTOL, atol=1e-6)
    assert np.array_equal(res[not keep_maps][0]["scores"], d["scores"])
    assert np.array_equal(res[not keep_maps][1], mask)


def test_banded_host_feed_gives_the_same_map():
    """A page-locked 1080p frame is fed to K0 / the novelty kernel / K1 in row bands; the result equals the unbanded
    update bit for bit, and sampled pixels match the oracle."""
    from pcm import capi
    from pcm.providers import grid_segments
    rng = np.random.default_rng(4)
    n, spaces, F = _features("8 hsv_lab")
    frame = rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    rect = (0, 0, 1920, 1080)
    seg = grid_segments(frame, 16)
    S = int(seg.max()) + 1
    t0, t1 = _random_forest_arrays(rng, 10, 6, F), _random_forest_arrays(rng, 10, 6, F)
    pcas = [_pca(rng, F, 3), _pca(rng, F, 5)]
    h = capi.Handle(0, debug=True)
    h.set_features(n, spaces)
    h.add_model_arrays(0, t0)
    h.add_model_arrays(3, t1)
    for m, (mean, comps) in enumerate(pcas):
        h.set_novelty(m, mean, comps)
    prm = capi.Handle.make_params(0, 1, 0.25, 0.75, novelty=True, dilation_kernel=7, outlier_threshold=3.0)
    got = []
    pinned = np.empty_like(frame)
    pinned[...] = frame
    for src in (frame, capi.host_register(pinned)):
        mask = np.zeros(frame.shape, np.uint8)
        h.update(src, rect, seg, S, None, prm, mask)
        d = h.debug_last(1080, 1920, S)
        got.append((d["sa"], d["scores"], mask))
    capi.host_unregister(pinned)
    h.close()
    assert got[0][0].tobytes() == got[1][0].tobytes()
    assert got[0][1].tobytes() == got[1][1].tobytes() and got[0][2].tobytes() == got[1][2].tobytes()
    rows = np.concatenate([rng.integers(0, 1080, 300), [0, 1079, 517, 518, 519]])
    cols = np.concatenate([rng.integers(0, 1920, 300), [0, 1919, 5, 1917, 960]])
    X = orc.features_at(orc.build_planes(frame, spaces), n, rows, cols)
    want = orc.blend(orc.novelty_error(X, *pcas[0]), orc.novelty_error(X, *pcas[1]), 0.75)
    np.testing.assert_allclose(got[0][0][rows * 1920 + cols], want, rtol=NOVELTY_RTOL, atol=0)


def _config(name, k):
    g = GoldenSeq(name)
    cfg = dict(g.config)
    cfg["params"] = dict(g.params, n_components=k)
    return g, cfg


def _add_models(m, g):
    poly = polygons()[g.meta["video"]]
    pts, ronis = poly["pts"][0], poly["bboxes_roni"][0]
    for s in range(g.n_models):
        fn = g.model_frames()[s]
        m.addModel(frame=g.frames[fn], poly_roi=pts[s], bbox=cv.boundingRect(np.array(pts[s])), bbox_roni=ronis[s], n_frame=fn)


def _port(name, k):
    from pcm.providers import make_segment_provider
    from ref_port import RefPortMasker
    g, cfg = _config(name, k)
    poly = polygons()[g.meta["video"]]
    ref = RefPortMasker(debug=False, frame=g.frames[0], config=cfg, poly_roi=poly["pts"][0][0],
                        segment_fn=make_segment_provider(g.meta["segments"]))
    _add_models(ref, g)
    return g, cfg, ref


@pytest.mark.parametrize("name", ["parachute_novelty", "frog_sweep"])
def test_addmodel_gpu_pca_with_three_components_matches_sklearn(name):
    """addModel(n_components=3) with the GPU trainer: mean, components and the 90th-percentile threshold equal
    scikit-learn's PCA(n_components=3) fitted on the same rows (the CPU port trains it)."""
    from maskers import getMaskerByName
    g, cfg, ref = _port(name, 3)
    m = getMaskerByName("PC", debug=False, frame=g.frames[0], config=cfg, poly_roi=None, update_mask=False, train_provider="gpu")
    _add_models(m, g)
    for s in range(g.n_models):
        got, want = m.novelty_det[s]["model"], ref.novelty_det[s]["model"]
        assert got.n_components == 3 and got.components_.shape == want.components_.shape
        np.testing.assert_allclose(got.mean_, want.mean_, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(got.components_, want.components_, rtol=1e-7, atol=1e-9)
        np.testing.assert_allclose(m.novelty_det[s]["threshold"], ref.novelty_det[s]["threshold"], rtol=1e-8)
    m.close()


# sampled frames of these sequences, trained with n_components = 3, where a label's score (the port's) lies within 1e-4
# of 0.5: there the float tolerance of the novelty error may decide the label
NEAR_HALF = {"parachute_novelty": [], "frog_sweep": [186]}


@pytest.mark.parametrize("provider", ["gpu", "sklearn"])
@pytest.mark.parametrize("name", ["parachute_novelty", "frog_sweep"])
def test_sequence_with_three_components_matches_the_port(name, provider):
    """The product masker and the CPU port (scikit-learn's inverse_transform), both trained with n_components = 3, over
    the sampled frames of the golden sequence: same return protocol, mask bytes and IoU counts on every frame except
    the frames of NEAR_HALF, where every label farther than 1e-4 from 0.5 must still get the port's decision."""
    from maskers import getMaskerByName
    from pcm.providers import make_segment_provider
    g, cfg, ref = _port(name, 3)
    m = getMaskerByName("PC", debug=False, frame=g.frames[0], config=cfg, poly_roi=None, update_mask=False,
                        segment_fn=make_segment_provider(g.meta["segments"]), train_provider=provider)
    _add_models(m, g)
    near = []
    for i in g.sample_frames():
        ref.index, ref.current_model = g.state_at(i)
        m.index, m.current_model = g.state_at(i)
        bbox = tuple(int(v) for v in g.z["bbox"][i])
        want_mask, mask = np.zeros_like(g.frames[i]), np.zeros_like(g.frames[i])
        want_ret = ref.update(bbox=bbox, frame=g.frames[i], mask=want_mask)
        ret = m.update(bbox=bbox, frame=g.frames[i], mask=mask, color=(0, 0, 255))
        assert ret == want_ret, "return protocol, frame %d" % i
        ref_scores = ref.last["scores"].astype(np.float64)
        far = np.abs(ref_scores - 0.5) >= 1e-4
        if not far.all():
            near.append(i)
            got = m.native.debug_scores(len(ref_scores))["scores"].astype(np.float64)
            assert np.array_equal(got[far] > 0.5, ref_scores[far] > 0.5), "decisions differ at frame %d" % i
            continue
        assert sha1(mask[:, :, 2]) == sha1(want_mask[:, :, 2]), "mask differs at frame %d" % i
        tg = cv.cvtColor(g.truth[i], cv.COLOR_BGR2GRAY)
        assert m.native.iou_counts(mask[:, :, 2], tg) == orc.iou_counts(want_mask[:, :, 2], tg)
    assert near == NEAR_HALF[name]
    m.close()


def test_clip_resident_sequence_with_three_components():
    """pcm.fastseq (device-resident clip, asynchronous frames) equals pcm.sequence.run_sequence with n_components = 3."""
    from pcm import fastseq, sweep
    from pcm.sequence import run_sequence
    with open(os.path.join(PKG, "config_benchmark.yaml")) as f:
        base = yaml.full_load(f)
    base["tracker_provider"] = "truth"
    params = dict(n_estimators=20, max_depth=7, n_components=3, novelty_detection=True, over_segmentation="quickshift",
                  features="6 lab", dilation_kernel=7, prior_weight=0.0)
    cfg = sweep.sequence_config(base, polygons(), "worm", params, "Input/SegTrack2/Video", "Input/SegTrack2/Truth")
    n = 40
    want = run_sequence(cfg, max_frames=n)
    clip = fastseq.ClipContext(cfg["input_video"], cfg["input_truth"], 1, 0, max_frames=n)
    got = fastseq.run_sequence_fast(cfg, clip)
    clip.close()
    assert got["n_frames"] == want["n_frames"] == n
    assert np.array_equal(np.asarray(got["iou"]), np.asarray(want["iou"]), equal_nan=True)


_PDL_SCRIPT = r'''
import hashlib, os, sys
sys.path[:0] = [%r, %r, %r]
import numpy as np, torch
from pcm import capi
from pcm.providers import voronoi_segments
from test_gpu_parity import _random_forest_arrays
rng = np.random.default_rng(6)
H, W, n, spaces = 360, 640, 8, ["hsv", "lab"]
F = 3 * (1 + 8 * n) * len(spaces)
frames = rng.integers(0, 256, (6, H, W, 3), dtype=np.uint8)
truth = (rng.random((6, H, W)) < 0.3).astype(np.uint8) * 255
h = capi.Handle(0)
h.set_features(n, spaces)
for m, nf in enumerate((0, 9)):
    h.add_model_arrays(nf, _random_forest_arrays(rng, 20, 5, F))
    q, _ = np.linalg.qr(rng.normal(size=(F, 3)))
    h.set_novelty(m, rng.random(F), np.ascontiguousarray(q.T))
rect = (0, 0, W, H)
seg = voronoi_segments(frames[0], 300, 1)
S = int(seg.max()) + 1
dev = torch.device("cuda", 0)
d_frames, d_truth, d_seg = torch.from_numpy(frames).to(dev), torch.from_numpy(truth).to(dev), torch.from_numpy(seg).to(dev)
d_mask = torch.zeros((H, W), dtype=torch.uint8, device=dev)
d_counts = torch.zeros((60, 2), dtype=torch.int64, device=dev)
torch.cuda.synchronize()
if os.environ.get("PCM_TEST_STREAM", "torch") != "own":
    h.set_stream(torch.cuda.current_stream().cuda_stream)
digest = hashlib.sha1()
for s in range(60):                      # back to back, no synchronisation between frames
    f = s %% 6
    prm = capi.Handle.make_params(0, 1, 1 - s / 60, s / 60, novelty=True, dilation_kernel=7, outlier_threshold=4.0)
    h.update_device(d_frames[f].data_ptr(), H, W, W * 3, rect, d_seg.data_ptr(), S, 0, prm, d_mask.data_ptr(), W)
    h.iou_device(d_mask.data_ptr(), W, d_truth[f].data_ptr(), W, 1, H, W, d_counts[s].data_ptr())
    if s %% 7 == 0:
        h.synchronize()
        digest.update(d_mask.cpu().numpy().tobytes())
h.synchronize()
digest.update(d_counts.cpu().numpy().tobytes())
print("DIGEST", digest.hexdigest(), int(d_counts[:, 1].min()))
'''


def test_dependent_launch_chain_with_three_components():
    """60 back-to-back device-path frames with two blended rank-3 models (novelty kernel between K0 and K1): the same
    masks and IoU counts with PCM_PDL=0 and PCM_PDL=1, on a caller's stream and on the handle's own stream."""
    here = os.path.dirname(os.path.abspath(__file__))
    out = {}
    for pdl, mode in (("0", "torch"), ("1", "own"), ("1", "torch")):
        res = subprocess.run([sys.executable, "-c", _PDL_SCRIPT % (PKG, here, os.path.join(os.path.dirname(here), "oracle"))],
                             env=dict(os.environ, PCM_PDL=pdl, PCM_TEST_STREAM=mode), capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = [l for l in res.stdout.splitlines() if l.startswith("DIGEST")][0].split()
        out[(pdl, mode)] = line[1]
        assert int(line[2]) > 0, "empty union: the test frames must produce masks"
    assert len(set(out.values())) == 1, out


def test_component_limits():
    from maskers import getMaskerByName
    from pcm import capi
    h = capi.Handle(0)
    h.set_features(1, ["rgb"])
    h.add_model_arrays(0, _random_forest_arrays(np.random.default_rng(0), 2, 2, 27))
    with pytest.raises(capi.PcmError) as e:
        h.set_novelty(0, np.zeros(27), np.eye(9, 27))
    assert e.value.code == -4                                   # PCM_E_LIMIT
    with pytest.raises(capi.PcmError) as e:
        h.set_novelty(0, np.zeros(27), np.zeros((0, 27)))
    assert e.value.code == -1                                   # PCM_E_INVALID
    h.set_novelty(0, np.zeros(27), np.eye(8, 27))               # the limit itself is accepted
    h.close()
    g, cfg = _config("parachute_novelty", 0.95)
    m = getMaskerByName("PC", debug=False, frame=g.frames[0], config=cfg, poly_roi=None, update_mask=False)
    with pytest.raises(ValueError, match="between 1 and 8"):
        _add_models(m, g)
    assert m.models == [] and m.novelty_det == []
    m.close()


def test_pca_fits_of_different_widths_in_parallel_threads():
    """The sweep fits PCAs of several feature sets at once, one handle per thread: residual launches of different
    shared-memory sizes must not interfere (each launch is checked; every result equals the same fit done alone)."""
    import threading
    from pcm import capi, train
    rng = np.random.default_rng(12)
    jobs = []
    for i, (F, k) in enumerate([(147, 1), (390, 3), (1161, 8), (27, 2)]):
        X = rng.integers(-1, 256, (3000, F)).astype(np.int16)
        y = (rng.random(3000) < 0.5).astype(np.uint8)
        jobs.append((X, y, k, 1000 + i))
    alone = []
    for X, y, k, rid in jobs:
        h = capi.Handle(0)
        train.upload_rows(h, X, y, rid)
        pca, thr = train.fit_pca(h, rid, len(y), X.shape[1], k)
        alone.append((pca.components_.tobytes(), thr))
        h.close()
    errors, got = [], {}

    def run(j):
        X, y, k, rid = jobs[j]
        h = capi.Handle(0)
        try:
            train.upload_rows(h, X, y, rid + 100)
            for _ in range(15):
                pca, thr = train.fit_pca(h, rid + 100, len(y), X.shape[1], k)
            got[j] = (pca.components_.tobytes(), thr)
        except Exception as e:           # reported below
            errors.append(repr(e))
        finally:
            h.close()
    threads = [threading.Thread(target=run, args=(j,)) for j in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert [got[j] for j in range(len(jobs))] == alone
