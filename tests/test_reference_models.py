"""Pins the conv-network oracle (and the whole CPU restatement) to the reference's OWN predictor tests:
trained fixture models + real frames + ground-truth labels, same assertions and tolerances as
tests/nn/test_inference.py (test_single_instance_predictor :585-610, test_topdown_predictor_centroid :638-656,
test_topdown_predictor_centered_instance-style matching :728-757, test_bottomup_predictor :770-800).
Also exercises the in-tree HDF5 reader on the committed Keras .h5 / .slp files."""
import os

import numpy as np
from numpy.testing import assert_allclose

from oracle import inference as oinf
import reference_models as rm


def _matched(points_gt, points_pr, atol):
    i1, i2 = oinf.match_points(points_gt, points_pr)
    assert len(i1) == len(points_gt)
    assert_allclose(points_gt[i1], points_pr[i2], atol=atol)


REF_H5 = rm.h5py_file("models", "minimal_robot.UNet.single_instance", "best_model.h5")
REF_SLP = rm.h5py_file("slp_hdf5", "minimal_instance.slp")


def test_h5_reader_keras_weights_match_npz_export():
    """The in-tree HDF5 reader on a Keras ``best_model.h5`` written by h5py: every array equals the committed ``.npz``."""
    from sleap_b200.io import h5lite
    from sleap_b200.nn.model import load_weights_h5, load_weights_npz
    f = h5lite.File(REF_H5)
    assert set(f.keys()) >= {"model_weights"}
    assert f.attrs["backend"] == "tensorflow"
    w = load_weights_h5(REF_H5)
    assert w["stack0_enc0_conv0"]["kernel"].shape[:2] == (3, 3)
    assert "SingleInstanceConfmapsHead" in w
    n = sum(a.size for p in w.values() for a in p.values())
    from sleap_b200.nn import architectures as A
    _, spec, wz, in_ch = rm.load_fixture_model("minimal_robot.single_instance")
    assert n == A.count_params(A.compile_model(spec, in_ch))
    for layer, params in w.items():
        for k, a in params.items():
            np.testing.assert_array_equal(a, wz[layer][k])


def test_h5_reader_slp_tables():
    from sleap_b200.io import h5lite
    f = h5lite.File(REF_SLP)
    assert sorted(f.keys()) == ["frames", "instances", "metadata", "points", "pred_points", "suggestions_json",
                                "tracks_json", "videos_json"]
    pts = f["points"].read()
    assert pts.dtype.names == ("x", "y", "visible", "complete") and len(pts) == 4
    assert_allclose([pts["x"][0], pts["y"][0]], [92.65220773, 202.72597774], rtol=1e-9)
    inst = f["instances"].read()
    assert list(inst["point_id_end"]) == [2, 4]
    assert f["metadata"].attrs["format_id"] == 1.1 or str(f["metadata"].attrs["format_id"]).startswith("1.1")
    _, gt = rm.frames("minimal_instance")
    assert_allclose(gt[0, 0, 0], [pts["x"][0], pts["y"][0]], rtol=1e-6)
    g = h5lite.File(rm.h5py_file("slp_hdf5", "dance.mp4.labels.slp"))          # chunked tables, 450 frames of predictions
    assert g["frames"].read().shape == (450,) and g["pred_points"].read().shape == (7650,)
    assert g["instances"].read().dtype.names[-1] == "tracking_score"


def test_oracle_bottomup_on_trained_model():
    """test_bottomup_predictor: 1 frame, 2 instances, matched points within 1.75 px of the labels."""
    cfg, spec, w, in_ch = rm.load_fixture_model("minimal_instance.bottomup")
    imgs, gt = rm.frames("minimal_instance")
    pre = cfg["data"]["preprocessing"]
    out = oinf.bottomup_layer(imgs, spec, w, in_ch, pre["input_scaling"], spec["backbone_cfg"]["max_stride"])
    assert len(out["instance_peaks"][0]) == 2
    _matched(gt[0].reshape(-1, 2), out["instance_peaks"][0].reshape(-1, 2), 1.75)
    hi = oinf.bottomup_layer(imgs, spec, w, in_ch, pre["input_scaling"], spec["backbone_cfg"]["max_stride"],
                             min_line_scores=1.1)
    assert len(hi["instance_peaks"][0]) == 0


def test_oracle_topdown_on_trained_models():
    """test_topdown_predictor_centroid (:638-656, atol 1.5 on centroid-only instances) and the full
    centroid -> centered-instance chain (atol 1.5 as :757)."""
    ccfg, cspec, cw, cin = rm.load_fixture_model("minimal_instance.centroid")
    icfg, ispec, iw, iin = rm.load_fixture_model("minimal_instance.centered_instance")
    imgs, gt = rm.frames("minimal_instance")
    crop = icfg["data"]["instance_cropping"]["crop_size"]
    out = oinf.topdown_model(imgs, cspec, cw, ispec, iw, crop, cin, iin,
                             ccfg["data"]["preprocessing"]["input_scaling"], icfg["data"]["preprocessing"]["input_scaling"],
                             cspec["backbone_cfg"]["max_stride"], ispec["backbone_cfg"]["max_stride"])
    assert len(out["instance_peaks"][0]) == 2
    # full predicted chain: the reference has no test of this model pair against the labels (its centroid-only /
    # instance-only tests stand in ground truth for the other stage); 2 px is our own sanity bound
    _matched(gt[0].reshape(-1, 2), out["instance_peaks"][0].reshape(-1, 2), 2.0)
    # centroid stage alone vs the labels' bounding-box midpoints (instance_centroids.py:12-33, anchor_part=None)
    cent_gt = np.stack([(g.min(0) + g.max(0)) * 0.5 for g in gt[0]]).astype(np.float32)
    _matched(cent_gt, out["centroids"][0], 1.5)
    # test_topdown_predictor_centered_instance (:728-757): crops at the GROUND-TRUTH centroids
    # (CentroidCropGroundTruth, inference.py:743-809), instance peaks within 1.5 px of the labels
    from oracle import tf_ops
    crops = tf_ops.crop_bboxes(imgs, tf_ops.make_centered_bboxes(cent_gt, crop, crop), np.zeros(2, np.int32))
    pts, _ = oinf.find_instance_peaks_layer(crops, (cent_gt - np.float32(crop / 2)).astype(np.float32), ispec, iw, iin,
                                            1.0, ispec["backbone_cfg"]["max_stride"])
    _matched(gt[0].reshape(-1, 2), pts.reshape(-1, 2), 1.5)
    for k in (1, 2, 3):                                     # test_topdown_predictor_centroid_max_instances :659-671
        o = oinf.topdown_model(imgs, cspec, cw, ispec, iw, crop, cin, iin, 1.0, 1.0, 8, 8, max_instances=k)
        assert len(o["instance_peaks"][0]) == min(k, 2)
    hi = oinf.topdown_model(imgs, cspec, cw, ispec, iw, crop, cin, iin, 1.0, 1.0, 8, 8, peak_threshold=1.5)
    assert len(hi["instance_peaks"][0]) == 0                # :674-683


def test_oracle_single_instance_on_trained_model():
    """test_single_instance_predictor (:585-610): 2 frames, 1 instance each, atol 10 px;
    _high_peak_thresh (:613-635): threshold 0 -> 2 visible points, 1.5 -> none."""
    cfg, spec, w, in_ch = rm.load_fixture_model("minimal_robot.single_instance")
    imgs, gt = rm.frames("robot")
    pre = cfg["data"]["preprocessing"]
    out = oinf.single_instance_layer(imgs, spec, w, in_ch, pre["input_scaling"], spec["backbone_cfg"]["max_stride"],
                                     peak_threshold=0.2)
    assert out["instance_peaks"].shape == (2, 1, 2, 2)
    assert_allclose(out["instance_peaks"][:, 0], gt[:, 0], atol=10.0)
    lo = oinf.single_instance_layer(imgs, spec, w, in_ch, pre["input_scaling"], 4, peak_threshold=0.0)
    assert not np.isnan(lo["instance_peaks"]).any()
    hi = oinf.single_instance_layer(imgs, spec, w, in_ch, pre["input_scaling"], 4, peak_threshold=1.5)
    assert np.isnan(hi["instance_peaks"]).all()


def test_oracle_centered_instance_with_scaling():
    """test_topdown_predictor_centered_instance_with_scaling (:708-729): instance model trained at input_scaling 0.5,
    crops of 56 px cut at the ground-truth centroids from the half-size frame (CentroidCropGroundTruth.input_scale),
    FindInstancePeaks with resize_input_image=False; matched points within 1.5 px of the labels."""
    cfg, spec, w, in_ch = rm.load_fixture_model("minimal_instance.centered_instance_with_scaling")
    imgs, gt = rm.frames("minimal_instance")
    scale = cfg["data"]["preprocessing"]["input_scaling"]
    crop = cfg["data"]["instance_cropping"]["crop_size"]
    assert scale == 0.5 and crop == 56
    cent_gt = np.stack([(g.min(0) + g.max(0)) * 0.5 for g in gt[0]]).astype(np.float32)
    cc = oinf.centroid_crop_ground_truth_layer(imgs, [cent_gt], crop, input_scale=scale)
    assert cc["crops"].shape == (2, 56, 56, 1) and cc["crops"].dtype == np.uint8
    pts, vals = oinf.find_instance_peaks_layer(cc["crops"], cc["crop_offsets"], spec, w, in_ch, input_scale=scale, pad_stride=1,
                                               resize_input_image=False)
    _matched(gt[0].reshape(-1, 2), pts.reshape(-1, 2), 1.5)


def test_bottomup_multiclass_oracle():
    """tests/nn/test_inference.py:809-852 (test_bottomup_multiclass_predictor / _high_threshold) on the CPU restatement:
    the reference's trained identity model (confidence maps + sigmoid class maps), frame 0 of its ``min_tracks_2node``
    labels; two instances, each on the track of its class, points within 2 % of the ground truth."""
    from oracle import convnet, peak_finding as opf, preprocess as opre
    from sleap_b200.nn import identity
    cfg, spec, w, in_ch = rm.load_fixture_model("min_tracks_2node.bottomup_multiclass")
    assert spec["head_type"] == "multi_class_bottomup" and spec["classes"] == ["female", "male"]
    z = np.load(os.path.join(rm.GOLDEN, "frames_tracks_2node.npz"))
    imgs, gt, names = z["images"], z["points_gt"][0], [str(n) for n in z["track_names"][0]]
    scale = float(cfg["data"]["preprocessing"]["input_scaling"])
    x = opre.preprocess(imgs, ensure_gray=(in_ch == 1), input_scale=scale, pad_stride=spec["backbone_cfg"]["max_stride"])
    cms, cls = convnet.model_forward(x, spec, w)
    with np.errstate(over="ignore"):
        cls = (1.0 / (1.0 + np.exp(-cls))).astype(np.float32)
    cs, ks = spec["heads"][0]["output_stride"], spec["heads"][1]["output_stride"]
    for thr, want in ((0.7, 2), (1.5, 0)):
        p, v, si, ci = opf.find_local_peaks(cms, thr, "local", 5)
        p = ((p * np.float32(cs)).astype(np.float32) / np.float32(ks)).astype(np.float32)
        pts, pv, pr = identity.classify_peaks_from_maps(cls, p, v, si, ci, n_channels=cms.shape[3])
        pts = (pts * np.float32(ks)) / np.float32(scale) + np.float32(0.5)
        found = [j for j in range(pts.shape[1]) if not np.isnan(pts[0, j]).all()]
        assert len(found) == want
        for j in found:
            assert_allclose(pts[0, j], gt[names.index(spec["classes"][j])], rtol=0.02)


def test_topdown_multiclass_oracle():
    """tests/nn/test_inference.py:855-894 (test_topdown_multiclass_predictor / _high_threshold) on the CPU restatement:
    ground-truth centroids (anchor part thorax) -> 128-px crops -> the reference's trained centered-instance + class-vector
    model (ClassVectorsHead = global max pool + 3 x Dense(64) + softmax on the stride-16 encoder output) -> global peaks ->
    classify_peaks_from_vectors; both flies on the track of their class, points within 2 % of the ground truth."""
    from oracle import convnet, peak_finding as opf, preprocess as opre
    from sleap_b200.nn import identity
    cfg, spec, w, in_ch = rm.load_fixture_model("min_tracks_2node.topdown_multiclass")
    assert spec["head_type"] == "multi_class_topdown" and spec["classes"] == ["female", "male"]
    assert spec["heads"][1]["vector"] and spec["heads"][1]["num_fc_layers"] == 3 and spec["heads"][1]["output_stride"] == 16
    z = np.load(os.path.join(rm.GOLDEN, "frames_tracks_2node.npz"))
    imgs, gt, names = z["images"], z["points_gt"][0], [str(n) for n in z["track_names"][0]]
    crop = cfg["data"]["instance_cropping"]["crop_size"]
    cc = oinf.centroid_crop_ground_truth_layer(imgs, [gt[:, 1, :]], crop, 1.0)          # anchor = thorax = node 1
    x = opre.preprocess(cc["crops"], ensure_gray=(in_ch == 1), input_scale=1.0, pad_stride=spec["backbone_cfg"]["max_stride"])
    cms, probs = convnet.model_forward(x, spec, w)
    assert probs.shape == (2, 2) and np.allclose(probs.sum(1), 1.0, atol=1e-6)
    for thr, want in ((0.7, 2), (1.5, 0)):
        pts, vals = opf.find_global_peaks(cms, thr, "local", 5)
        pts = (pts * np.float32(spec["heads"][0]["output_stride"]) + cc["crop_offsets"][:, None, :]).astype(np.float32)
        P, V, C = identity.classify_peaks_from_vectors(pts, vals, probs, cc["crop_sample_inds"], 1)
        found = [j for j in range(P.shape[1]) if not np.isnan(P[0, j]).all()]
        assert len(found) == want
        for j in found:
            assert_allclose(P[0, j], gt[names.index(spec["classes"][j])], rtol=0.02)
            assert C[0, j] > 0.99
