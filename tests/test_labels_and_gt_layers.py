"""Caller side of the path (SURVEY 8f): ``.slp`` labels -> LabelsReader examples -> ground-truth stand-in layers
of the top-down model (sleap/nn/inference.py:723-893).  Host logic only; no GPU."""
import os

import numpy as np
from numpy.testing import assert_allclose

from sleap_b200.io.labels import Labels, LabelsReader, Skeleton, find_instance_centroids, find_points_bbox_midpoint
from sleap_b200.io.video import Video
from sleap_b200.nn.inference import FindInstancePeaksGroundTruth

import reference_models as rm

REF_SLP = rm.h5py_file("slp_hdf5", "minimal_instance.slp")


def _labels():
    z = np.load(os.path.join(rm.GOLDEN, "frames_minimal_instance.npz"))
    return rm.labels_minimal_instance(), z


def test_labels_load_file():
    lab = Labels.load_file(REF_SLP)
    z = np.load(os.path.join(rm.GOLDEN, "frames_minimal_instance.npz"))
    assert len(lab) == 1 and len(lab[0]) == 2 and lab[0].frame_idx == 0
    assert lab.skeleton.node_names == ["A", "B"] and lab.skeleton.edge_names == [("A", "B")] and lab.skeleton.edge_inds == [(0, 1)]
    assert lab.video_specs[0]["backend"]["grayscale"] is True
    assert_allclose(np.stack([i.numpy() for i in lab[0].instances]), z["points_gt"][0], rtol=1e-6)
    assert lab[0][0].n_visible_points == 2 and not lab[0][0].predicted
    robot = Labels.load_file(rm.h5py_file("slp_hdf5", "small_robot_minimal.slp"))
    assert [lf.frame_idx for lf in robot] == [0, 79] and len(robot[1]) == 1
    dance = Labels.load_file(rm.h5py_file("slp_hdf5", "dance.mp4.labels.slp"))
    assert len(dance) == 450 and len(dance.skeleton) == 17 and len(dance.skeleton.edge_names) == 15
    assert sum(len(lf.predicted_instances) for lf in dance) == 450 and sum(len(lf.user_instances) for lf in dance) == 3
    # the rebuilt fixture used by the GPU tests equals what the file holds
    mine = rm.labels_minimal_instance()
    assert_allclose(np.stack([i.numpy() for i in mine[0].instances]), np.stack([i.numpy() for i in lab[0].instances]))
    assert mine.video_specs == lab.video_specs and mine.skeleton.edge_names == lab.skeleton.edge_names


def test_skeleton_from_jsonpickle_backrefs():
    """Edge types after the first are ``{"py/id": k}`` back-references; type 2 = symmetry is not a body edge."""
    nodes = [{"name": n, "weight": 1.0} for n in "abcd"]
    sk = {"graph": {"name": "S"}, "nodes": [{"id": 2}, {"id": 0}, {"id": 1}, {"id": 3}],
          "links": [{"edge_insert_idx": 1, "source": 0, "target": 1, "type": {"py/id": 1}},
                    {"edge_insert_idx": 0, "source": 2, "target": 0, "type": {"py/reduce": [{"py/type": "sleap.skeleton.EdgeType"}, {"py/tuple": [1]}]}},
                    {"edge_insert_idx": 2, "source": 1, "target": 3, "type": {"py/reduce": [{"py/type": "sleap.skeleton.EdgeType"}, {"py/tuple": [2]}]}},
                    {"edge_insert_idx": 3, "source": 3, "target": 1, "type": {"py/id": 2}}]}
    s = Skeleton.from_dict(sk, nodes)
    assert s.node_names == ["c", "a", "b", "d"]
    assert s.edge_names == [("c", "a"), ("a", "b")] and s.symmetry_names == [("b", "d"), ("d", "b")]


def test_centroids():
    pts = np.asarray([[[0, 0], [4, 2]], [[1, 1], [np.nan, np.nan]]], np.float32)
    assert_allclose(find_points_bbox_midpoint(pts), [[2, 1], [1, 1]])                 # instance_centroids.py:12-33
    assert_allclose(find_instance_centroids(pts, anchor_ind=1), [[4, 2], [1, 1]])     # anchor where visible, else midpoint


def test_labels_reader_examples():
    lab, z = _labels()
    r = LabelsReader(lab, with_centroids=True)
    ex = list(r)
    assert len(r) == 1 and set(r.output_keys) <= set(ex[0])
    assert ex[0]["image"].shape == (384, 384, 1) and ex[0]["instances"].shape == (2, 2, 2)
    assert_allclose(ex[0]["centroids"], (z["points_gt"][0].min(1) + z["points_gt"][0].max(1)) / 2, rtol=1e-6)
    assert int(ex[0]["frame_ind"]) == 0 and ex[0]["scale"].tolist() == [1.0, 1.0]


def test_find_instance_peaks_ground_truth():
    """tests/nn/test_inference.py:120-166: every centroid gets the ground-truth instance with the closest node."""
    inst = [np.asarray([[[0, 1], [2, 3]], [[10, 11], [12, 13]]], np.float32), np.asarray([[[5, 5], [6, 6]]], np.float32),
            np.zeros((0, 2, 2), np.float32)]
    cents = [np.asarray([[11.5, 12.5], [1, 2]], np.float32), np.asarray([[100, 100]], np.float32), np.zeros((0, 2), np.float32)]
    out = FindInstancePeaksGroundTruth().call({"instances": inst}, {"centroids": cents, "centroid_vals": [np.ones(2), np.ones(1), np.ones(0)]})
    assert_allclose(out["instance_peaks"][0], inst[0][[1, 0]])
    assert_allclose(out["instance_peaks"][1], inst[1])
    assert out["instance_peaks"][2].shape == (0, 2, 2) and out["instance_peak_vals"][0].shape == (2, 2)
    assert np.all(out["instance_peak_vals"][0] == 1)


def test_find_instance_peaks_ground_truth_nans():
    """tests/nn/test_inference.py:168-209: ground-truth instances with missing nodes still match."""
    nan = np.nan
    inst = [np.asarray([[[0, 0], [0, 0]], [[1, 1], [1, 1]]], np.float32), np.asarray([[[0, 0], [nan, nan]], [[1, 1], [nan, nan]]], np.float32)]
    cents = [np.asarray([[0, 0], [1, 1]], np.float32)] * 2
    out = FindInstancePeaksGroundTruth().call({"instances": inst}, {"centroids": cents, "centroid_vals": [np.ones(2)] * 2})
    assert [p.shape for p in out["instance_peaks"]] == [(2, 2, 2), (2, 2, 2)]
    assert_allclose(out["instance_peaks"][1][:, 0], [[0, 0], [1, 1]])
    allnan = [np.full((1, 2, 2), nan, np.float32)]
    out = FindInstancePeaksGroundTruth().call({"instances": allnan}, {"centroids": [np.zeros((1, 2), np.float32)], "centroid_vals": [np.ones(1)]})
    assert out["instance_peaks"][0].shape == (0, 2, 2)
