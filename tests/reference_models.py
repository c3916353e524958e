"""Shared helpers for the trained-fixture-model parity tests (CPU oracle and CUDA path).

Fixtures under tests/golden/ are made by tests/golden/make_reference_fixtures.py from the
reference's own test data; the assertions restate tests/nn/test_inference.py:585-800."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def model_dir(name):
    """Path handed to the predictors: the config JSON inside the fixture model folder (the reference accepts "a model
    folder or a training job JSON file inside a model folder", inference.py:3166-3168)."""
    return os.path.join(GOLDEN, "models", name, "fixture_config.json")


def load_fixture_model(name):
    """-> (cfg, spec, weights, in_ch)"""
    from sleap_b200.nn import architectures as A
    from sleap_b200.nn.model import load_weights
    cfg_path = model_dir(name)
    cfg = json.load(open(cfg_path))
    spec = A.spec_from_config(cfg["model"])
    w = load_weights(os.path.dirname(cfg_path))
    first = next(v for k, v in w.items() if k.endswith("enc0_conv0"))
    return cfg, spec, w, int(first["kernel"].shape[2])


def frames(name):
    z = np.load(os.path.join(GOLDEN, f"frames_{name}.npz"))
    return z["images"], z["points_gt"]


def h5py_file(*parts):
    """A file of the reference's test data that h5py wrote, stored under tests/golden/h5py/ by its path in that data."""
    return os.path.join(GOLDEN, "h5py", *parts)


def labels_minimal_instance():
    """The reference's ``min_labels`` fixture (tests/fixtures/datasets.py:52-54: 1 frame, 2 instances, skeleton A-B),
    rebuilt from the committed frame + ground-truth points."""
    from sleap_b200.io.labels import Instance, LabeledFrame, Labels, Skeleton
    from sleap_b200.io.video import Video
    z = np.load(os.path.join(GOLDEN, "frames_minimal_instance.npz"))
    sk = Skeleton(["A", "B"], [("A", "B")])
    lfs = [LabeledFrame(0, int(fi), [Instance(p, sk) for p in pts]) for fi, pts in zip(z["frame_idx"], z["points_gt"])]
    lab = Labels(lfs, [json.loads(str(z["video_json"]))], [sk])
    lab.set_video(0, Video.from_numpy(z["images"]))
    return lab


def labels_tracks_2node():
    """Frame 0 of the reference's ``min_tracks_2node_labels`` fixture (tests/fixtures/datasets.py:94-97: clip.2node.slp,
    skeleton head-thorax, two tracked flies), rebuilt from the committed frame + ground-truth points."""
    from sleap_b200.io.labels import Instance, LabeledFrame, Labels, Skeleton
    from sleap_b200.io.video import Video
    z = np.load(os.path.join(GOLDEN, "frames_tracks_2node.npz"))
    sk = Skeleton(["head", "thorax"], [("head", "thorax")])
    lfs = [LabeledFrame(0, int(fi), [Instance(p, sk) for p in pts]) for fi, pts in zip(z["frame_idx"], z["points_gt"])]
    lab = Labels(lfs, [json.loads(str(z["video_json"]))], [sk])
    lab.set_video(0, Video.from_numpy(z["images"]))
    return lab
