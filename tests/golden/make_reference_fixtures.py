"""Generates the committed fixtures under tests/golden/ from the reference's own test data.

Run in the build container only (needs /root/reference; the GPU box does not have it):

    python tests/golden/make_reference_fixtures.py

Sources (all data files, no reference code is imported or copied):
  tests/data/models/*/best_model.h5 + training_config.json   (trained fixture models used by
      tests/nn/test_inference.py:585-800: test_single_instance_predictor, test_topdown_predictor_*,
      test_bottomup_predictor)
  tests/data/slp_hdf5/minimal_instance.slp, small_robot_minimal.slp  (ground-truth labels, fixtures
      min_labels / min_labels_robot, tests/fixtures/datasets.py:52-68)
  tests/data/json_format_v1/centered_pair_low_quality.mp4 frame 0, tests/data/videos/small_robot.mp4 frames

Outputs:
  models/<name>/fixture_config.json    the training config reduced to the keys the inference path reads
  models/<name>/best_model.npz         float32 weights {layer/param} read out of best_model.h5 (optimizer state dropped)
  frames_minimal_instance.npz, frames_robot.npz   uint8 frames + ground-truth points (frame, instance, node, xy)
  h5py/<path under tests/data>         files written by h5py, for the in-tree HDF5 reader and writer tests (H5PY_FILES)
"""
import json
import os
import shutil
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from sleap_b200.io import h5lite                      # noqa: E402
from sleap_b200.nn.model import load_weights_h5, save_weights_npz   # noqa: E402

REF = "/root/reference/tests/data"
MODELS = {
    "minimal_instance.bottomup": "minimal_instance.UNet.bottomup",
    "minimal_instance.centroid": "minimal_instance.UNet.centroid",
    "minimal_instance.centered_instance": "minimal_instance.UNet.centered_instance",
    "minimal_robot.single_instance": "minimal_robot.UNet.single_instance",
    "minimal_instance.centered_instance_with_scaling": "minimal_instance.UNet.centered_instance_with_scaling",
    "min_tracks_2node.bottomup_multiclass": "min_tracks_2node.UNet.bottomup_multiclass",
    "min_tracks_2node.topdown_multiclass": "min_tracks_2node.UNet.topdown_multiclass",
}


H5PY_FILES = ["slp_hdf5/minimal_instance.slp", "slp_hdf5/small_robot_minimal.slp", "slp_hdf5/dance.mp4.labels.slp",
              "models/minimal_robot.UNet.single_instance/best_model.h5"]


def copy_h5py_files():
    """Byte-for-byte copies, except that the data of every ``optimizer_weights`` dataset of a ``best_model.h5`` (the Adam
    state, 60 % of the file, which inference never reads) is overwritten with zeros so that the stored file compresses.
    The HDF5 structure, the model weights and every other byte stay as h5py wrote them."""
    for rel in H5PY_FILES:
        src, dst = os.path.join(REF, rel), os.path.join(HERE, "h5py", rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if not rel.endswith(".h5"):
            shutil.copyfile(src, dst)
            continue
        f = h5lite.File(src)
        r = f._r
        buf = bytearray(r.b)
        for _, ds in f["optimizer_weights"].visit_datasets():
            for t, _, p, _ in r.messages(ds._addr):
                if t == 0x08:                                  # data layout message, version 3, contiguous storage
                    assert r.b[p] == 3 and r.b[p + 1] == 1, rel
                    a, n = r.u64(p + 2), r.u64(p + 10)
                    buf[a:a + n] = bytes(n)
        with open(dst, "wb") as out:
            out.write(buf)


def reduced_config(cfg):
    sk = (cfg["data"]["labels"].get("skeletons") or [None])[0]
    return {"data": {"preprocessing": cfg["data"]["preprocessing"],
                     "instance_cropping": cfg["data"]["instance_cropping"],
                     "labels": {"skeletons": [sk] if sk else []}},
            "model": cfg["model"]}


def gt_points(slp_path):
    """(n_frames, n_instances, n_nodes, 2) float32 from the .slp tables (sleap/io/format/hdf5.py:231-330)."""
    f = h5lite.File(slp_path)
    frames, inst, pts = f["frames"].read(), f["instances"].read(), f["points"].read()
    out = []
    for fr in frames:
        rows = []
        for i in range(int(fr["instance_id_start"]), int(fr["instance_id_end"])):
            p = pts[int(inst[i]["point_id_start"]):int(inst[i]["point_id_end"])]
            xy = np.stack([p["x"], p["y"]], -1).astype(np.float32)
            xy[p["visible"] == 0] = np.nan
            rows.append(xy)
        out.append(np.stack(rows))
    return np.stack(out), [int(fr["frame_idx"]) for fr in frames], json.loads(f["videos_json"].read()[0])


def gt_tracks(slp_path, n_frames):
    """Track name of every instance of the first ``n_frames`` labeled frames (instances table column ``track``,
    ``tracks_json`` rows ``[spawned_on, name]``; sleap/io/format/hdf5.py:250-262)."""
    f = h5lite.File(slp_path)
    frames, inst = f["frames"].read(), f["instances"].read()
    names = [json.loads(t)[1] for t in f["tracks_json"].read()]
    out = []
    for fr in frames[:n_frames]:
        out.append([names[int(inst[i]["track"])] if int(inst[i]["track"]) >= 0 else "" for i in
                    range(int(fr["instance_id_start"]), int(fr["instance_id_end"]))])
    return out


def read_frames(path, idxs, grayscale):
    cap = cv2.VideoCapture(path)
    out = []
    for i in idxs:
        cap.set(cv2.CAP_PROP_POS_FRAMES, i)
        ok, fr = cap.read()
        assert ok, (path, i)
        fr = fr[..., ::-1]                            # MediaVideo(bgr=True) flips to RGB (sleap/io/video.py:420-438)
        out.append(fr[..., :1] if grayscale else fr)
    return np.ascontiguousarray(np.stack(out)).astype(np.uint8)


def main():
    for short, name in MODELS.items():
        src, dst = os.path.join(REF, "models", name), os.path.join(HERE, "models", short)
        os.makedirs(dst, exist_ok=True)
        cfg = json.load(open(os.path.join(src, "training_config.json")))
        json.dump(reduced_config(cfg), open(os.path.join(dst, "fixture_config.json"), "w"), indent=1, sort_keys=True)
        w = load_weights_h5(os.path.join(src, "best_model.h5"))
        save_weights_npz(os.path.join(dst, "best_model.npz"), w)

    pts, idxs, vid = gt_points(os.path.join(REF, "slp_hdf5", "minimal_instance.slp"))
    frames = read_frames(os.path.join(REF, "json_format_v1", "centered_pair_low_quality.mp4"), idxs, True)
    np.savez_compressed(os.path.join(HERE, "frames_minimal_instance.npz"), images=frames, points_gt=pts, frame_idx=np.asarray(idxs),
                        video_json=np.asarray(json.dumps(vid)))
    print("minimal_instance", frames.shape, pts.shape, idxs, vid)

    pts, idxs, vid = gt_points(os.path.join(REF, "slp_hdf5", "small_robot_minimal.slp"))
    gray = bool(vid["backend"].get("grayscale"))
    frames = read_frames(os.path.join(REF, "videos", "small_robot.mp4"), idxs, gray)
    np.savez_compressed(os.path.join(HERE, "frames_robot.npz"), images=frames, points_gt=pts, frame_idx=np.asarray(idxs),
                        video_json=np.asarray(json.dumps(vid)))
    print("robot", frames.shape, pts.shape, idxs, vid)

    # identity (multi-class) models: fixture min_tracks_2node_labels = tests/data/tracks/clip.2node.slp over clip.mp4
    # (tests/fixtures/datasets.py:94-97); the reference's predictor tests use labeled frame 0 only (test_inference.py:809-852)
    slp = os.path.join(REF, "tracks", "clip.2node.slp")
    f = h5lite.File(slp)
    fr0 = f["frames"].read()[:1]
    inst, ptab = f["instances"].read(), f["points"].read()
    rows = []
    for i in range(int(fr0[0]["instance_id_start"]), int(fr0[0]["instance_id_end"])):
        p = ptab[int(inst[i]["point_id_start"]):int(inst[i]["point_id_end"])]
        xy = np.stack([p["x"], p["y"]], -1).astype(np.float32)
        xy[p["visible"] == 0] = np.nan
        rows.append(xy)
    vid = json.loads(f["videos_json"].read()[0])
    idxs = [int(fr0[0]["frame_idx"])]
    gray = bool(vid["backend"].get("grayscale"))
    frames = read_frames(os.path.join(REF, "tracks", "clip.mp4"), idxs, gray)
    np.savez_compressed(os.path.join(HERE, "frames_tracks_2node.npz"), images=frames, points_gt=np.stack(rows)[None], frame_idx=np.asarray(idxs),
                        track_names=np.asarray(gt_tracks(slp, 1)), video_json=np.asarray(json.dumps(vid)))
    print("tracks_2node", frames.shape, np.stack(rows).shape, idxs, gt_tracks(slp, 1), vid)

    copy_h5py_files()


if __name__ == "__main__":
    main()
