"""`.slp` writer (SURVEY 8f row 3): the in-tree HDF5 writer must emit what h5py emits.  No HDF5 library exists here, so
the evidence is (1) byte-for-byte equality of the datatype / dataspace messages and the superblock prefix with files
written by h5py (the reference's own label fixtures), (2) structural equality of the object graph, and (3) a round
trip through the independent reader."""
import json
import os

import numpy as np
from numpy.testing import assert_array_equal

from sleap_b200.io import h5lite, h5write
from sleap_b200.io import labels as L

import reference_models as rm

GOLDEN = rm.h5py_file("slp_hdf5", "minimal_instance.slp")          # written by h5py


def _messages(path, name):
    f = h5lite.File(path)
    r = f._r
    addr = r.group_links(r.root_header)[name]
    return r, {t: r.b[p:p + sz] for t, fl, p, sz in r.messages(addr)}


def test_datatype_and_dataspace_messages_match_h5py_bytes():
    legacy_instance = np.dtype([(n, L.INSTANCE_DTYPE.fields[n][0]) for n in L.INSTANCE_DTYPE.names[:-1]])   # fixture predates tracking_score
    for name, dt in (("frames", L.FRAME_DTYPE), ("instances", legacy_instance), ("points", L.POINT_DTYPE),
                     ("pred_points", L.PRED_POINT_DTYPE)):
        r, msgs = _messages(GOLDEN, name)
        enc = h5write.encode_datatype(dt)
        assert msgs[0x0003][:len(enc)] == enc, name
        assert not any(msgs[0x0003][len(enc):]), name                      # only alignment padding follows
        n = h5lite.File(GOLDEN)[name].read().shape[0]
        assert msgs[0x0001][:24] == h5write.encode_dataspace((n,), unlimited=True)
    _, msgs = _messages(GOLDEN, "videos_json")
    assert msgs[0x0003][:8] == h5write.encode_datatype(np.dtype("S144"))
    _, msgs = _messages(GOLDEN, "suggestions_json")
    assert msgs[0x0003][:20] == h5write.encode_datatype(np.dtype("f8"))


def test_superblock_and_group_structures_match_h5py(tmp_path):
    p = str(tmp_path / "w.slp")
    with h5write.File(p) as f:
        g = f.create_group("metadata")
        g.attrs["format_id"] = np.float64(1.1)
        g.attrs["json"] = "{}"
        f.create_dataset("frames", np.zeros(3, L.FRAME_DTYPE))
    mine, ref = open(p, "rb").read(), open(GOLDEN, "rb").read()
    assert mine[:40] == ref[:40]                                            # signature, versions, sizes, K values, base address, free-space address
    assert mine[48:64] == ref[48:64]                                        # driver-info address + root link-name offset
    assert mine[72:80] == ref[72:80]                                        # root entry: cache type 1 (cached B-tree / heap addresses)
    assert int.from_bytes(mine[40:48], "little") == len(mine)               # end-of-file address
    r = h5lite.File(p)._r
    for t, fl, pos, sz in r.messages(r.root_header):
        assert t == 0x0011
        bt, hp = r.u64(pos), r.u64(pos + 8)
        assert r.b[bt:bt + 8] == b"TREE\x00\x00\x01\x00" and r.b[hp:hp + 8] == b"HEAP\x00\x00\x00\x00"
        assert r.u64(hp + 16) == 1                                           # H5HL_FREE_NULL
        snod = r.u64(bt + 32)
        assert r.b[snod:snod + 8] == b"SNOD\x01\x00\x02\x00"
    # the attribute message of format_id is what h5py wrote, bit for bit (same name, float64 scalar)
    gr = h5lite.File(GOLDEN)._r
    ga = gr.group_links(gr.root_header)["metadata"]
    gold_attr = [gr.b[pos:pos + sz] for t, fl, pos, sz in gr.messages(ga) if t == 0x000C][0]
    ma = r.group_links(r.root_header)["metadata"]
    my_attr = [r.b[pos:pos + sz] for t, fl, pos, sz in r.messages(ma) if t == 0x000C][0]
    assert my_attr == gold_attr


def test_labels_round_trip(tmp_path):
    lab = rm.labels_minimal_instance()
    sk = lab.skeleton
    pred = L.Instance(np.asarray([[10.5, 20.25], [np.nan, np.nan]], np.float32), sk, -1, 0.75, np.asarray([0.9, 0.0], np.float32), True)
    lab.labeled_frames.append(L.LabeledFrame(0, 7, [pred]))
    p = str(tmp_path / "out.slp")
    lab.save_file(p)
    back = L.Labels.load_file(p)
    assert len(back) == 2 and [lf.frame_idx for lf in back] == [0, 7]
    assert back.skeleton.node_names == sk.node_names and back.skeleton.edge_names == sk.edge_names
    assert back.video_specs == lab.video_specs
    for a, b in zip(lab[0].instances, back[0].instances):
        assert_array_equal(a.numpy(), b.numpy())
        assert not b.predicted
    q = back[1][0]
    assert q.predicted and abs(q.score - 0.75) < 1e-6
    assert_array_equal(np.isnan(q.numpy()), [[False, False], [True, True]])
    assert_array_equal(q.numpy()[0], [10.5, 20.25])
    assert abs(float(q.point_scores[0]) - 0.9) < 1e-6
    f = h5lite.File(p)
    assert abs(float(f["metadata"].attrs["format_id"]) - 1.2) < 1e-12
    meta = json.loads(f["metadata"].attrs["json"])
    assert meta["nodes"] == [{"name": "A", "weight": 1.0}, {"name": "B", "weight": 1.0}]
    assert f["instances"].read().dtype.names[-1] == "tracking_score"
    assert f["points"].read().dtype == np.dtype([("x", "<f8"), ("y", "<f8"), ("visible", "i1"), ("complete", "i1")])


def test_labels_from_predictions(tmp_path):
    from sleap_b200.nn.inference import LabeledFrame, PredictedInstance
    sk = L.Skeleton(["a", "b", "c"], [("a", "b"), ("b", "c")])
    frames = [LabeledFrame(0, 3, [PredictedInstance.from_numpy(np.asarray([[1, 2], [3, 4], [np.nan, np.nan]], np.float32),
                                                              np.asarray([0.5, 0.6, np.nan], np.float32), 1.1)]),
              LabeledFrame(0, 4, [])]
    lab = L.labels_from_predictions(frames, sk, video_filename="movie.mp4")
    p = str(tmp_path / "pred.slp")
    lab.save(p)
    back = L.Labels.load_file(p)
    assert [len(lf) for lf in back] == [1, 0] and back[0][0].predicted and back[0][0].n_visible_points == 2
    assert back.video_specs[0]["backend"]["filename"] == "movie.mp4" and back.skeleton.edge_inds == [(0, 1), (1, 2)]


def test_tracked_predictions_round_trip(tmp_path):
    """Tracker output -> Labels -> .slp -> Labels: track table ('[spawned_on,"name"]' rows) and per-instance track indices."""
    from sleap_b200.nn import tracking as T
    from sleap_b200.nn.inference import LabeledFrame, PredictedInstance
    shape = np.array([[-5.0, -5.0], [0.0, 0.0], [5.0, 5.0]])
    frames = [LabeledFrame(0, t, [PredictedInstance.from_numpy(shape + [[10.0 + t, 10.0]], [1, 1, 1], 1.0),
                                  PredictedInstance.from_numpy(shape + [[60.0 - t, 40.0]], [1, 1, 1], 2.0)]) for t in range(4)]
    T.run_tracker(frames, T.Tracker.make_tracker_by_name(tracker="simple"))
    lab = L.labels_from_predictions(frames, L.Skeleton(["a", "b", "c"], [("a", "b"), ("b", "c")]), video_filename="m.mp4")
    assert lab.tracks == [[0, "track_0"], [0, "track_1"]]
    p = str(tmp_path / "tracked.slp")
    lab.save(p)
    back = L.Labels.load_file(p)
    assert back.tracks == [[0, "track_0"], [0, "track_1"]]
    assert [[i.track for i in lf.instances] for lf in back] == [[0, 1]] * 4
    assert h5lite.File(p)["tracks_json"].read()[0] == b'[0,"track_0"]'


def test_tracking_score_and_legacy_format(tmp_path):
    """hdf5.py:143-155, 221-224: tracking_score is carried from format 1.2 on; user points of files older than format 1.1
    are shifted by -0.5 px on load (predicted points are not)."""
    sk = L.Skeleton(["a", "b"], [("a", "b")])
    user = L.Instance(np.asarray([[4.0, 5.0], [6.0, 7.0]], np.float32), sk)
    pred = L.Instance(np.asarray([[1.5, 2.5], [3.5, 4.5]], np.float32), sk, 0, 0.5, np.asarray([0.9, 0.8], np.float32), True,
                      tracking_score=0.625)
    lab = L.Labels([L.LabeledFrame(0, 0, [user, pred])], [{"backend": {"filename": "m.mp4"}}], [sk], [[0, "track_0"]])
    p = str(tmp_path / "ts.slp")
    lab.save(p)
    back = L.Labels.load_file(p)
    assert back[0][1].predicted and back[0][1].tracking_score == 0.625 and back[0][0].tracking_score == 0.0
    assert_array_equal(back[0][0].numpy(), user.numpy())
    # the same tables under a pre-1.1 format id: user points shift, predicted points and tracking_score do not survive
    f = h5lite.File(p)
    q = str(tmp_path / "old.slp")
    with h5write.File(q) as w:
        g = w.create_group("metadata")
        g.attrs["format_id"] = np.float64(1.0)
        g.attrs["json"] = f["metadata"].attrs["json"]
        for name in ("videos_json", "tracks_json", "suggestions_json", "frames", "instances", "points", "pred_points"):
            w.create_dataset(name, f[name].read())
    old = L.Labels.load_file(q)
    assert_array_equal(old[0][0].numpy(), user.numpy() - np.float32(0.5))
    assert_array_equal(old[0][1].numpy(), pred.numpy())
    assert old[0][1].tracking_score == 0.0
