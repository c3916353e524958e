"""Record exchange over peer memory (sb_gather_*, SURVEY 8e): the grouping kernel's epilogue stores each frame's record into
every rank's gather window.  (a) world = 1 in process: the window of a rank is its own memory, so push / arrival words /
generations / acknowledgement flow control run on a single GPU; (b) world = 2 under torchrun when two GPUs are visible:
every rank must see exactly the records an NCCL all-gather of the same device records delivers."""
import os
import subprocess
import sys

import numpy as np
import pytest
from numpy.testing import assert_array_equal

from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _predictor(batch_size=3, seed=31):
    from sleap_b200.nn import architectures as A
    from sleap_b200.nn.inference import BottomUpPredictor
    from sleap_b200.nn.model import DeviceModel
    spec = dict(backbone="unet", head_type="multi_instance", part_names=synth.FLIES13_NODES, edges=synth.FLIES13_EDGES,
                backbone_cfg=dict(filters=16, filters_rate=2, max_stride=16, output_stride=4, middle_block=True, up_interpolate=False),
                heads=[dict(name="MultiInstanceConfmapsHead", channels=13, output_stride=4),
                       dict(name="PartAffinityFieldsHead", channels=24, output_stride=8)])
    w = A.make_synthetic_weights(A.compile_model(spec, 1), seed)
    model = DeviceModel(spec, w, input_channels=1, precision=0)
    imgs = np.random.default_rng(seed).integers(0, 256, size=(2, 128, 128, 1), dtype=np.uint8)
    thr = float(np.quantile(model.forward(imgs)[0], 0.998))
    pred = BottomUpPredictor(model, synth.FLIES13_NODES, synth.FLIES13_EDGES, peak_threshold=thr, batch_size=batch_size,
                             max_peaks_per_sample=2048, max_node_peaks=32, max_instances_per_frame=16, min_line_scores=-100.0)
    return model, pred


def _records_of(out, I, C):
    import torch
    from sleap_b200 import parallel
    pad = lambda a: np.pad(a, [(0, 0), (0, I - a.shape[1])] + [(0, 0)] * (a.ndim - 2), constant_values=np.nan)
    return parallel.pack_records(torch.from_numpy(pad(out["instance_peaks"])), torch.from_numpy(pad(out["instance_peak_vals"])),
                                 torch.from_numpy(pad(out["instance_scores"])), torch.from_numpy(out["n_valid"]),
                                 torch.from_numpy(out["flags"])).numpy()


@pytest.mark.filterwarnings("ignore:device capacity reached")
def test_single_rank_window_roundtrip_and_flow_control():
    from sleap_b200 import parallel
    model, pred = _predictor()
    frames = np.random.default_rng(3).integers(0, 256, size=(3 * 11, 128, 128, 1), dtype=np.uint8)
    want = pred.predict(frames, make_labels=False)                         # no exchange yet
    pg = parallel.PeerGather(model, generations=4)                         # 11 steps through 4 generations: acks are needed
    got = pred.predict(frames, make_labels=False)
    assert pg.pushed() == 11 and pg.consumed == 11
    I, C = 16, 13
    for g, x in zip(got, want):
        assert_array_equal(g["n_valid"], x["n_valid"])
        assert list(g["gathered_counts"]) == [3]
        rec = g["gathered_records"]
        assert rec.shape == (3, parallel.record_width(I, C))
        assert_array_equal(np.nan_to_num(rec, nan=-7.0), np.nan_to_num(_records_of(x, I, C), nan=-7.0))
    # the synchronous entry is an exchange step as well
    one = pred.inference_model.predict_on_batch(frames[:2])
    assert one["gathered_records"].shape[0] == 2 and list(one["gathered_counts"]) == [2]
    pg.close()
    again = pred.predict(frames[:6], make_labels=False)
    assert "gathered_records" not in again[0]


def test_two_ranks_match_nccl_all_gather():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29731", os.path.join(ROOT, "tools", "gather_check.py")], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "GATHER_CHECK_OK" in r.stdout
