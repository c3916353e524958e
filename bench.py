#!/usr/bin/env python
"""Benchmark of the north-star path: bottom-up UNet+PAF pose inference on 1024x1024x1 frames
(BASELINE.json config C4: 13 nodes / 12 edges, 8 frames per GPU per step, frames sharded over
the GPUs of one node, one gather of detected instances).

One "step" = one batch of 8 synthetic uint8 frames per GPU through
preprocess -> UNet (tconv variant, 92.32 GFLOP/frame) -> local peaks + integral refinement ->
PAF line scoring -> per-edge assignment -> greedy grouping (-> all_gather of instances, N > 1).

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, C-ABI)
  python bench.py --impl reference --steps K --warmup W    # CPU restatement of the reference path

Prints ONE JSON line (rank 0).  `value` = frames/s with frames resident in HBM; `e2e` = the same
metric through the public `predict_on_batch` call with pinned host frames (H2D + D2H inside).
Frames and weights are seeded, so `--dump-outputs DIR` gives the same inputs' results from any build.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 1024
NODES = ["head", "thorax", "abdomen", "wingL", "wingR", "forelegL", "forelegR", "midlegL", "midlegR",
         "hindlegL", "hindlegR", "eyeL", "eyeR"]
EDGES = [("thorax", "head"), ("thorax", "abdomen"), ("thorax", "wingL"), ("thorax", "wingR"),
         ("thorax", "forelegL"), ("thorax", "forelegR"), ("thorax", "midlegL"), ("thorax", "midlegR"),
         ("thorax", "hindlegL"), ("thorax", "hindlegR"), ("head", "eyeL"), ("head", "eyeR")]
UNET_CFG = dict(filters=16, filters_rate=2, max_stride=32, output_stride=4, middle_block=True,
                up_interpolate=False, stacks=1)          # baseline_medium_rf.bottomup, tconv variant
SEED = 1004
FRAMES_PER_GPU = 8
GFLOP_PER_FRAME = 92.32
TARGET_PEAKS_PER_CHANNEL = 5


def c4_spec():
    return dict(backbone="unet", backbone_cfg=dict(UNET_CFG), head_type="multi_instance",
                heads=[dict(name="MultiInstanceConfmapsHead", channels=13, output_stride=4),
                       dict(name="PartAffinityFieldsHead", channels=24, output_stride=8)],
                part_names=NODES, edges=EDGES)


def make_frames(n, seed0=0):
    return np.stack([np.random.default_rng(SEED * 1000 + seed0 + i).integers(0, 256, size=(H, W, 1), dtype=np.uint8)
                     for i in range(n)])


def local_max_values(cm):
    """Values of the strict 8-neighbour maxima of one (H, W) map (workload calibration only)."""
    p = np.pad(cm, 1, constant_values=-np.inf)
    nb = np.max(np.stack([p[dy:dy + cm.shape[0], dx:dx + cm.shape[1]] for dy in range(3) for dx in range(3)
                          if not (dy == 1 and dx == 1)]), axis=0)
    return cm[cm > nb]


def calibrate_heads(weights, cms, pafs, n_frames):
    """Random-init weights give arbitrary maps.  To make the post-processing load look like a trained
    model's (SURVEY 8d: ~5 peaks per channel, ~65 peaks and ~300 candidates per frame) the two 1x1
    heads get a per-channel affine: the (5*n_frames+1)-th largest local maximum of each confidence
    channel is moved to the 0.2 threshold and the largest to 1.0; PAFs are scaled to unit std.
    This only rescales head weights/biases (setup time, not timed)."""
    k = np.asarray(weights["MultiInstanceConfmapsHead"]["kernel"]).copy()
    b = np.asarray(weights["MultiInstanceConfmapsHead"]["bias"]).copy()
    for c in range(cms.shape[-1]):
        vals = np.sort(np.concatenate([local_max_values(cms[i, :, :, c]) for i in range(cms.shape[0])]))[::-1]
        kth = min(len(vals) - 1, TARGET_PEAKS_PER_CHANNEL * n_frames)
        t, top = float(vals[kth]), float(vals[0])
        g = 0.8 / max(top - t, 1e-6)
        k[..., c] *= g
        b[c] = (b[c] - t) * g + 0.2
    weights["MultiInstanceConfmapsHead"] = dict(kernel=k, bias=b)
    s = 1.0 / max(float(pafs.std()), 1e-6)
    weights["PartAffinityFieldsHead"] = dict(kernel=np.asarray(weights["PartAffinityFieldsHead"]["kernel"]) * s,
                                             bias=np.asarray(weights["PartAffinityFieldsHead"]["bias"]) * s)
    return weights


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [s for s in sm if s > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks_file():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# --------------------------------------------------------------------------------------------
def cpu_oracle_fps(n_frames, weights, threads=None, warm=0):
    """The reference path restated on the CPU (oracle/): torch-CPU fp32 UNet + NumPy peak finding +
    PAF grouping (SciPy LSAP), on `n_frames` frames of the same workload."""
    import torch
    from oracle import convnet, paf_grouping as opg, peak_finding as opf, preprocess as opre
    threads = threads or best_threads(weights)
    torch.set_num_threads(threads)
    frames = make_frames(n_frames, 900)
    scorer = opg.PAFScorer(NODES, EDGES, pafs_stride=8)
    for i in range(warm):                               # untimed: first-touch allocations, oneDNN primitive caches
        x = opre.preprocess(frames[i:i + 1], ensure_gray=True, input_scale=1.0, pad_stride=32)
        cms, pafs = convnet.model_forward(x, c4_spec(), weights)
        p, v, si, ci = opf.find_local_peaks(cms, 0.2, "integral", 5)
        scorer.predict(pafs, [(p * np.float32(4)).astype(np.float32)], [v], [ci])
    t0 = time.perf_counter()
    for i in range(n_frames):
        x = opre.preprocess(frames[i:i + 1], ensure_gray=True, input_scale=1.0, pad_stride=32)
        cms, pafs = convnet.model_forward(x, c4_spec(), weights)
        p, v, si, ci = opf.find_local_peaks(cms, 0.2, "integral", 5)
        p = (p * np.float32(4)).astype(np.float32)
        scorer.predict(pafs, [p], [v], [ci])
    dt = time.perf_counter() - t0
    return n_frames / dt, threads


_BEST_THREADS = None


def best_threads(weights):
    """All the host threads the CPU path can *use*: torch-CPU convs stop scaling (and regress) well
    before 128 threads, so pick the fastest count among a few candidates (one forward each)."""
    global _BEST_THREADS
    if _BEST_THREADS is not None:
        return _BEST_THREADS
    import torch
    from oracle import convnet, preprocess as opre
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count()
    x = opre.preprocess(make_frames(1, 700), True, 1.0, 32)
    best, best_t = None, None
    for t in sorted({c for c in (8, 16, 32, 64, avail) if c <= avail}):
        torch.set_num_threads(t)
        convnet.model_forward(x, c4_spec(), weights)
        t0 = time.perf_counter()
        convnet.model_forward(x, c4_spec(), weights)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    _BEST_THREADS = best
    return best



# --------------------------------------------------------------------------------------------
def _peak_sets(cms, thr=0.2):
    """(sample, channel, y, x) of every strict local maximum above the threshold (the rough peaks of
    peak_finding.find_local_peaks_rough, restated by the oracle)."""
    from oracle import peak_finding as opf
    rough, vals, si, ci = opf.find_local_peaks_rough(cms, thr)
    xy = np.rint(np.asarray(rough)).astype(np.int64)
    return {(int(s), int(c), int(y), int(x)) for (x, y), s, c in zip(xy, si, ci)}


def _instances_key(peaks, stride):
    """Order-free signature of a frame's grouping: each instance as the tuple of its nodes' integer map cells
    (-1 for a missing node).  Two runs agree iff the same peaks were assigned to the same instances."""
    out = set()
    for inst in peaks:
        cell = np.where(np.isnan(inst), -1.0, np.rint(inst / np.float32(stride))).astype(np.int64)
        out.add(tuple(cell.reshape(-1).tolist()))
    return out


def c4_parity(spec, weights, handle, frames, pred16, model16, n_oracle=2, stride=4, thr=0.2, tag="fp16"):
    """End-to-end parity of the BENCHMARKED path (fp16 activations, tcgen05 convs) on the bench frames themselves:
    against the strict fp32 CUDA path (precision=1, same post-processing kernels) on all frames, and against the fp32
    CPU oracle network (torch) on the first `n_oracle` frames.  Not timed.  Reference being matched:
    sleap/nn/inference.py:2864-3003 (BottomUpInferenceLayer.call)."""
    from sleap_b200.nn.inference import BottomUpPredictor
    from sleap_b200.nn.model import DeviceModel
    from oracle import convnet, preprocess as opre
    B = len(frames)
    cms16, pafs16 = model16.forward(frames)
    out16 = pred16.inference_model.predict_on_batch(frames)
    m32 = DeviceModel(spec, weights, input_channels=1, precision=1, handle=handle)
    cms32, pafs32 = m32.forward(frames)
    L = pred16.inference_model.bottomup_layer
    p32 = BottomUpPredictor(m32, NODES, EDGES, peak_threshold=thr, batch_size=B, integral_refinement=True,
                            max_peaks_per_sample=L.max_peaks_per_sample, max_node_peaks=L.max_node_peaks,
                            max_instances_per_frame=L.max_instances)
    out32 = p32.inference_model.predict_on_batch(frames)
    cm_scale, paf_scale = float(np.abs(cms32).max()), float(np.abs(pafs32).max())
    res = {"frames": B, "reference": "fp32 CUDA-core path (precision=1) on the same frames; fp32 torch-CPU oracle on the first %d" % n_oracle,
           "max_abs_cm": float(np.abs(cms16 - cms32).max()), "max_abs_paf": float(np.abs(pafs16 - pafs32).max()),
           "cm_absmax": cm_scale, "paf_absmax": paf_scale,
           "max_rel_cm": float(np.abs(cms16 - cms32).max()) / cm_scale, "max_rel_paf": float(np.abs(pafs16 - pafs32).max()) / paf_scale,
           "rms_cm": float(np.sqrt(np.mean((cms16 - cms32) ** 2))), "rms_paf": float(np.sqrt(np.mean((pafs16 - pafs32) ** 2)))}
    s16, s32 = _peak_sets(cms16, thr), _peak_sets(cms32, thr)
    res["peaks_fp32"], res["peaks_" + tag], res["peaks_common"] = len(s32), len(s16), len(s16 & s32)
    res["peak_index_match"] = len(s16 & s32) / max(1, len(s16 | s32))
    # sub-pixel offsets of the peaks both paths found, through the whole device pipeline (instance_peaks)
    n_inst32 = n_inst_match = n_frames_match = 0
    max_off = 0.0
    max_score = 0.0
    for b in range(B):
        n16, n32 = int(out16["n_valid"][b]), int(out32["n_valid"][b])
        a, c = out16["instance_peaks"][b, :n16], out32["instance_peaks"][b, :n32]
        k16, k32 = _instances_key(a, stride), _instances_key(c, stride)
        n_inst32 += len(k32)
        n_inst_match += len(k16 & k32)
        n_frames_match += int(k16 == k32)
        sig16 = {tuple(np.where(np.isnan(i), -1.0, np.rint(i / np.float32(stride))).astype(np.int64).reshape(-1).tolist()): j
                 for j, i in enumerate(a)}
        for j32, i in enumerate(c):
            key = tuple(np.where(np.isnan(i), -1.0, np.rint(i / np.float32(stride))).astype(np.int64).reshape(-1).tolist())
            if key in sig16:
                d = np.abs(a[sig16[key]] - i)
                if np.isfinite(d).any():
                    max_off = max(max_off, float(np.nanmax(d)))
                max_score = max(max_score, abs(float(out16["instance_scores"][b, sig16[key]]) - float(out32["instance_scores"][b, j32])))
    res["instances_fp32"] = n_inst32
    res["instance_assignment_match"] = n_inst_match / max(1, n_inst32)
    res["frames_identical_grouping"] = n_frames_match / B
    res["max_offset_err_px"] = max_off
    res["max_instance_score_err"] = max_score
    if n_oracle > 0:
        x = opre.preprocess(frames[:n_oracle], ensure_gray=True, input_scale=1.0, pad_stride=32)
        ocms, opafs = convnet.model_forward(x, spec, weights)
        res["oracle"] = {"frames": n_oracle,
                         "fp32_path_max_rel_cm": float(np.abs(cms32[:n_oracle] - ocms).max() / np.abs(ocms).max()),
                         "fp32_path_max_rel_paf": float(np.abs(pafs32[:n_oracle] - opafs).max() / np.abs(opafs).max()),
                         tag + "_path_max_rel_cm": float(np.abs(cms16[:n_oracle] - ocms).max() / np.abs(ocms).max()),
                         tag + "_path_max_rel_paf": float(np.abs(pafs16[:n_oracle] - opafs).max() / np.abs(opafs).max()),
                         tag + "_path_max_abs_cm": float(np.abs(cms16[:n_oracle] - ocms).max()),
                         tag + "_path_max_abs_paf": float(np.abs(pafs16[:n_oracle] - opafs).max()),
                         "peak_index_match_vs_oracle": (lambda a, b: len(a & b) / max(1, len(a | b)))(
                             _peak_sets(cms16[:n_oracle], thr), _peak_sets(ocms, thr))}
    del p32, m32
    return res


def analytic_parity(handle, n_frames=8, n_instances=5):
    """Network-bypassing entry (sb_bottomup_from_maps) on analytic C4-size maps (256x256x13 confidence maps,
    128x128x24 PAFs per 1024x1024 frame): peak indices, candidate lists, assignments bit-exact against the
    oracle, refined coordinates / scores <= 1e-4."""
    from oracle import paf_grouping as opg, peak_finding as opf, synth
    from sleap_b200.nn import paf_grouping as pg
    from sleap_b200.nn.inference import bottomup_from_maps
    fr = [synth.make_bottomup_frame(seed=3100 + i, height=H, width=W, n_instances=n_instances, noise=0.01) for i in range(n_frames)]
    cms = np.stack([f[1] for f in fr]); pafs = np.stack([f[2] for f in fr])
    p, v, si, ci = opf.find_local_peaks(cms, 0.2, "integral", 5)
    p = (p * np.float32(4)).astype(np.float32)
    peaks = [p[si == b] for b in range(n_frames)]; vals = [v[si == b] for b in range(n_frames)]; chans = [ci[si == b] for b in range(n_frames)]
    winst, wps, wisc, wei, wepi, wls = opg.PAFScorer(synth.FLIES13_NODES, synth.FLIES13_EDGES, 8).predict(pafs, peaks, vals, chans)
    got = bottomup_from_maps(cms, pafs, pg.PAFScorer(synth.FLIES13_NODES, synth.FLIES13_EDGES, 8), 4, 0.2, "integral", 5, handle=handle)
    idx_ok = asg_ok = True
    max_xy = max_sc = max_ls = 0.0
    n_peaks = n_inst = 0
    for b in range(n_frames):
        idx_ok &= bool(np.array_equal(got["peak_channel_inds"][b], chans[b]) and np.array_equal(got["peak_vals"][b], vals[b]) and
                       np.array_equal(got["edge_inds"][b], wei[b]) and np.array_equal(got["edge_peak_inds"][b], wepi[b]))
        same_shape = got["instance_peaks"][b].shape == winst[b].shape
        asg_ok &= bool(same_shape and np.array_equal(np.isnan(got["instance_peaks"][b]), np.isnan(winst[b])) and
                       np.array_equal(got["instance_peak_vals"][b], wps[b]))
        n_peaks += len(chans[b]); n_inst += len(winst[b])
        if same_shape and len(winst[b]):
            max_xy = max(max_xy, float(np.nanmax(np.abs(got["instance_peaks"][b] - winst[b]))))
            max_sc = max(max_sc, float(np.abs(got["instance_scores"][b] - wisc[b]).max()))
        if len(wls[b]) and len(got["line_scores"][b]) == len(wls[b]):
            max_ls = max(max_ls, float(np.nanmax(np.abs(got["line_scores"][b] - wls[b]))))
    return {"frames": n_frames, "peaks": n_peaks, "instances": n_inst, "peak_indices_bit_exact": idx_ok,
            "instance_assignments_bit_exact": asg_ok, "max_peak_xy_err_px": max_xy, "max_line_score_err": max_ls,
            "max_instance_score_err": max_sc}


def run_reference(args):
    """--impl reference: TensorFlow (the reference's engine) is not installable offline, so the
    reference arm is the CPU restatement of its algorithm (oracle/), on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sleap_b200.nn import architectures as A
    cm = A.compile_model(c4_spec(), 1)
    weights = A.make_synthetic_weights(cm, SEED)
    import torch
    from oracle import convnet, preprocess as opre
    threads = best_threads(weights)
    torch.set_num_threads(threads)
    calib = make_frames(2, 500)
    cms0, pafs0 = convnet.model_forward(opre.preprocess(calib, True, 1.0, 32), c4_spec(), weights)
    weights = calibrate_heads(weights, cms0, pafs0, len(calib))      # same workload shaping as the CUDA arm
    for _ in range(min(args.warmup, 1)):
        cpu_oracle_fps(1, weights, threads)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        cpu_oracle_fps(1, weights, threads)
        times.append(time.perf_counter() - t0)
    fps = len(times) / sum(times)
    line = {"impl": "reference", "metric": "frames/sec (1024x1024 bottom-up UNet+PAF)", "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C4 bottom-up UNet(f16,ms32,os4,tconv)+PAF 1024x1024x1, 13 nodes/12 edges",
                       "step": "1 frame per step (bounded sample of the 8-frame batch)"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": f"{args.steps} steps x 1 frame, torch-CPU fp32 UNet + NumPy/SciPy post-processing"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def dump_outputs(out_dir, records, max_instances, n_nodes):
    """Writes the results of the last timed step as ``out_dir/<name>.npy`` (float32): the per-frame records the grouping
    kernel left on the device, split into the arrays ``predict_on_batch`` returns for the same frames.

    Those arrays hold NaN in instance slots past ``n_valid``, for nodes an instance lacks and for peaks whose refinement
    failed.  Every file written here is finite: each of the three result arrays is stored with 0 in place of those
    entries, next to ``<name>_finite.npy`` (1 where the library returned a finite value, 0 where it returned NaN)."""
    from sleap_b200 import parallel
    rec = records.cpu()
    peaks, vals, scores, n_valid = parallel.unpack_records(rec, max_instances, n_nodes)
    flags = rec[:, max_instances * n_nodes * 3 + max_instances + 1]
    out = {"n_valid": n_valid.numpy(), "flags": flags.numpy()}
    for name, a in (("instance_peaks", peaks), ("instance_peak_vals", vals), ("instance_scores", scores)):
        a = a.numpy()
        finite = np.isfinite(a)
        out[name], out[name + "_finite"] = np.where(finite, a, 0.0), finite
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


# --------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from ctypes import byref, c_int32, c_void_p

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from sleap_b200 import _lib
    from sleap_b200.nn import architectures as A
    from sleap_b200.nn.inference import BottomUpPredictor
    from sleap_b200.nn.model import DeviceModel

    handle = _lib.default_handle(local_rank)
    stream = torch.cuda.Stream()
    handle.set_stream(stream.cuda_stream)
    B = args.frames_per_gpu
    prec = {"fp16": 0, "fp32": 1, "split": 2}[args.precision]

    spec = c4_spec()
    cm = A.compile_model(spec, 1)
    weights = A.make_synthetic_weights(cm, SEED)
    # calibrated on the fp32 CPU oracle network, as the reference arm is: the head weights are an input of the benchmark
    # and must not depend on the build under test or on the conv variants its autotuner picks in this run
    from oracle import convnet, preprocess as opre
    calib = make_frames(2, 500)
    cms0, pafs0 = convnet.model_forward(opre.preprocess(calib, True, 1.0, 32), spec, weights)
    weights = calibrate_heads(weights, cms0, pafs0, len(calib))
    model = DeviceModel(spec, weights, input_channels=1, precision=prec, handle=handle)
    pred = BottomUpPredictor(model, NODES, EDGES, peak_threshold=0.2, batch_size=B, integral_refinement=True,
                             max_peaks_per_sample=1024, max_node_peaks=32, max_instances_per_frame=32)
    layer = pred.inference_model.bottomup_layer
    n_sets = 3
    host = [torch.from_numpy(make_frames(B, 10000 * rank + 100 * s)).pin_memory() for s in range(n_sets)]
    dev = [h.cuda(non_blocking=True) for h in host]
    torch.cuda.synchronize()
    out0 = pred.inference_model.predict_on_batch(host[0].numpy())          # configures everything
    n_inst_mean = float(np.mean(out0["n_valid"]))
    I, C = layer.max_instances, 13
    from sleap_b200 import parallel
    # The path's one exchange step (N > 1).  Default: the grouping kernel's epilogue stores every frame's record into every
    # rank's gather window over NVLink peer memory (sb_gather_*; no collective call in the step).  SB_EXCHANGE=nccl, or a box
    # where CUDA IPC peer mappings are not available, falls back to one ncclAllGather of the same records per step.
    pg, exchange = None, "none (1 GPU)"
    gather_out = None
    if world > 1:
        if os.environ.get("SB_EXCHANGE", "p2p") == "p2p":
            try:
                pg = parallel.PeerGather(model, generations=8)
                exchange = "peer-memory stores from the grouping kernel's epilogue (CUDA IPC over NVLink), 8 generations, device consumer lag 2"
            except Exception as e:
                sys.stderr.write(f"[bench] peer-memory exchange unavailable, using NCCL: {e}\n")
                exchange = f"ncclAllGather of the device records (peer-memory exchange unavailable: {str(e)[:80]})"
        else:
            exchange = "ncclAllGather of the device records (SB_EXCHANGE=nccl)"
        if pg is None:
            gather_out = torch.empty((world * B, parallel.record_width(I, C)), dtype=torch.float32, device="cuda")

    def as_tensor(p, shape, typestr):
        """torch view of a library-owned device buffer (plain pointer -> __cuda_array_interface__)."""
        class _V:
            pass
        v = _V()
        v.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (p.value, False), "version": 2}
        return torch.as_tensor(v, device="cuda")

    rec_ptr = c_void_p()
    handle.call("sb_bottomup_device_records", model.model_id, byref(rec_ptr))
    t_rec = as_tensor(rec_ptr, (B, parallel.record_width(I, C)), "<f4")      # written by the grouping kernel's epilogue

    def gather_step():
        parallel.all_gather_records(t_rec, gather_out)                        # NCCL fallback: zero torch ops besides the collective

    EX_LAG = 2

    post_ptr = c_void_p()
    handle.call("sb_get_post_stream", byref(post_ptr))
    post_stream = torch.cuda.ExternalStream(post_ptr.value)      # post-processing runs here, overlapping the next net

    def step_device(i):
        with torch.cuda.stream(stream):
            handle.call("sb_infer_bottomup_dev", model.model_id, c_void_p(dev[i % n_sets].data_ptr()), B)
        if pg is not None:
            n_pushed, n_consumed = pg._status()
            if n_pushed - n_consumed > EX_LAG:                    # device consumer: all ranks' records of step (now - 2)
                pg.consume_next_dev()
        elif world > 1:
            with torch.cuda.stream(post_stream):                  # queued behind this step's grouping kernel
                gather_step()

    def drain_exchange():
        if pg is not None:
            n_pushed, n_consumed = pg._status()
            for _ in range(n_pushed - n_consumed):
                pg.consume_next_dev()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput ("value") ----------------
    for i in range(args.warmup):
        step_device(i)
    drain_exchange()
    barrier()
    if args.ncu_step:
        # `ncu --profile-from-start off ... bench.py --ncu-step --steps K`: exactly K warm steps inside the
        # cudaProfilerStart/Stop window (a profiling aid; prints no bench line)
        torch.cuda.profiler.start()
        for i in range(args.steps):
            step_device(args.warmup + i)
        drain_exchange()
        barrier()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    l0 = handle.gpu_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    # live timing of the dominant kernel family: the library brackets the conv launches of every timed step with a
    # CUDA event pair on the launching stream (sb_model_forward_times); read back after the region
    handle.call("sb_model_forward_times", model.model_id, 1, 0, None, None)
    with torch.cuda.stream(stream):
        ev0.record(stream)
    for i in range(args.steps):
        step_device(i)
    drain_exchange()                                              # every step's records are consumed inside the timed region
    stream.wait_stream(post_stream)                               # last step's post-processing (+ gather) is inside the timing
    with torch.cuda.stream(stream):
        ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, t_rec, I, C)
    fwd_ms = np.zeros(max(args.steps, 1), np.float32)
    n_fwd = c_int32(0)
    handle.call("sb_model_forward_times", model.model_id, 0, len(fwd_ms), _lib.ptr(fwd_ms), byref(n_fwd))
    fwd_ms = fwd_ms[:n_fwd.value]
    launches = handle.gpu_launches() - l0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max / 1e3)

    # ---------------- sustained: the same loop for >= --sustained-seconds (power-capped clocks) ----------------
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(np.ceil(args.sustained_seconds * 1e3 / (ms_max / args.steps))))
        sampler2 = ClockSampler(local_rank) if rank == 0 else None
        if sampler2:
            sampler2.start()
            time.sleep(0.25)
        barrier()
        with torch.cuda.stream(stream):
            ev0.record(stream)
        for i in range(n_sus):
            step_device(i)
        drain_exchange()
        stream.wait_stream(post_stream)
        with torch.cuda.stream(stream):
            ev1.record(stream)
        barrier()
        ts = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sus_ms = float(ts.item())
        sustained = {"value": world * B * n_sus / (sus_ms / 1e3), "unit": "frames/s", "steps": n_sus, "seconds": sus_ms / 1e3,
                     "ms_per_step": sus_ms / n_sus, "clocks": sampler2.stop() if sampler2 else None}

    # ---------------- end to end through the public API ("e2e") ----------------
    # Predictor.predict(frames) on a pinned host stack of steps*B frames: every step's frames are
    # copied H2D and its results D2H inside the timed region (double-buffered, so the upload of
    # batch i+1 overlaps the compute of batch i); N > 1 adds the one gather of all instance records.
    big = torch.empty((args.steps * B, H, W, 1), dtype=torch.uint8).pin_memory()
    for i in range(args.steps):
        big[i * B:(i + 1) * B].copy_(host[i % n_sets])
    big_np = big.numpy()
    for i in range(min(args.warmup, 3)):
        pred.predict(big_np[:2 * B], make_labels=False)
    def e2e_once():
        barrier()
        t0 = time.perf_counter()
        outs = pred.predict(big_np, make_labels=False)
        if world > 1 and pg is None:                             # NCCL fallback: one all-gather of the K steps' records
            recs = torch.cat([parallel.pack_records(*[torch.from_numpy(np.ascontiguousarray(
                np.pad(o[k], [(0, 0), (0, I - o[k].shape[1])] + [(0, 0)] * (o[k].ndim - 2), constant_values=np.nan)))
                for k in ("instance_peaks", "instance_peak_vals", "instance_scores")] + [torch.from_numpy(o["n_valid"].astype(np.int32))])
                for o in outs]).cuda()
            with torch.cuda.stream(stream):
                parallel.all_gather_records(recs)
        elif pg is not None:                                     # peer-memory exchange: predict() collected every step's records
            assert all(o["gathered_records"].shape[0] == world * B for o in outs)
        barrier()
        return time.perf_counter() - t0, outs

    # the K-step end-to-end pass is run three times and the median reported: a single pass of ~40 ms is at the
    # mercy of one host scheduling hiccup (observed spread 5.0-6.0 k frames/s between otherwise identical runs)
    runs = [e2e_once() for _ in range(3)]
    e2e_s = sorted(r[0] for r in runs)[1]
    outs = runs[-1][1]
    assert sum(len(o["n_valid"]) for o in outs) == args.steps * B
    d2h = B * (I * C * 2 + I * C + I + 2) * 4
    te = torch.tensor([e2e_s], device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = world * B * args.steps / float(te.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (k_conv_tc) ----------------
    n_ops = c_int32(0)
    cap = 256
    op_ms = np.zeros(cap, np.float32); op_kind = np.zeros(cap, np.int32); op_fl = np.zeros(cap, np.float64)
    reps = []
    for r in range(3):
        handle.call("sb_model_profile_ops", model.model_id, c_void_p(dev[r % n_sets].data_ptr()), B, cap,
                    _lib.ptr(op_ms), _lib.ptr(op_kind), _lib.ptr(op_fl), byref(n_ops))
        reps.append((op_ms[:n_ops.value].copy(), op_kind[:n_ops.value].copy(), op_fl[:n_ops.value].copy()))
    op_ms_m = np.median(np.stack([r[0] for r in reps]), axis=0)
    kind, fl = reps[0][1], reps[0][2]
    tc = kind == 1
    if os.environ.get("BENCH_VERBOSE"):
        for i in range(len(kind)):
            sys.stderr.write(f"[op {i:2d}] kind={int(kind[i])} {op_ms_m[i]*1e3:8.1f} us  {fl[i]/1e9:7.2f} GF  {(fl[i]/max(op_ms_m[i],1e-6)/1e9):8.1f} TF/s\n")
    per_op_ms, tc_flops = float(op_ms_m[tc].sum()), float(fl[tc].sum())
    # the conv launches of one step, timed inside the timed region (mean over its K steps); the per-op pass above
    # serialises the forked transposed-conv phases and adds an event per op, so its sum is only the fallback
    tc_ms = float(fwd_ms.mean()) if len(fwd_ms) else per_op_ms
    peaks, peaks_src = peaks_file()
    # a timed region shorter than ~1 s runs at boost clocks (1965 MHz, ~300 W): the honest denominator is the BURST
    # cuBLAS figure; the power-capped "sustained" figure belongs to the seconds-long loop reported under `sustained`
    burst_region = ms_max < 1000.0
    peak_key = "bf16_tflops" if burst_region else "bf16_tflops_sustained"
    peak_tf = float(peaks.get(peak_key, peaks.get("bf16_tflops")))
    achieved_tf = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    step_ms = ms_max / args.steps
    traffic, traffic_src = None, None
    for tname in ("r02_tc_traffic.json",):                               # ncu capture of THIS round's code and autotune picks only
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath) and B == FRAMES_PER_GPU and prec == 0:  # ncu dram__bytes_read+write of the same launches
            tj = json.load(open(tpath))
            traffic = tj.get("traffic_bytes_per_step")
            traffic_src = (f"profiles/{tname}: ncu dram__bytes_read.sum+dram__bytes_write.sum summed over the conv launches of "
                           f"{tj.get('steps_captured', 1)} captured step(s), divided by that count")
            break
    roofline = {"bound": "tensor", "kernel": "k_conv_tc (tcgen05 implicit-GEMM conv, all %d launches of a step)" % int(tc.sum()),
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "peak_source": f"{peaks_src} {peak_key} ({'timed region < 1 s: boost clocks' if burst_region else 'timed region >= 1 s'})",
                "frac_of_sustained_peak": achieved_tf / float(peaks.get("bf16_tflops_sustained", peak_tf)),
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel_ms_per_step": tc_ms, "kernel_share_of_step": tc_ms / step_ms if step_ms else None,
                "kernel_timing": (f"CUDA event pair around the conv launches of each of the {len(fwd_ms)} timed steps, on the launching "
                                  "stream (sb_model_forward_times); the previous step's peak / grouping kernels overlap on a second stream"
                                  if len(fwd_ms) else "per-op CUDA events of a separate pass (sb_model_profile_ops)"),
                "per_op_sum_ms": per_op_ms,
                "algorithmic_flops_per_step": tc_flops,
                "hbm_model": {"unfused_activation_bytes_per_frame": 357e6,
                              "achieved_gbs": 357e6 * B / (float(op_ms_m.sum()) * 1e-3) / 1e9,
                              "peak_gbs": float(peaks["hbm_gbs"])}}

    # per-layer floors: a layer is bound by the larger of its tensor floor (FLOPs / sustained bf16 peak) and its HBM
    # floor (activation bytes in + out at storage width / measured copy bandwidth); the whole network's attainable
    # time is the sum of those floors.  Informational (tools/layer_rooflines.py writes the per-layer table).
    try:
        c4_layers = [(1, 1, 16, 1024, 1024, 9, 1.0, 2), (2, 16, 16, 1024, 1024, 9, 1.25, 2), (4, 16, 32, 512, 512, 9, 1.0, 2),
                     (5, 32, 32, 512, 512, 9, 1.25, 2), (7, 32, 64, 256, 256, 9, 1.0, 2), (8, 64, 64, 256, 256, 9, 1.25, 2),
                     (10, 64, 128, 128, 128, 9, 1.0, 2), (11, 128, 128, 128, 128, 9, 1.25, 2), (13, 128, 256, 64, 64, 9, 1.0, 2),
                     (14, 256, 256, 64, 64, 9, 1.25, 2), (16, 256, 512, 32, 32, 9, 1.0, 2), (17, 512, 512, 32, 32, 9, 1.0, 2),
                     (18, 512, 256, 32, 64, 2.25, 1.0, 2), (19, 512, 256, 64, 64, 9, 1.0, 2), (20, 256, 256, 64, 64, 9, 1.0, 2),
                     (21, 256, 128, 64, 128, 2.25, 1.0, 2), (22, 256, 128, 128, 128, 9, 1.0, 2), (23, 128, 128, 128, 128, 9, 1.0, 2),
                     (24, 128, 64, 128, 256, 2.25, 1.0, 2), (25, 128, 64, 256, 256, 9, 1.0, 2), (26, 64, 64, 256, 256, 9, 1.0, 2),
                     (27, 64, 13, 256, 256, 1, 1.0, 4), (28, 128, 24, 128, 128, 1, 1.0, 4)]   # op, Cin, Cout, Hin, Hout, taps, pool factor, out B/elem
        hbm = float(peaks["hbm_gbs"]) * 1e9
        fsum = msum = 0.0
        n_hbm = 0
        if B == FRAMES_PER_GPU and prec == 0 and len(op_ms_m) > 28:
            for op, cin, cout, hin, hout, taps, pf, ob in c4_layers:
                fl_op = 2.0 * taps * cin * cout * hout * hout * B
                if abs(fl_op - float(fl[op])) > 0.02 * fl_op:
                    raise ValueError(f"op {op}: layer table does not match the compiled model")
                t_t = fl_op / (peak_tf * 1e12) * 1e3            # same denominator as `peak` above
                t_h = (B * hin * hin * cin * (1 if cin == 1 else 2) + B * hout * hout * cout * ob * pf) / hbm * 1e3
                fsum += max(t_t, t_h)
                n_hbm += int(t_h > t_t)
                msum += float(op_ms_m[op])
            roofline["per_layer_floors"] = {"sum_of_floors_ms": fsum, "measured_ms": msum, "frac": fsum / msum if msum else None,
                                            "hbm_bound_layers": n_hbm, "tensor_bound_layers": len(c4_layers) - n_hbm,
                                            "hbm_peak_gbs": float(peaks["hbm_gbs"]), "tensor_peak_tflops": peak_tf}
    except Exception as e:                       # never let the informational block break the bench line
        roofline["per_layer_floors"] = {"error": str(e)}

    # ---------------- CPU baseline (oracle port) on a bounded sample ----------------
    cpu = None
    if not args.no_cpu_baseline:
        fps, threads = cpu_oracle_fps(args.cpu_frames, weights, warm=1)
        cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"1 warm-up + {args.cpu_frames} timed frames of the same workload: torch-CPU fp32 UNet + NumPy/SciPy "
                         "post-processing (tf-cpu is not installable offline)"}

    # ---------------- parity of the benchmarked path on the bench frames (untimed) ----------------
    parity = parity_maps = None
    if not args.no_parity and world == 1 and B == FRAMES_PER_GPU and prec == 0:
        try:
            parity = c4_parity(spec, weights, handle, host[0].numpy(), pred, model, n_oracle=2)
            parity_maps = analytic_parity(handle, n_frames=4)
        except Exception as e:                    # informational block: never lose the bench line over it
            parity = {"error": f"{type(e).__name__}: {e}"}

    # ---------------- the strict tensor-core path (precision 2: split fp16 pairs) on the same frames ----------------
    # Same kernels, same post-processing; activations / weights as hi + lo fp16 pairs (3 tensor-core products per term).
    # Reported beside the headline: its device-resident throughput (K steps, CUDA events) and its parity numbers.
    strict = None
    if not args.no_parity and world == 1 and B == FRAMES_PER_GPU and prec == 0:
        try:
            m2 = DeviceModel(spec, weights, input_channels=1, precision=2, handle=handle)
            p2 = BottomUpPredictor(m2, NODES, EDGES, peak_threshold=0.2, batch_size=B, integral_refinement=True,
                                   max_peaks_per_sample=1024, max_node_peaks=32, max_instances_per_frame=32)
            p2.inference_model.predict_on_batch(host[0].numpy())
            for i in range(args.warmup):
                handle.call("sb_infer_bottomup_dev", m2.model_id, c_void_p(dev[i % n_sets].data_ptr()), B)
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                ev0.record(stream)
                for i in range(args.steps):
                    handle.call("sb_infer_bottomup_dev", m2.model_id, c_void_p(dev[i % n_sets].data_ptr()), B)
            stream.wait_stream(post_stream)
            with torch.cuda.stream(stream):
                ev1.record(stream)
            torch.cuda.synchronize()
            ms2 = ev0.elapsed_time(ev1)
            strict = {"precision": "split fp16 pairs on tcgen05 (hi*Wh + lo*Wh + hi*Wl, fp32 accumulate), precision=2",
                      "value": B * args.steps / (ms2 / 1e3), "unit": "frames/s", "ms_per_step": ms2 / args.steps, "steps": args.steps,
                      "tensor_tflops_issued": 3 * GFLOP_PER_FRAME * 1e9 * B * args.steps / (ms2 / 1e3) / 1e12,
                      "parity": c4_parity(spec, weights, handle, host[0].numpy(), p2, m2, n_oracle=2, tag="split")}
            del p2, m2
        except Exception as e:
            strict = {"error": f"{type(e).__name__}: {e}"}

    if sustained is not None:
        sustained["tensor_tflops"] = GFLOP_PER_FRAME * 1e9 * sustained["value"] / 1e12
        sustained["frac_of_sustained_peak"] = sustained["tensor_tflops"] / world / float(peaks.get("bf16_tflops_sustained", peak_tf))
    line = {"metric": "frames/sec (1024x1024 bottom-up UNet+PAF)", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {0: "f16", 1: "f32", 2: "f16x3 (split fp16 pairs, fp32 accumulate)"}[prec], "data": "synthetic",
            "config": {"workload": "C4 bottom-up UNet(f16,r2,ms32,os4,tconv)+PAF 1024x1024x1, 13 nodes/12 edges (flies13)",
                       "frames_per_gpu_per_step": B, "global_batch": world * B, "parallelism": f"frame-shard x{world}",
                       "gflop_per_frame": GFLOP_PER_FRAME,
                       "l2": "3 rotating input batches; per-step activation working set ~2.9 GB >> 126 MB L2",
                       "accumulate": "fp32", "head_outputs": "fp32", "mean_instances_per_frame": n_inst_mean, "exchange": exchange,
                       "heads_calibrated_to_peaks_per_channel": TARGET_PEAKS_PER_CHANNEL,
                       "programmatic_dependent_launch": not bool(os.environ.get("SB_DISABLE_PDL"))},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * H * W, "d2h_bytes_per_step": d2h,
                    "api": "BottomUpPredictor.predict(pinned uint8 frame stack, make_labels=False), double-buffered batches",
                    "timing": "median of 3 passes of K steps (wall clock, barrier on both sides)"},
            "roofline": roofline, "cpu_baseline": cpu, "sustained": sustained, "parity": parity, "parity_analytic_maps": parity_maps, "strict_tensor_core": strict}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-gpu", type=int, default=FRAMES_PER_GPU)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "fp32", "split"],
                    help="fp16: tensor cores, fp16 activations (headline); fp32: CUDA cores; split: tensor cores, hi+lo fp16 pairs (fp32-grade results)")
    ap.add_argument("--cpu-frames", type=int, default=8)
    ap.add_argument("--sustained-seconds", type=float, default=3.0, help="length of the sustained (power-capped clocks) loop; 0 = skip")
    ap.add_argument("--no-parity", action="store_true", help="skip the (untimed) fp16-vs-fp32 parity block")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu-step", action="store_true", help="profiler window (cudaProfilerStart/Stop) around --steps warm steps, no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results (rank 0's frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    # keep stdout clean for the ONE JSON line (NCCL / torchrun print banners on stdout)
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import builtins
    _print = builtins.print

    def print_json(*a, **k):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        _print(*a, **k)
        sys.stdout.flush()
        os.dup2(2, 1)

    globals()["print"] = print_json
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
