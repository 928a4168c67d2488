#!/usr/bin/env python
"""bench.py -- image-pairs/sec of the B200 matching hot path on the BASELINE.json configurations.

  python bench.py --gpus 1 --steps K --warmup W [--config 2]     our arm (CUDA engine through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...          reference arm: the CPU path (oracle port of the
                                                                   reference modules) on the host cores, rank 0 only
  torchrun ... bench.py --gpus N ...                               one rank per GPU, the pair stream dealt round-robin

--config 2 (default, BASELINE `metric`): SuperPoint+LightGlue, 64 synthetic 640x480 pairs per GPU per step.
--config 1: the reference's own CPU-runnable case (SuperPoint + mutual NN + MAGSAC on the tests/data pair).
--config 3: LoFTR, 32 synthetic 1024x1024 pairs per step.   --config 4: ALIKED + LightGlue + MAGSAC++ F stream.
--config 5: dual-softmax / mutual NN on 4096 x 128-d descriptors (the matcher side of DISK+NN).

A step = one batch of pairs through the whole path.  The synthetic stream is a cycle of NB = 5 distinct batches dealt
round-robin: global batch g = step * world + rank takes stream batch g mod 5 (gcd(5, N) = 1 for N = 1, 2, 4, 8, so
every rank meets every batch equally often).  Prints ONE JSON line.  The only collective is one all_gather of the
per-pair match counts after the timed loop (SURVEY.md 8(e)).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

NB = 5                      # distinct batches in the synthetic stream
H, W = 480, 640
SP_CONF = {"nms_radius": 3, "keypoint_threshold": 0.005, "max_keypoints": 1024, "remove_borders": 4}
# algorithmic work (SURVEY.md 8(d) / BASELINE.md section 4), GFLOP per 480x640 image
SP_GFLOP_PER_IMAGE = 52.10
SP_LAYER_GFLOP = {"conv1a": 0.354, "conv1b": 22.65, "conv2a": 5.66, "conv2b": 5.66, "conv3a": 2.83, "conv3b": 5.66, "conv4a": 1.415,
                  "conv4b": 1.415, "convPa": 2.83, "convPb": 0.160, "convDa": 2.83, "convDb": 0.629}


def lg_gflop(n, layers):
    return (layers * (4.98e6 * n + 3584.0 * n * n) + 2.6e5 * n + 512.0 * n * n) / 1e9


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--pairs", type=int, default=0, help="pairs per GPU per step (default: the config's batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--f1-pairs", type=int, default=8, help="pairs of the timed stream checked against the oracle (match_f1)")
    ap.add_argument("--fp32", action="store_true", help="everything on the fp32 CUDA-core path (no tensor cores)")
    ap.add_argument("--tf32", action="store_true", help="LightGlue linears as single TF32 (fast mode, not parity-grade)")
    ap.add_argument("--sp-simt", action="store_true", help="SuperPoint convs on fp32 CUDA cores")
    ap.add_argument("--dump-sites", default="", help="write the launch-site profile of one step to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------------------
# measurement plumbing
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=100):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(period_ms)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """One DIR/<name>.npy per output: float32 stays float32, everything else (int32 counts and indices) becomes float64,
    which holds it exactly.  An output larger than its share of DUMP_BYTES keeps a fixed seeded sample of its rows, listed
    in DIR/<name>_rows.npy.  The inputs are seeded, so two builds given the same arguments can be compared file by file."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // max(len(arrays), 1)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.nbytes > share:
            keep = max(1, share // max(a.nbytes // len(a), 1))
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            np.save(out_dir / f"{name}_rows.npy", rows.astype(np.float64))
            a = a[rows]
        np.save(out_dir / f"{name}.npy", a)


def host_threads():
    """Usable host cores: CPU affinity capped by the cgroup quota (os.cpu_count() reports the whole box)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def best_cpu_threads(fn):
    """Thread count that runs the reference CPU path fastest on this box (torch CPU convs stop scaling, and
    oversubscription past the cgroup quota is catastrophic): quick calibration of `fn` (one small unit of the workload)."""
    cap = host_threads()
    best = (None, 1)
    for t in sorted({min(cap, c) for c in (8, 16, 32, 64, cap)}):
        torch.set_num_threads(t)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best[0] is None or dt < best[0]:
            best = (dt, t)
    torch.set_num_threads(best[1])
    return best[1]


def peaks():
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        return {}


def roofline_from_sites(prof, needles, work_per_step, unit, bound, kernel, note=None, traffic=None, sustained=True):
    """roofline of the dominant kernel from the live launch-site profile of one step: achieved = algorithmic work of all
    launches of that site in the step / their summed duration (CUDA events behind every launch on the launching stream)."""
    sites = prof.find(*needles)
    if not sites:
        return {"kernel": kernel, "error": f"launch site {needles} not seen in the step"}
    ms = sum(s[2] for s in sites)
    n = sum(s[1] for s in sites)
    pk = peaks()
    if bound == "tensor":
        peak = pk.get("bf16_tflops_sustained" if sustained else "bf16_tflops", 1444.3 if sustained else 1590.0)
        src = ("measured bf16 %s (MEASURED_PEAKS.json)" % ("sustained: kernel timed inside the step" if sustained else "burst")) if pk else "fallback (B200_PROFILING.md)"
    else:
        peak = pk.get("hbm_gbs", 6550.0)
        src = "measured HBM copy bandwidth (MEASURED_PEAKS.json)" if pk else "fallback (B200_PROFILING.md)"
    ach = work_per_step / ms            # G-units / ms == T-units / s   (GB/ms == TB/s -> x1000 below for GB/s)
    if bound == "hbm":
        ach *= 1e3
    return {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak, "traffic": traffic,
            "launches_per_step": n, "launch_ms": ms / max(n, 1), "share_of_step": ms / max(prof.total_ms, 1e-9),
            "algorithmic_per_step": work_per_step, "peak_source": src, **({"note": note} if note else {})}


# ---------------------------------------------------------------------------------------------------------
# configs
# ---------------------------------------------------------------------------------------------------------
class Config2:
    """SuperPoint+LightGlue, batch = 64 synthetic 640x480 pairs (BASELINE configs[1], the headline metric)."""
    metric = "image-pairs/sec @640x480 SuperPoint+LightGlue"
    default_pairs = 64

    ref_pairs_per_step = 2

    def __init__(self, dev, rank, world, args):
        from imcui_b200.utils import synth
        self.dev, self.args, self.P = dev, args, args.pairs or self.default_pairs
        P = self.P
        host_only = dev is None                       # reference arm: no engine, only the few pairs the CPU leg needs
        # the stream: NB batches of P pairs, seeds b*P .. b*P+P-1 (identical on every rank, dealt round-robin); decoded RGB
        # frames [2P,480,640,3] uint8, slot 2p+side -- what the reference's extract() is handed (extract_features.py:106)
        self.h_batches = []
        for b in range(1 if host_only else NB):
            n = self.ref_pairs_per_step if host_only else P
            a, c = synth.make_pair_batch(range(b * P, b * P + n), H, W)
            g = np.empty((2 * n, H, W), np.uint8)
            g[0::2], g[1::2] = a, c
            rgb = synth.to_rgb(g)
            self.h_batches.append(torch.from_numpy(rgb) if host_only else torch.from_numpy(rgb).pin_memory())
        if host_only:
            return
        from imcui_b200.engine import PairEngine, PairStream
        from imcui_b200.hloc.configs import confs_dict
        from imcui_b200.utils import synth_weights
        lg_mode = 0 if args.fp32 else (2 if args.tf32 else 1)
        self.pre = dict(confs_dict["extractors"]["superpoint_max"]["preprocessing"])     # grayscale, resize_max 1600, dfactor 8
        self.eng = PairEngine(dev, P, H, W, sp_conf={**SP_CONF, "tensor_cores": not (args.fp32 or args.sp_simt)},
                              lg_conf={"use_tensor_cores": lg_mode}, frame_shape=(H, W, 3), pre_conf=self.pre,
                              sp_state_dict=synth_weights.superpoint_random_weights(0), lg_state_dict=synth_weights.lightglue_random_weights(0))
        self.stream = PairStream(self.eng)
        self.record = self.eng.new_record()
        self.d_batches = [hb.to(dev) for hb in self.h_batches]       # decoded uint8 frames, resident in HBM
        self.dtype = "f32" if args.fp32 else ("f32-equivalent: split-fp16 (2 planes, 3 products) tcgen05 convs (SuperPoint), " + ("single-TF32 linears," if args.tf32 else "split-fp16 linears /") +
                                              " split-fp16 attention / assignment on tcgen05 (LightGlue), f32 detector post-processing")

    def step_device(self, b):
        """decoded frames resident in HBM -> match records resident in HBM (pre-processing, SuperPoint, LightGlue, match gather).
        Returns per-pair match counts [P] int32."""
        return self.eng.match_frames_device(self.d_batches[b], self.record)["mcount"]

    def e2e(self, batch_ids):
        """the stream driver a match_from_paths-style caller uses: pinned host frames in, pinned host match records out,
        H2D / compute / D2H double-buffered (engine.PairStream).  Returns the number of matches seen (forces the host read)."""
        total = 0
        for rec in self.stream.run(self.h_batches[b] for b in batch_ids):
            total += int(rec["mcount"].sum())
        return total

    @property
    def h2d_bytes(self):
        return self.stream.h2d_bytes

    @property
    def d2h_bytes(self):
        return self.stream.d2h_bytes

    def outputs(self):
        """The match record of the last step (what match_frames_device hands its caller), slots past each pair's match
        count zeroed."""
        rec = self.record
        valid = torch.arange(rec["mconf"].shape[1], device=rec["mconf"].device)[None] < rec["mcount"][:, None]
        return {k: (v * valid[..., None] if v.dim() == 3 else v * valid if v.shape == valid.shape else v) for k, v in rec.items()}

    def stats(self):
        return {"mean_keypoints": float(self.record["n_kpts"].float().mean()), "mean_stop_layer": float(self.record["stop"].float().mean())}

    def workload(self, world):
        st = self.stats()
        return {"workload": "SuperPoint+LightGlue, batch=64 synthetic 640x480 pairs per GPU (BASELINE configs[1]); each step starts from the decoded RGB frames "
                            "(GPU gray conversion / normalisation = extract()'s pre-processing) and ends with the matched keypoints in original-frame coordinates",
                "pairs_per_gpu": self.P, "max_keypoints": 1024, "weights": "deterministic synthetic SuperPoint + LightGlue (utils/synth_weights.py)",
                "lightglue": "depth_confidence 0.95, width_confidence 0.99, CUDA pruning threshold 1536 (reference CUDA semantics)",
                **st, "stream": f"cycle of {NB} distinct batches dealt round-robin over ranks (seeds 0..{NB * self.P - 1})",
                "l2": "per-step working set (> 1 GB of activations per 32-image conv pass) >> 126 MB L2, and consecutive steps take different batches; no explicit flush"}

    def gflop_per_pair(self):
        st = self.stats()
        return 2 * SP_GFLOP_PER_IMAGE + lg_gflop(st["mean_keypoints"], st["mean_stop_layer"])

    def roofline(self, prof):
        n_img = 2 * self.P
        tc = not (self.args.fp32 or self.args.sp_simt)
        if tc:
            traffic = None
            try:  # per-launch DRAM bytes of this kernel from the committed ncu --set full capture
                traffic = json.loads((ROOT / "profiles" / "r2d_conv1b_ncu.json").read_text()).get("dram_bytes_per_launch")
            except Exception:
                pass
            return roofline_from_sites(prof, ["tc_conv1ab_fused"], (SP_LAYER_GFLOP["conv1a"] + SP_LAYER_GFLOP["conv1b"]) * n_img, "TFLOP/s", "tensor",
                                       "tc_conv3x3_c64_pair_kernel<fused conv1a> (SuperPoint conv1a 1->64 + conv1b 64->64 @480x640, tcgen05 cta_group::2 split-fp16 = fp32-equivalent)",
                                       note="split precision: three fp16 partial products per fp32-equivalent product (issued as two MMAs over N-concatenated weight planes): tensor-pipe FLOP/s = 3 x achieved",
                                       traffic=traffic)
        return roofline_from_sites(prof, ["sp_conv3x3"], 0.0, "TFLOP/s", "tensor", "conv3x3_nhwc_kernel (fp32 CUDA cores)")

    # ---- CPU legs (oracle = test infrastructure, used here only as the measured baseline / checker) -------------
    def cpu_unit(self):
        import oracle
        from oracle import superpoint as osp
        from oracle.check import to_float
        ws = oracle.synthetic_weights("superpoint")
        img = to_float(self._gray(0, 1)[:1])
        return lambda: osp.forward(ws, img, SP_CONF)

    def _gray(self, first_pair, n_pairs):
        """the reference's own first step on the host: cv2.cvtColor(RGB2GRAY) of the decoded frames (extract_features.py:159-162)"""
        import cv2
        rgb = self.h_batches[0][2 * first_pair: 2 * (first_pair + n_pairs)].numpy()
        return np.stack([cv2.cvtColor(f, cv2.COLOR_RGB2GRAY) for f in rgb])

    def cpu_pairs(self, n_pairs, first=0):
        """The reference's CPU path (oracle port: same PyTorch fp32 graph as the reference modules, CPU semantics =
        pruning at every layer) on pairs [first, first + n_pairs) of stream batch 0.  Returns seconds."""
        from oracle import check
        t0 = time.perf_counter()
        check.oracle_pairs(self._gray(first, n_pairs), SP_CONF, {"pruning_min_kpts": -1})
        return time.perf_counter() - t0

    cpu_sample_desc = "SuperPoint x2 + LightGlue per pair, torch CPU fp32, reference CPU semantics (early stop + pruning every layer)"

    def match_f1(self, n_pairs):
        """match-F1 of the engine (the timed defaults) vs the oracle with the same (CUDA) LightGlue semantics on the first
        n_pairs pairs of stream batch 0 -- BASELINE metric 'match-F1 vs ref' (SURVEY.md 8(d))."""
        from oracle import check
        self.eng.match_frames_device(self.d_batches[0], self.record)
        sp, lg = self.eng.sp_out, self.eng.lg_out
        got = check.engine_pairs(lg["matches"].cpu().numpy(), sp["keypoints"].cpu().numpy(), sp["counts"].cpu().numpy(), lg["stop"].cpu().numpy(), n_pairs)
        ref = check.oracle_pairs(self._gray(0, n_pairs), SP_CONF)
        return check.summarize([check.compare_pair(g, r) for g, r in zip(got, ref)])


def make_config(n, dev, rank, world, args):
    if n == 2:
        return Config2(dev, rank, world, args)
    import bench_configs
    return bench_configs.make(n, dev, rank, world, args)


# ---------------------------------------------------------------------------------------------------------
def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of the path (oracle port -- the reference is Python and not
    installable offline, DESIGN.md section 2) on the host cores; each step = a bounded sample of the workload."""
    if rank != 0:
        return
    cfg = make_config(args.config, None, 0, 1, args)      # dev = None: host-only construction
    sample = cfg.ref_pairs_per_step
    threads = best_cpu_threads(cfg.cpu_unit())
    with torch.no_grad():
        cfg.cpu_pairs(1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cfg.cpu_pairs(sample)
        dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": cfg.metric, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": getattr(cfg, "ref_workload", "SuperPoint+LightGlue, synthetic 640x480 pairs (BASELINE configs[1])"),
                   "pairs_per_step": sample},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} pairs/step x {args.steps} steps: {cfg.cpu_sample_desc}"},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.set_grad_enabled(False)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    assert torch.cuda.is_available(), "bench.py (b200 arm) needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from imcui_b200 import _lib as L
    from imcui_b200 import shard

    cfg = make_config(args.config, dev, rank, world, args)
    P, K, Wu = cfg.P, args.steps, max(args.warmup, 3)
    batch_of = lambda g: (g * world + rank) % NB          # round-robin deal of the stream

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_times(ms):
        """per-rank milliseconds -> list over ranks (tiny all_gather outside every timed region)."""
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if dist is None:
            return [float(ms)]
        out = torch.empty(world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(out, t)
        return [float(x) for x in out.tolist()]

    # ---- device-resident throughput (inputs already in HBM) -----------------------------------------
    counts_log = torch.zeros(K, P, dtype=torch.int32, device=dev)
    for g in range(Wu):
        cfg.step_device(batch_of(g))
    barrier()
    sampler = ClockSampler(local_rank, 100 if world == 1 else 250) if rank == 0 else None
    l0 = L.lib().imw_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        counts_log[k] = cfg.step_device(batch_of(Wu + k))
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cfg.outputs() if hasattr(cfg, "outputs") else {"mcount": counts_log[K - 1]})
    per_rank = rank_times(e0.elapsed_time(e1))
    launches = L.lib().imw_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    ms_max = max(per_rank)
    value = world * P * K / (ms_max / 1e3)
    # the path's only exchange step: ONE all_gather of the per-pair match counts of the whole stream (SURVEY.md 8(e))
    all_counts = shard.gather_stream_counts(counts_log.reshape(-1))
    mean_matches = float(all_counts.float().mean())
    stats = cfg.workload(world)

    # ---- end to end through the public host API (pinned host buffers in, host results out) --------
    run_host = cfg.e2e if hasattr(cfg, "e2e") else (lambda ids: [cfg.step_host(b) for b in ids])
    run_host([batch_of(g) for g in range(2)])
    barrier()
    t0 = time.perf_counter()
    run_host([batch_of(2 + k) for k in range(K)])
    barrier()
    e2e_rank = rank_times((time.perf_counter() - t0) * 1e3)
    e2e_value = world * P * K / (max(e2e_rank) / 1e3)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- live launch-site profile of one step -> roofline of the dominant kernel --------------------------
    torch.cuda.synchronize()
    with L.launch_profile(dev) as prof:
        cfg.step_device(0)
    if args.dump_sites:
        Path(args.dump_sites).parent.mkdir(parents=True, exist_ok=True)
        with open(args.dump_sites, "w") as f:
            f.write(f"# bench.py --config {args.config}: launch sites of one step ({prof.launches} launches, {prof.total_ms:.3f} ms)\n")
            for s, n, ms in prof.sites:
                f.write(f"{ms:10.4f} ms {100 * ms / prof.total_ms:6.2f}% {n:5d}x  {s}\n")
    roof = cfg.roofline(prof)
    top = [{"site": s.split("(")[0].split()[-1] + (" [" + s.split("[with ")[1].split("]")[0] + "]" if "[with " in s else ""),
            "launches": n, "ms": round(ms, 3)} for s, n, ms in prof.sites[:6]]

    cpu, f1 = None, None
    if not args.no_cpu_baseline:
        threads = best_cpu_threads(cfg.cpu_unit())
        sample = getattr(cfg, "cpu_sample_pairs", 8)
        cfg.cpu_pairs(1)
        dt = cfg.cpu_pairs(sample)
        cpu = {"value": sample / dt, "unit": "pairs/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} pairs of the same synthetic stream: {cfg.cpu_sample_desc}"}
    if args.f1_pairs > 0 and hasattr(cfg, "match_f1"):
        torch.set_num_threads(min(32, host_threads()))
        f1 = cfg.match_f1(min(args.f1_pairs, P))

    line = {
        "metric": cfg.metric, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wu,
        "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": cfg.dtype, "data": "synthetic",
        "config": {**stats, "mean_matches": mean_matches,
                   "parallelism": (f"pair stream dealt round-robin over {world} ranks, one NCCL all_gather of match counts after the stream"
                                   if world > 1 else "single GPU")},
        "achieved_tflops": value * cfg.gflop_per_pair() / 1e3 if hasattr(cfg, "gflop_per_pair") else None,
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": cfg.h2d_bytes, "d2h_bytes_per_step": cfg.d2h_bytes},
        "gpu_launches": int(launches),
        "rank_ms_per_step": {"min": min(per_rank) / K, "median": float(np.median(per_rank)) / K, "max": ms_max / K},
        "clocks": clocks,
        "roofline": roof,
        "step_profile": {"launches": prof.launches, "ms": round(prof.total_ms, 3), "top_sites": top},
        "cpu_baseline": cpu,
    }
    if f1 is not None:
        line["match_f1"] = f1["match_f1"]
        line["parity"] = f1
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
