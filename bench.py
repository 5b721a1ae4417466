"""Benchmark of the StreamYOLO hot path: frame-pairs/s of forward+loss (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model l] [--batch 8] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE for N > 1).  A "step" is one pass of
the hot path -- DFPPAFPN (CSPDarknet + PAFPN on both frames, DFP fusion) + TALHead + SimOTA/TAL loss,
model.train() semantics (batch-statistics BatchNorm, running-stat update) -- over one per-GPU batch of
synthetic 600x960 frame pairs with random-init weights.  Frame pairs are independent, so ranks run
with no data-path collective (weak scaling: per-GPU batch fixed).

value      whole-job pairs/s with inputs resident in HBM, the step replayed as one CUDA graph,
           timed with CUDA events, max over ranks.
e2e        same metric through the public API call ``model(x, targets)`` contract with HOST (pinned)
           inputs: every step copies the frame pairs + labels host->device (double buffered on a copy
           stream, like the reference's DataPrefetcher) and reads the 6 loss scalars back.
roofline   dominant kernel (tcgen05 implicit-GEMM conv) timed alone, live, with CUDA events on its
           heaviest layer shape; achieved algorithmic TFLOP/s vs the measured cuBLAS bf16 peak.
cpu_baseline / --impl reference
           the CPU oracle (oracle/, a restatement of the reference's PyTorch path; the reference itself
           needs the un-installable yolox package) on the host cores, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

MODELS = {"s": (0.33, 0.50), "m": (0.67, 0.75), "l": (1.0, 1.0), "tiny": (0.33, 0.125)}
TAL = {"s": (1.0, 0.5, 1.5), "m": (1.0, 0.4, 1.7), "l": (1.0, 0.5, 1.6), "tiny": (1.0, 0.5, 1.5)}   # cfgs/*.py
GFLOP_PER_PAIR = {"s": 61.43, "m": 176.81, "l": 384.30}     # BASELINE.md section 2 (600x960, convs, 2*MAC)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"burst": d.get("bf16_tflops", 1590.0), "sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm": d.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML polled every 2 ms
    from a thread (the timed region can be shorter than nvidia-smi's start-up), `nvidia-smi -lms` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml = index, [], None, None
        self.sm, self.mx, self.reasons, self._stop = [], None, set(), False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                mask = int(get_reasons(self.h))
                for name, bit in self.BITS:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            self.t.join(timeout=1.0)
            sm = sorted(self.sm)
            load = [v for v in sm if v >= 0.5 * sm[-1]] if sm else []
            return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml, 2 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        # "under load": ignore idle samples well below the maximum seen
        load = [v for v in sm if v >= 0.5 * sm[-1]] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


def build_model(tag, device):
    from streamyolo_b200 import synth
    from streamyolo_b200.model import DFPPAFPN, TALHead, YOLOX
    depth, width = MODELS[tag]
    gamma, thr, val = TAL[tag]
    ch = [256, 512, 1024]
    model = YOLOX(DFPPAFPN(depth, width, in_channels=ch), TALHead(8, width, in_channels=ch, gamma=gamma,
                                                                    ignore_thr=thr, ignore_value=val))
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps, m.momentum = 1e-3, 0.03                      # init_yolo, cfgs/*.py:40-44
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth.synth_state_dict(shapes))
    model.head.use_l1 = True                                    # double_trainer.py:209-216
    return model.to(device).train()


def time_dominant_kernel(tag, batch, peaks):
    """The heaviest conv of the net (head tower 3x3 at stride 8) alone: a CUDA graph of 16 launches that rotate
    over 8 input/output buffer sets (8 x 74 MB > the 126 MB L2, so every launch reads its operands from HBM and
    no host launch overhead is inside the timed region), CUDA events around the replay, best of 5."""
    from streamyolo_b200 import ops
    from streamyolo_b200.ops import View
    width = MODELS[tag][1]
    c = int(256 * width)
    n, h, w = batch, 75, 120
    sets = 8
    xs = [View(torch.randn((n, h, w, c), device="cuda").to(torch.bfloat16)) for _ in range(sets)]
    ys = [View.empty(n, h, w, c, "cuda") for _ in range(sets)]
    wt = ops.pack_conv_weight(torch.randn((c, c, 3, 3), device="cuda") * 0.02)
    part = torch.empty((ops.conv_stat_rows(), 4 * c), device="cuda")
    launches = 16

    def go(i):
        ops.conv2d(xs[i % sets], wt, ys[i % sets], 3, 1, ops.SY_CONV_RAW, partials=part)
    for i in range(3):
        go(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        with torch.cuda.graph(g):
            for i in range(launches):
                go(i)
        g.replay()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            g.replay()
            e1.record(st)
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / launches)
    ms = best
    flops = 2.0 * n * h * w * c * c * 9
    ach = flops / (ms * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": f"conv_tc_kernel<{min(256, c)}> 3x3 s1 {c}->{c} @{n}x{h}x{w}",
            "achieved": round(ach, 1), "peak": peaks["burst"], "unit": "TFLOP/s", "frac": round(ach / peaks["burst"], 4),
            "peak_source": peaks["source"] + " cuBLAS bf16 burst", "ms_per_launch": round(ms, 4),
            "algorithmic_flop_per_launch": flops,
            # dram__bytes_read.sum + dram__bytes_write.sum of this launch shape (8x75x120, 256->256) from the ncu --set full
            # capture summarised in profiles/r01_ncu_full_summary.txt (38.12 MB read + 2.96 MB written; the 36.9 MB
            # output is still L2-resident when the kernel ends).  Only meaningful for that shape.
            "traffic": (41.07e6 if (n, c) == (8, 256) else None), "traffic_unit": "bytes/launch (ncu, r01)",
            "algorithmic_bytes_per_launch": 2 * n * h * w * c * 2 + 9 * c * c * 2,
            "how": "graph of 16 launches over 8 rotating buffer sets (operands > L2), CUDA events, best of 5"}


def host_threads():
    """Threads the CPU leg may really use: the affinity mask, capped (torch CPU convs of this size stop
    scaling -- and on an oversubscribed container collapse -- beyond a few dozen threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, int(os.environ.get("SY_CPU_THREADS", 32))))


def cpu_oracle_run(tag, pairs, steps, warmup, height=600, width_px=960):
    """Times the CPU oracle (fp32) forward+loss; returns pairs/s."""
    from oracle.streamyolo_oracle import OracleCfg, StreamYoloOracle, model_shapes
    from streamyolo_b200 import synth
    depth, width = MODELS[tag]
    gamma, thr, val = TAL[tag]
    torch.set_num_threads(host_threads())
    o = StreamYoloOracle(OracleCfg(depth=depth, width=width, gamma=gamma, ignore_thr=thr, ignore_value=val),
                         synth.synth_state_dict(model_shapes(depth, width)))
    x = synth.synth_frames(pairs, height, width_px)
    tg = synth.synth_labels(pairs, height, width_px)
    ts = []
    global LAST_ORACLE_LOSS
    with torch.no_grad():
        for i in range(warmup + steps):
            if i > 0:                                   # every run on fresh running statistics: same result each time
                o = StreamYoloOracle(o.cfg, synth.synth_state_dict(model_shapes(depth, width)))
            t0 = time.perf_counter()
            r = o.forward(x, tg)
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    LAST_ORACLE_LOSS = {k: float(v) for k, v in r.items()}
    sec = sum(ts) / len(ts)
    return pairs / sec, sec


def oracle_losses(tag, pairs, bf16_storage, height=600, width_px=960):
    from oracle.streamyolo_oracle import OracleCfg, StreamYoloOracle, bf16_round, model_shapes
    from streamyolo_b200 import synth
    depth, width = MODELS[tag]
    gamma, thr, val = TAL[tag]
    torch.set_num_threads(host_threads())
    o = StreamYoloOracle(OracleCfg(depth=depth, width=width, gamma=gamma, ignore_thr=thr, ignore_value=val),
                         synth.synth_state_dict(model_shapes(depth, width)), q=bf16_round if bf16_storage else None)
    with torch.no_grad():
        r = o.forward(synth.synth_frames(pairs, height, width_px), synth.synth_labels(pairs, height, width_px))
    return {k: float(v) for k, v in r.items()}


LAST_ORACLE_LOSS = None
LOSS_KEYS = ("total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg")


def capture(fn):
    """fn() captured as a CUDA graph after one warm-up call on a side stream; returns (graph, fn's result)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    from streamyolo_b200.model import engine
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=engine.graph_capture_stream(torch.cuda.current_device())):
        out = fn()
    return g, out


def time_replays(g, steps, warmup=3):
    for _ in range(warmup):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def conv_family_time(model, x_dev, tg_dev, reps=5):
    """The dominant kernel family -- every conv_tc_kernel launch of one step -- timed live: the conv launches of one step are
    recorded (same descriptors, same buffers) and re-issued alone, in order, as one CUDA graph (programmatic edges like the
    real step); CUDA events around the replay on the launching stream.  Returns (ms per pass over all launches, launches)."""
    from streamyolo_b200 import ops
    calls = []
    orig = ops.conv2d

    def spy(*a, **k):
        calls.append((a, k))
        return orig(*a, **k)

    ops.conv2d = spy
    try:
        with torch.no_grad():
            model(x_dev, tg_dev)
        torch.cuda.synchronize()
    finally:
        ops.conv2d = orig

    def all_convs():
        for a, k in calls:
            orig(*a, **k)
    g, _ = capture(all_convs)
    best = min(time_replays(g, 5, warmup=2) for _ in range(reps))
    return best, len(calls)


def measure_train(tag, batch, dev, rank, world, steps, warmup, peaks):
    """BASELINE.json configs 2-4: one optimisation step = recording forward + backward walk + (N > 1: bucketed NCCL gradient
    all-reduce launched from the walk) + fused SGD-nesterov/EMA kernel, streamyolo_b200.train.Trainer, replayed as CUDA
    graph(s).  Same barrier / CUDA-event / max-over-ranks protocol as the headline."""
    from streamyolo_b200 import dist as sydist, ops, synth, train
    model = build_model(tag, dev)
    tr = train.Trainer(model, lr=0.01 / 64 * batch * world)
    x = synth.synth_frames(batch, 600, 960, seed=4321 + rank).to(dev)
    fut, cur = synth.synth_labels(batch, 600, 960, seed=11 + rank)
    tg = (fut.to(dev), cur.to(dev))
    ops.LAUNCHES = 0
    segments = tr.capture(x, tg)
    launches = ops.LAUNCHES // 2                        # capture() runs the step twice (warm-up + capture)
    for _ in range(warmup):
        loss = tr.replay()
    torch.cuda.synchronize()
    sydist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = tr.replay()
    e1.record()
    torch.cuda.synchronize()
    sydist.barrier()
    ms = sydist.max_over_ranks(e0.elapsed_time(e1), dev) / steps
    pairs = world * batch / (ms * 1e-3)
    gf = GFLOP_PER_PAIR[tag] * 3.0
    tf = pairs / world * gf / 1e3
    out = {"metric": "frame-pairs/sec StreamYOLO-%s 600x960 fwd+bwd+optimizer step" % tag, "value": round(pairs, 2),
           "unit": "pairs/s", "ms_per_step": round(ms, 3), "pairs_per_gpu": batch, "steps": steps, "warmup": warmup,
           "tflops_per_gpu": round(tf, 1), "frac_of_sustained_peak": round(tf / peaks["sustained"], 4), "gflop_per_pair": gf,
           "loss": float(loss["total_loss"]), "launches_per_step": launches, "cuda_graph_segments": segments,
           "allreduce": {"world": world, "bytes_per_step": 4 * tr.fs.n_param if world > 1 else 0,
                         "buckets": len(tr.sink.launched), "in_timed_region": world > 1,
                         "how": "one NCCL all-reduce per ~25 MB bucket of the flat gradient buffer, enqueued when the walk "
                                "finishes the bucket (between two graph segments), overlapping the rest of the walk"}}
    del tr, model
    torch.cuda.empty_cache()
    return out


def measure_eval_modes(model, dev, batch, steps):
    """BASELINE.json config 5 (eval forward, decoded [B, 11850, 13], NMS excluded) and SURVEY 8f-1 (on_pipe streaming, one
    frame per call with the buffered previous-frame features, CUDA-graphed)."""
    from streamyolo_b200 import synth
    out = {}
    model.eval()
    try:
        with torch.no_grad():
            x = synth.synth_frames(batch, 600, 960, seed=99).to(dev)
            for _ in range(2):
                model(x)
            g, y = capture(lambda: model(x))
            ms = time_replays(g, steps)
            out["eval"] = {"metric": "frame-pairs/sec eval forward (model.eval()(imgs) -> [B, 11850, 13], NMS excluded)",
                           "value": round(batch / ms * 1e3, 1), "unit": "pairs/s", "ms_per_step": round(ms, 4),
                           "pairs_per_gpu": batch, "out_shape": list(y.shape)}
            f0 = synth.synth_frames(1, 600, 960, seed=98)[:, :3].contiguous().to(dev)
            _, buf = model(f0, mode="on_pipe")
            buf_static = tuple(b.clone() for b in buf)

            def frame():
                o2, nb = model(f0, buffer=buf_static, mode="on_pipe")
                for d_, s_ in zip(buf_static, nb):
                    d_.copy_(s_)                          # carry the feature buffer to the next frame
                return o2
            frame()
            g2, _ = capture(frame)
            ms2 = time_replays(g2, max(steps, 20))
            out["on_pipe"] = {"metric": "ms per 600x960 frame, on_pipe streaming (batch 1, buffered features, CUDA graph)",
                              "value": round(ms2, 4), "unit": "ms/frame", "higher_is_better": False, "fps": round(1e3 / ms2, 1),
                              "budget_ms": 33.3}
    finally:
        model.train()
    return out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU path for this workload, timed on the host cores with EXACTLY the --steps /
    --warmup it prints.  It is the fp32 oracle (kind "port"): the reference's modules need the un-vendored yolox==0.3.0
    package and /root/reference does not exist on the GPU box (DESIGN.md section 6); the oracle is pinned to outputs of the
    unmodified reference files (oracle/make_golden.py).  Each step = one forward+loss over a bounded sample of the per-GPU
    batch (2 frame pairs of the same 600x960 workload), so that the run stays within a few minutes."""
    if rank != 0:
        return
    pairs = 2
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    v, sec = cpu_oracle_run(args.model, pairs, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: LAST_ORACLE_LOSS[k] for k in LOSS_KEYS})
    line = {"impl": "reference", "metric": "frame-pairs/sec StreamYOLO-%s 600x960 fwd+loss" % args.model,
            "value": round(v, 4), "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": round(sec * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            # the same workload as the GPU arm (its `config.workload` string), timed on a bounded sample of it
            "config": {"workload": "StreamYOLO-%s (random init) 600x960 frame pairs, forward+loss, train-mode BN, "
                                   "%d pairs/GPU" % (args.model, args.batch),
                       "pairs_per_gpu": args.batch, "sample_pairs_per_step": pairs,
                       "device": "host CPU cores (the reference's own CPU path: fp32 PyTorch)"},
            "cpu_baseline": {"value": round(v, 4), "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "%d pairs/step x %d steps (+%d warm-up), fp32 oracle restatement of the reference PyTorch "
                                       "path (yolox not installable, /root/reference absent on the GPU box)" % (pairs, steps, warmup)},
            "e2e": {"value": round(v, 4), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(json.dumps(line))


_JSON_OUT = None


def guard_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner on fd 1
    whatever NCCL_DEBUG says), so keep a private copy of the real stdout for the JSON line and point fd 1 at stderr for
    everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(text):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    print(text, file=out, flush=True)


def dump_outputs(path, outputs):
    """--dump-outputs: what the timed path returned in its last step, one float32 DIR/<name>.npy per output, so that two
    builds run with the same arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(v, dtype=np.float32))


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="l", choices=list(MODELS))
    ap.add_argument("--batch", type=int, default=8, help="frame pairs per GPU")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurements (configs 2-4)")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained run, eval / on_pipe modes and the conv-family timing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the six loss outputs of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    from streamyolo_b200 import dist as sydist
    rank, local_rank, world = sydist.env_world()
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200 (no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # keep stdout to the one JSON line: whatever NCCL_DEBUG level the launcher asked for goes to a file (even WARN prints
    # the "NCCL version" banner on stdout otherwise)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/sy_nccl.%h.%p.log")
    sydist.init("nccl")
    from streamyolo_b200 import ops, synth
    from streamyolo_b200.build import build
    if rank == 0:
        build()
    sydist.barrier()
    ops.lib()
    peaks = load_peaks()
    B, H, W = args.batch, 600, 960
    model = build_model(args.model, dev)
    # per-rank inputs (different seed per rank = different frame pairs; the shard of a global batch)
    x_host = synth.synth_frames(B, H, W, seed=1234 + rank).pin_memory()
    fut, cur = synth.synth_labels(B, H, W, seed=1 + rank)
    fut_host, cur_host = fut.pin_memory(), cur.pin_memory()
    x_dev, fut_dev, cur_dev = x_host.to(dev), fut_host.to(dev), cur_host.to(dev)

    ops.LAUNCHES = 0
    with torch.no_grad():
        for _ in range(2):                                    # warm caches (weight packing, func attributes)
            out = model(x_dev, (fut_dev, cur_dev))
        torch.cuda.synchronize()
        ops.LAUNCHES = 0
        out = model(x_dev, (fut_dev, cur_dev))
        launches_per_step = ops.LAUNCHES
        torch.cuda.synchronize()
        loss_ref = float(out["total_loss"])
        graph = None
        if not args.no_graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                model(x_dev, (fut_dev, cur_dev))
            torch.cuda.current_stream().wait_stream(side)
            from streamyolo_b200.model import engine
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=engine.graph_capture_stream(dev)):
                g_out = model(x_dev, (fut_dev, cur_dev))
                g_loss = torch.stack([g_out[k] for k in ("total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg")])

        def step():
            if graph is not None:
                graph.replay()
                return g_loss
            o = model(x_dev, (fut_dev, cur_dev))
            return torch.stack([o[k] for k in ("total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg")])

        # ---------------- device-resident timing
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank)
        sampler.start()
        sydist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            loss_vec = step()
        e1.record()
        torch.cuda.synchronize()
        sydist.barrier()
        ms_total = sydist.max_over_ranks(e0.elapsed_time(e1), dev)
        clocks = sampler.stop()
        ms_step = ms_total / args.steps
        value = world * B / (ms_step * 1e-3)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dict(zip(LOSS_KEYS, loss_vec.cpu().tolist())))

        # ---------------- end-to-end: host inputs, H2D every step (double buffered), D2H of the result
        copy_stream = torch.cuda.Stream()
        stage = [(torch.empty_like(x_dev), torch.empty_like(fut_dev), torch.empty_like(cur_dev)) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        res_host = torch.empty(6, dtype=torch.float32).pin_memory()

        # one CUDA graph per staging buffer: the forward reads the freshly copied inputs in place (no device-to-device copy
        # into the device-resident run's input tensors inside the timed region)
        e2e_graphs = None
        if graph is not None:
            from streamyolo_b200.model import engine as _engine
            e2e_graphs = []
            for k in range(2):
                for t_src, t_dst in zip((x_dev, fut_dev, cur_dev), stage[k]):
                    t_dst.copy_(t_src)
                torch.cuda.synchronize()
                gk = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gk, stream=_engine.graph_capture_stream(dev), pool=graph.pool()):
                    ok = model(stage[k][0], (stage[k][1], stage[k][2]))
                    lk = torch.stack([ok[n_] for n_ in ("total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg")])
                e2e_graphs.append((gk, lk))

        def prefetch(i):
            s = stage[i % 2]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i % 2])
                s[0].copy_(x_host, non_blocking=True)
                s[1].copy_(fut_host, non_blocking=True)
                s[2].copy_(cur_host, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_loop(n):
            for c in consumed:
                c.record()
            prefetch(0)
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                cs = torch.cuda.current_stream()
                cs.wait_event(ready[i % 2])
                s = stage[i % 2]
                if e2e_graphs is not None:
                    gk, lv = e2e_graphs[i % 2]
                    gk.replay()
                    consumed[i % 2].record(cs)
                else:
                    o = model(s[0], (s[1], s[2]))
                    consumed[i % 2].record(cs)
                    lv = torch.stack([o[k] for k in ("total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg")])
                res_host.copy_(lv, non_blocking=True)
            torch.cuda.synchronize()

        e2e_loop(args.warmup)
        sydist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        e2e_loop(args.steps)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        e2e_ms = sydist.max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3), dev) / args.steps
        e2e_value = world * B / (e2e_ms * 1e-3)
        h2d = x_host.numel() * 4 + fut_host.numel() * 4 + cur_host.numel() * 4
        loss_e2e = float(res_host[0])

        # ---------------- sustained: the same graph replayed for >= 3 s (clocks settle under the power cap), own clock record
        extras = {}
        if graph is not None and not args.no_extras:
            n_sus = max(args.steps, int(3200.0 / ms_step) + 1)
            sampler2 = ClockSampler(local_rank)
            sampler2.start()
            sydist.barrier()
            e0.record()
            for _ in range(n_sus):
                graph.replay()
            e1.record()
            torch.cuda.synchronize()
            sus_ms = sydist.max_over_ranks(e0.elapsed_time(e1), dev) / n_sus
            extras["sustained"] = {"value": round(world * B / (sus_ms * 1e-3), 2), "unit": "pairs/s", "ms_per_step": round(sus_ms, 4),
                                   "steps": n_sus, "seconds": round(sus_ms * n_sus * 1e-3, 2), "clocks": sampler2.stop()}
        if rank == 0 and not args.no_extras and args.model in GFLOP_PER_PAIR:
            fam_ms, fam_n = conv_family_time(model, x_dev, (fut_dev, cur_dev))
            extras["conv_family"] = (fam_ms, fam_n)
            extras.update(measure_eval_modes(model, dev, B, args.steps))
            # parity of the timed model: its loss on the oracle's own sample (2 pairs, default seeds) -- compared below
            x2 = synth.synth_frames(2, H, W).to(dev)
            t2 = synth.synth_labels(2, H, W)
            o2 = model(x2, (t2[0].to(dev), t2[1].to(dev)))
            extras["product_loss_2pairs"] = {k: float(o2[k]) for k in LOSS_KEYS}
        del graph
        torch.cuda.empty_cache()

    # ---------------- training step (BASELINE.json configs 2-4), all ranks: N > 1 puts the NCCL gradient all-reduce in the timed region
    train_out = {}
    if not args.no_train and args.model in GFLOP_PER_PAIR:
        tsteps = max(5, min(args.steps, 20))
        try:
            train_out["l_b4_ddp"] = measure_train("l", 4, dev, rank, world, tsteps, 3, peaks)        # config 4: 32 pairs / 8 GPUs
            if world == 1:
                train_out["s_b8"] = measure_train("s", 8, dev, rank, world, tsteps, 3, peaks)       # config 2
                train_out["m_b8"] = measure_train("m", 8, dev, rank, world, tsteps, 3, peaks)       # config 3
        except Exception as ex:  # never lose the headline to the secondary measurement
            train_out["error"] = "%s: %s" % (type(ex).__name__, str(ex)[:300])
    sydist.shutdown()
    if rank != 0:
        return
    gf = GFLOP_PER_PAIR.get(args.model)
    roof = time_dominant_kernel(args.model, B, peaks) if args.model in GFLOP_PER_PAIR else None
    line = {
        "metric": "frame-pairs/sec StreamYOLO-%s 600x960 fwd+loss" % args.model,
        "value": round(value, 2), "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "StreamYOLO-%s (random init) 600x960 frame pairs, forward+loss, train-mode BN, "
                               "%d pairs/GPU" % (args.model, B),
                   "pairs_per_gpu": B, "global_pairs": world * B, "parallelism": "dp%d (no data-path collective)" % world,
                   "cuda_graph": not args.no_graph,
                   "l2": "per-step inputs (%.0f MB) + activations (>1 GB) exceed the 126 MB L2" % (h2d / 1e6)},
        "e2e": {"value": round(e2e_value, 2), "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 24,
                "ms_per_step": round(e2e_ms, 4), "note": "pinned fp32 frames+labels copied every step on a copy stream "
                                                        "(double buffered), 6 loss scalars read back"},
        "gpu_launches": launches_per_step * args.steps,
        "launches_per_step": launches_per_step,
        "clocks": clocks,
        "loss_check": {"eager": loss_ref, "timed": float(loss_vec[0]), "e2e": loss_e2e},
    }
    if train_out:
        line["train"] = train_out
    for k in ("sustained", "eval", "on_pipe"):
        if k in extras:
            line[k] = extras[k]
    if gf:
        tf = value / world * gf / 1e3
        line["roofline_step"] = {"bound": "tensor", "achieved": round(tf, 1), "peak": peaks["sustained"], "unit": "TFLOP/s",
                                 "frac": round(tf / peaks["sustained"], 4), "gflop_per_pair": gf,
                                 "peak_source": peaks["source"] + " cuBLAS bf16 sustained"}
    if roof:
        line["roofline_best_shape"] = roof
        line["roofline"] = roof
    if gf and "conv_family" in extras:
        # the dominant kernel FAMILY over the step: every conv_tc_kernel launch, FLOP-weighted (the whole conv work of the
        # step / the sum of their live event-timed durations); the best single shape stays in roofline_best_shape
        fam_ms, fam_n = extras["conv_family"]
        ach = B * gf / fam_ms                      # GFLOP / ms = TFLOP/s
        line["roofline"] = {"bound": "tensor", "kernel": "conv_tc_kernel<*>: all %d conv launches of one step" % fam_n,
                            "achieved": round(ach, 1), "peak": peaks["burst"], "unit": "TFLOP/s", "frac": round(ach / peaks["burst"], 4),
                            "peak_source": peaks["source"] + " cuBLAS bf16 burst", "launches": fam_n,
                            "avg_launch_ms": round(fam_ms / fam_n, 5), "sum_launch_ms": round(fam_ms, 4),
                            "algorithmic_flop_per_step": B * gf * 1e9,
                            # dram__bytes_read.sum + dram__bytes_write.sum per launch, averaged over the family's 114 launches of
                            # one step (ncu launch list of this command, profiles/r02_launch_summary_final.txt; StreamYOLO-l, 8 pairs only)
                            "traffic": (50.5e6 if (args.model, B) == ("l", 8) else None), "traffic_unit": "bytes/launch (ncu launch list profiles/r02_launch_summary_final.txt: 5761 MB DRAM read+written over the 114 conv launches)",
                            "how": "the step's conv launches re-issued alone, in order, as one CUDA graph on the step's own buffers; "
                                   "CUDA events around the replay, best of 5; ncu launch list of the step: profiles/"}
    if not args.no_cpu_baseline:
        try:
            v, sec = cpu_oracle_run(args.model, 2, 2, 1)
            line["cpu_baseline"] = {"value": round(v, 4), "unit": "pairs/s", "cores": torch.get_num_threads(),
                                    "kind": "port", "sample": "2 pairs/step x 2 steps, fp32 oracle of the reference path"}
            if "product_loss_2pairs" in extras:
                got = extras["product_loss_2pairs"]
                want = oracle_losses(args.model, 2, bf16_storage=True)
                dev_rel = {k: round(abs(got[k] - want[k]) / (abs(want[k]) + 1e-12), 5) for k in LOSS_KEYS}
                line["parity_check"] = {"what": "losses of the timed model vs the oracle with the same bf16 storage points, same 2 frame pairs "
                                                "(a random-init train-mode BN net is chaotic under bf16 storage: the fp32 oracle's "
                                                "own losses are listed for scale)",
                                        "product": got, "oracle_bf16_storage": want, "oracle_fp32": LAST_ORACLE_LOSS, "rel_dev": dev_rel,
                                        "ok": bool(max(dev_rel[k] for k in LOSS_KEYS[:5]) < 0.08)}
        except Exception as ex:  # never lose the GPU numbers to a host-side problem
            line["cpu_baseline"] = {"value": None, "error": str(ex)[:200]}
    emit(json.dumps(line))


if __name__ == "__main__":
    main()
