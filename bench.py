#!/usr/bin/env python
"""bench.py — SSN forward/backward hot path on B200 (see DESIGN.md section 5).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--precision exact_tc|fast|exact] [--modality RGB|Flow] [--classes K] [--videos-per-gpu V]
                  [--mode train|infer] [--dump-outputs DIR]
  N>1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Default workload = BASELINE.json configs[1]: THUMOS14-shape synthetic, per GPU 4 videos x 8 proposals x 9 segments RGB
224x224 (32 proposals, 288 frames), K=20 classes, STPP (1,(1,2),1), dropout 0, frozen BN.  A training step = BNInception
fwd -> global-pool+STPP -> heads + multi-task loss (+ all gradients) -> backbone bwd -> NCCL gradient allreduce (N>1) ->
SGD step -> weight re-pack.  The other BASELINE configs are reachable through flags:
  configs[2]  --modality Flow                      (2x5-channel stacked flow)
  configs[3]  --classes 200 --videos-per-gpu 8     (ActivityNet-shape heads, 64 proposals per GPU; 1 video/GPU = global 64 on 8)
  configs[4]  --mode infer                         (ssn_test.py path: 10-crop forward of a 1000-tick video + test_fc + STPP
                                                    re-organisation of 1000 proposals, forward only)
The headline precision is exact_tc (split-operand tcgen05, meets the 1e-3 parity tolerance end to end); the fp16-operand
`fast` mode (parity partial: 9e-3 at the backbone output) is measured beside it in the same run and reported under
`modes`.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "action-detection_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

PROPS, SEG, STPP_CFG, FEAT_MULT = 8, 9, (1, (1, 2), 1), 5
# algorithmic conv MACs per frame (SURVEY section 8d): forward, data gradient (all layers but conv1), weight gradient = forward
MAC_FWD = {"RGB": 2031576064, "Flow": 2306941952}
MAC_DGRAD = 1913562112
IN_CH = {"RGB": 3, "Flow": 10}


def flop_per_frame(modality, train):
    f = MAC_FWD[modality]
    return 2.0 * (f + MAC_DGRAD + f) if train else 2.0 * f


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML every ~5 ms; nvidia-smi as a fallback)."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = [0x8, 0x40, 0x20, 0x4]          # nvmlClocksEventReason*: HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap

    def __init__(self, index):
        self.rows, self.stop_flag, self.index = [], False, index      # rows: (sm_mhz, max_mhz, [reason flags])
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        self.rows.append((float(sm), float(mx), [bool(r & b) for b in self.BITS]))

    def _sample_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [t.strip() for t in out.split(",")]
        if len(c) >= 6:
            self.rows.append((float(c[0]), float(c[1]), [t.lower().startswith("active") for t in c[2:6]]))

    def _run(self):
        while not self.stop_flag:
            try:
                if self.nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(0.005 if self.nvml else 0.1)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        mx = [r[1] for r in self.rows]
        reasons = [n for i, n in enumerate(self.NAMES) if any(r[2][i] for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "source": "nvml" if self.nvml else "nvidia-smi"}


def usable_cores():
    """threads the host really grants this process: affinity mask capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


# ---- workload description ------------------------------------------------------------------------------
def workload(args):
    if args.mode == "infer":
        return ("inference path (ssn_test.py:68-96): one synthetic video per step = %d ticks x %d crops %s 224x224 "
                "(%d frames) forward-only through BNInception + folded test_fc with the crop mean, then STPPReorgainzed over "
                "%d proposals; K=%d, STPP (1,(1,2),1)" % (args.infer_ticks, args.crops, args.modality,
                                                          args.infer_ticks * args.crops, args.infer_props, args.classes))
    n = args.videos_per_gpu * PROPS
    tag = {("RGB", 20): "THUMOS14-shape", ("Flow", 20): "THUMOS14-shape", ("RGB", 200): "ActivityNet-shape",
           ("Flow", 200): "ActivityNet-shape"}.get((args.modality, args.classes), "custom")
    return ("%s synthetic: batch %d proposals x 9 segments %s 224x224 per GPU, BNInception SSN fwd+bwd (+allreduce+SGD+repack), "
            "K=%d, STPP (1,(1,2),1), dropout 0, frozen BN" % (tag, n, "RGB" if args.modality == "RGB" else "Flow (2x5-ch stacked)",
                                                               args.classes))


def metric_name(args):
    return "proposals/sec (forward-only inference, 10-crop BNInception SSN + STPP re-organisation)" if args.mode == "infer" \
        else "proposals/sec (9-seg BNInception SSN fwd+bwd)"


# ---- reference arm: the UNMODIFIED reference on the host CPU cores ------------------------------------------
def run_reference(args):
    """`--impl reference`: the reference's own CPU PyTorch implementation of the same step (the checkout named by
    SSNB_REFERENCE_DIR, baseline/ref_harness.py; the oracle port without it), all host threads, same configuration as our
    arm.  Rank 0 alone works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import synth, ssn_oracle as O
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import ref_harness
    cores = usable_cores()
    torch.set_num_threads(cores)
    in_ch, K = IN_CH[args.modality], args.classes
    bb = synth.synth_backbone(in_ch, seed=0, calib_frames=2)
    hd = synth.synth_heads(K, FEAT_MULT, seed=0)
    kind = "reference" if ref_harness.available() else "port"
    budget = float(os.environ.get("SSNB_REF_BUDGET_S", "1500"))
    t_begin = time.perf_counter()
    times = []
    if args.mode == "train":
        videos = args.videos_per_gpu                       # the SAME per-GPU batch our arm steps through
        batch = synth.synth_batch(videos, K, in_ch, seed=0)
        if kind == "reference":
            model = ref_harness.build_model(K, args.modality, STPP_CFG, bb, hd)
            model.train()                                  # (the reference's SSN.train() returns None)

            def one():
                ref_harness.train_step(model, batch)
        else:
            for d in (bb, hd):
                for k in d:
                    if "_bn." not in k:
                        d[k].requires_grad_(True)

            def one():
                loss, _ = O.total_loss(O.ssn_train_forward(bb, hd, *batch, stpp_cfg=STPP_CFG, in_channels=in_ch))
                loss.backward()
                for d in (bb, hd):
                    for v in d.values():
                        v.grad = None
        units = videos * PROPS
        sample = "%d videos = %d proposals x 9 seg fwd+bwd per step (the full per-GPU batch)" % (videos, units)
    else:
        # bounded sample of one video: `ticks` of its infer_ticks ticks (x crops) and the same fraction of its proposals
        ticks = max(4, args.infer_ticks // 25)
        nprop = max(4, args.infer_props * ticks // args.infer_ticks)
        frames = synth.synth_frames(ticks * args.crops, in_ch, seed=5)
        g = torch.Generator().manual_seed(7)
        tk = torch.sort(torch.randint(0, ticks + 1, (nprop, 4), generator=g), dim=1)[0]
        sc = torch.rand(nprop, 2, generator=g)
        if kind == "reference":
            model = ref_harness.build_model(K, args.modality, STPP_CFG, bb, hd, test_mode=True)
            model.prepare_test_fc()
            model.eval()
            _, R = ref_harness.import_reference()
            reorg = R.STPPReorgainzed(model.test_fc.out_features, K + 1, K, 2 * K, True, stpp_cfg=STPP_CFG)

            def one():
                with torch.no_grad():
                    rst, _ = model(frames, None, None, None, None)
                    out = rst.view(args.crops, -1, rst.shape[1]).mean(dim=0)
                    reorg.forward(out, tk, sc)
        else:
            w, b = O.prepare_test_fc(hd, FEAT_MULT)

            def one():
                with torch.no_grad():
                    feat = O.backbone_forward(bb, frames, in_ch)
                    out = torch.nn.functional.linear(feat, w, b).view(args.crops, -1, w.shape[0]).mean(dim=0)
                    O.stpp_reorganized(out, tk, sc, K + 1, K, 2 * K, STPP_CFG)
        units = nprop
        sample = "%d of %d ticks x %d crops forward + test_fc + STPP re-organisation of %d proposals per step (1/%d of a video)" % (
            ticks, args.infer_ticks, args.crops, nprop, args.infer_ticks // ticks)
    done_w = 0
    for it in range(args.warmup + args.steps):
        if it >= args.warmup and times and time.perf_counter() - t_begin > budget:
            break                                           # time budget: report the steps really run
        t0 = time.perf_counter()
        one()
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
        else:
            done_w += 1
    mean = sum(times) / len(times)
    value = units / mean
    cfg = config_dict(args, world=args.gpus)
    cfg.update({"precision": "f32 CPU", "note": "reference CPU PyTorch path (%s), rank 0 only, %d host threads" % (
        "unmodified reference checkout" if kind == "reference" else "oracle restatement", cores)})
    line = {"impl": "reference", "metric": metric_name(args), "value": value, "unit": "proposals/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": done_w, "steps_requested": args.steps, "ms_per_step": mean * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": "proposals/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def config_dict(args, world):
    if args.mode == "infer":
        return {"workload": workload(args), "videos_per_step_per_gpu": 1, "frames_per_step_per_gpu": args.infer_ticks * args.crops,
                "proposals_per_video": args.infer_props, "parallelism": "replicas x%d (videos sharded, no collective)" % world,
                "modality": args.modality, "classes": args.classes}
    return {"workload": workload(args), "global_batch_proposals": args.videos_per_gpu * PROPS * world,
            "frames_per_gpu": args.videos_per_gpu * PROPS * SEG, "parallelism": "dp%d" % world, "modality": args.modality,
            "classes": args.classes}


# ---- our arm ---------------------------------------------------------------------------------------------------
DUMP_MAX_ELEMS = 1 << 20        # 4 MiB of float32 per array: a dump of at most nine arrays stays under 64 MB


def dump_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy (float64 stays float64, everything else float32), so that two builds
    can be compared output for output.  An array of more than DUMP_MAX_ELEMS elements is replaced by a fixed sample of its
    flattened elements (seeded: the same indices in every run)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def parse_timing(report):
    rows = []
    for ln in report.decode().splitlines():
        c = ln.split("\t")
        if len(c) == 5:
            rows.append({"kernel": c[0], "phase": int(c[1]), "launches": int(c[2]), "ms": float(c[3]), "flop": float(c[4])})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--precision", default="exact_tc", choices=["exact_tc", "fast", "exact"])
    ap.add_argument("--modality", default="RGB", choices=["RGB", "Flow"])
    ap.add_argument("--classes", type=int, default=20)
    ap.add_argument("--videos-per-gpu", type=int, default=4)
    ap.add_argument("--mode", default="train", choices=["train", "infer"])
    ap.add_argument("--infer-ticks", type=int, default=1000, help="sampled frames (ticks) per video in --mode infer")
    ap.add_argument("--infer-props", type=int, default=1000, help="proposals per video in --mode infer")
    ap.add_argument("--infer-chunk", type=int, default=40, help="ticks per forward call (x crops frames)")
    ap.add_argument("--crops", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-second-mode", action="store_true", help="skip the side measurement of the other tensor-core mode")
    ap.add_argument("--grad-scale", type=float, default=4096.0)
    ap.add_argument("--no-graph", action="store_true", help="do not capture the training step in a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl ours")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import ssn_models
    from ssn_b200 import _lib
    from oracle import synth          # synthetic weights/inputs generator (test infrastructure, not measured)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.set_num_threads(max(1, usable_cores() // max(1, world)))     # host-side setup (synthetic data) shares the cores
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # keep stdout to the one JSON line: whatever NCCL_DEBUG level the environment asks for goes to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/ssnb_nccl.%h.%p.log")
        import datetime       # a rank that falls out of step fails within minutes instead of NCCL's 10-minute default
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=int(os.environ.get("SSNB_NCCL_TIMEOUT_S", "240"))))

    PREC = {"fast": _lib.FAST_FP16, "exact": _lib.EXACT_FP32, "exact_tc": _lib.EXACT_TC}
    DTYPE = {"fast": "f16 operands / f32 accumulate (tcgen05 kind::f16); parity partial",
             "exact_tc": "f32 via split f16 operands (hi+lo, 3 tcgen05 MMAs per product) / f32 accumulate; f32 storage",
             "exact": "f32 (SIMT FMA)"}
    in_ch, K = IN_CH[args.modality], args.classes
    bb = synth.synth_backbone(in_ch, seed=0, calib_frames=2)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peaks, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def count_launches(fn):
        l0 = _lib.lib.ssnb_global_launch_count()
        fn()
        torch.cuda.synchronize()
        return _lib.lib.ssnb_global_launch_count() - l0

    def timed_loop(step_fn, batches, steps, warmup):
        """W untimed + K timed steps; CUDA events around each step, L2 flushed outside the event pairs"""
        for i in range(warmup):
            step_fn(batches[i % len(batches)])
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps)]
        out = None
        with ClockSampler(local) as clocks:
            for i in range(steps):
                l2_flush.zero_()
                ev[2 * i].record()
                out = step_fn(batches[i % len(batches)])
                ev[2 * i + 1].record()
            barrier()
        ms = sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(steps))
        return max_over_ranks(ms), clocks.summary(), out

    # ===================================== training =====================================
    def build_train(precision):
        torch.manual_seed(0)
        model = ssn_models.SSN(K, 2, 5, 2, args.modality, base_model="BNInception", dropout=0, stpp_cfg=STPP_CFG)
        sd = model.state_dict()
        for k, v in bb.items():
            sd["base_model." + k].copy_(v)
        model = model.to(dev).train()
        model.set_precision(PREC[precision], args.grad_scale)
        # fused SGD over flat buffers in model.parameters() order (ssn_train.py:141-144 semantics, per-group lr_mult / decay_mult);
        # gradients are exchanged bucket by bucket on a communication stream while the backward is still running
        from ssn_b200.optim import FusedSGD
        from ssn_b200.dp import GradSync
        order = [p for p in model.parameters() if p.requires_grad]
        opt = FusedSGD(model.get_optim_policies(), lr=1e-5, momentum=0.9, weight_decay=5e-4, order=order,
                       on_step=[model.base_model.invalidate_packed])
        flat_grad = opt.flat_grad
        sync = GradSync(flat_grad, order, model)

        def eager_step(batch):
            flat_grad.zero_()
            losses = model.fused_step(*batch, global_videos=args.videos_per_gpu * world, loss_scale=1.0 / world, grad_sync=sync)
            sync.finish()
            opt.step()
            return losses
        return model, flat_grad, opt, eager_step

    def graphed(eager_step, example):
        """the whole step (~400 launches + all-reduce + optimizer + weight re-pack) captured once in a CUDA graph; the step's
        inputs are copied into the graph's static input tensors"""
        static_batch = tuple(torch.empty_like(t) for t in example)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                for d_, s_ in zip(static_batch, example):
                    d_.copy_(s_)
                eager_step(static_batch)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_losses = eager_step(static_batch)

        def graph_step(batch):
            for d_, s_ in zip(static_batch, batch):
                d_.copy_(s_)
            graph.replay()
            return static_losses
        return graph_step

    def measure_train(precision, steps, warmup, batches, dump_dir=None):
        model, flat_grad, opt, eager_step = build_train(precision)
        step, used_graph = eager_step, False
        if not args.no_graph:
            try:
                step, used_graph = graphed(eager_step, batches[0]), True
            except Exception as ex:          # capture not possible on this stack: stay eager, say so
                if rank == 0:
                    print("CUDA graph capture failed, running eagerly: %r" % (ex,), file=sys.stderr)
                torch.cuda.synchronize()
                step, used_graph = eager_step, False
        ms_total, clocks, losses = timed_loop(step, batches, steps, warmup)
        if dump_dir and rank == 0:
            # the last timed step's results, before any later (eager) step overwrites them: the losses, the model outputs
            # of fused_step (a replayed graph writes into the tensors captured in model.last_fused), the gradient and the
            # parameters after the SGD update
            lf = model.last_fused
            dump_outputs(dump_dir, {"losses": losses, "act": lf["raw_act"], "comp": lf["raw_comp"], "reg": lf["raw_reg"],
                                    "feat": lf["feat"], "course": lf["course"], "stpp": lf["stpp"], "grads": flat_grad,
                                    "params": opt.flat_param})
        launches = count_launches(lambda: eager_step(batches[0])) * steps     # graph replays bypass the library's counter
        props_step = args.videos_per_gpu * PROPS * world
        res = {"value": props_step * steps / (ms_total / 1e3), "ms_per_step": ms_total / steps, "clocks": clocks,
               "losses": [float(v) for v in losses.tolist()], "cuda_graph": used_graph, "gpu_launches": int(launches)}
        return res, model, flat_grad, opt, eager_step

    if args.mode == "train":
        nb = 2   # distinct device-resident batches, alternated
        batches = [tuple(t.to(dev) for t in synth.synth_batch(args.videos_per_gpu, K, in_ch, seed=100 * rank + i)) for i in range(nb)]
        host_batches = [tuple(t.pin_memory() for t in synth.synth_batch(args.videos_per_gpu, K, in_ch, seed=100 * rank + i)) for i in range(nb)]
        main, model, flat_grad, opt, eager_step = measure_train(args.precision, args.steps, args.warmup, batches, args.dump_outputs)
        props_step = args.videos_per_gpu * PROPS * world
        frames_gpu = args.videos_per_gpu * PROPS * SEG

        # ---- e2e: the reference-facing module calls (ssn_train.py:207-236) with HOST inputs ----------
        import ops.ssn_ops as R
        act_crit, comp_crit, reg_crit = torch.nn.CrossEntropyLoss(), R.CompletenessLoss(), R.ClassWiseRegressionLoss()
        copy_stream = torch.cuda.Stream(device=dev)
        main_stream = torch.cuda.current_stream()

        def prefetch(hb):
            """host (pinned) -> device copy of one step's inputs on the copy stream; double-buffered so the copy of step i+1
            overlaps the compute of step i (both inside the timed region)"""
            with torch.cuda.stream(copy_stream):
                db_ = tuple(t_.to(dev, non_blocking=True) for t_ in hb)
                evc = torch.cuda.Event()
                evc.record(copy_stream)
            return db_, evc

        def e2e_compute(db_, evc):
            main_stream.wait_event(evc)
            for t_ in db_:
                t_.record_stream(main_stream)
            x, sc, tg, rt, pt = db_
            flat_grad.zero_()
            a, at, c, ct, r, rl, rtt = model(x, sc, tg, rt, pt)
            loss = act_crit(a, at) + 0.1 * comp_crit(c, ct, 1, 7) + 0.1 * reg_crit(r, rl, rtt)
            (loss / world).backward()
            if world > 1:
                dist.all_reduce(flat_grad)
            opt.step()
            return loss

        def e2e_run(n):
            nxt = prefetch(host_batches[0])
            last = None
            for i in range(n):
                cur = nxt
                if i + 1 < n:
                    nxt = prefetch(host_batches[(i + 1) % nb])
                loss = e2e_compute(*cur)
                if last is not None:
                    last.item()                 # device -> host read of the previous step's result (one step of lag)
                last = loss
            return last.item()

        e2e_steps = max(3, args.steps // 2)
        e2e_run(3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        e2e_run(e2e_steps)
        e1.record()
        barrier()
        e2e_value = props_step * e2e_steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
        h2d = sum(t_.numel() * t_.element_size() for t_ in host_batches[0])
        e2e = {"value": e2e_value, "unit": "proposals/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4, "steps": e2e_steps,
               "path": "SSN.forward + CrossEntropy/CompletenessLoss/ClassWiseRegressionLoss + backward + SGD from pinned host tensors, "
                       "H2D double-buffered on a copy stream, loss.item() every step"}

        # ---- roofline: every launch of two eager steps timed with CUDA events on the launching stream (ssnb_timing_*),
        #      aggregated per kernel and pass; algorithmic FLOPs tagged by the engine.  Eager, not graph-replayed: the
        #      per-launch figures include the (small) launch gaps of an eager run, so they are a lower bound.
        # EVERY rank runs the profiled steps (they contain the gradient all-reduce); rank 0 alone records and reports.
        import ctypes as C
        roof = None
        eager_step(batches[0]); torch.cuda.synchronize()
        n_prof = 2
        if rank == 0:
            _lib.lib.ssnb_timing_begin(C.c_void_p(torch.cuda.current_stream().cuda_stream))
        for i in range(n_prof):
            eager_step(batches[i % nb])
        if rank == 0:
            rows = parse_timing(_lib.lib.ssnb_timing_report())
            roof = roofline_from_rows(rows, n_prof, args.precision, peaks, peak_src, frames_gpu, args.modality)
        barrier()

        fused_bw = fused_gpool_stpp_bw(torch, _lib, model, frames_gpu, args.precision, l2_flush, peaks) if rank == 0 else None

        # ---- the other tensor-core mode, measured in the same run (half the steps) ----
        modes = None
        if not args.no_second_mode and args.precision in ("exact_tc", "fast"):
            other = "fast" if args.precision == "exact_tc" else "exact_tc"
            del model, opt, eager_step
            torch.cuda.empty_cache()
            o_res, o_model, _fg, _opt, _es = measure_train(other, max(5, args.steps // 2), args.warmup, batches)
            modes = {other: {"value": o_res["value"], "ms_per_step": o_res["ms_per_step"], "dtype": DTYPE[other],
                             "losses": o_res["losses"], "clocks": o_res["clocks"],
                             "parity": "backbone output 9e-3 rel-L2 vs the fp32 reference (tolerance 1e-3): partial" if other == "fast"
                             else "backbone output 2e-4 rel-L2 vs the fp32 reference (tolerance 1e-3): pass"}}
            model = o_model if args.precision == "fast" else None
            del o_model, _fg, _opt, _es
            torch.cuda.empty_cache()

        stpp_info = stpp_bandwidth(torch, _lib, dev, l2_flush, peaks) if rank == 0 else None
        if stpp_info is not None:
            stpp_info["fused_gpool_stpp"] = fused_bw
        cpu = cpu_baseline_subprocess(args) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None

        if rank == 0:
            cfg = config_dict(args, world)
            cfg.update({"precision": args.precision, "l2": "flushed between timed steps (256 MiB write)", "grad_scale": args.grad_scale,
                        "cuda_graph": main["cuda_graph"]})
            line = {"metric": metric_name(args), "value": main["value"], "unit": "proposals/s", "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": DTYPE[args.precision], "data": "synthetic", "config": cfg, "clocks": main["clocks"],
                    "gpu_launches": main["gpu_launches"],
                    "tflops_step": flop_per_frame(args.modality, True) * frames_gpu / (main["ms_per_step"] / 1e3) / 1e12,
                    "losses": main["losses"], "e2e": e2e, "roofline": roof, "modes": modes, "stpp": stpp_info, "cpu_baseline": cpu}
            print(json.dumps(line), flush=True)
    else:
        run_infer(args, torch, dist, ssn_models, _lib, synth, dev, rank, world, local, bb, PREC, DTYPE, timed_loop, count_launches,
                  barrier, max_over_ranks, peaks, peak_src)

    if world > 1:
        # all ranks leave together; skip NCCL/graph teardown (it can block when a captured graph holds the
        # communicator) — the process is done
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def roofline_from_rows(rows, n_steps, precision, peaks, peak_src, frames, modality):
    """dominant kernel = the tcgen05 convolution kernel (forward + data gradient, every launch of the step); second entry =
    the weight-gradient kernel.  achieved = sum(algorithmic FLOPs) / sum(launch time) over ALL launches of the kernel."""
    conv_names = ("umma_conv_v2_kernel", "umma_conv_kernel") if precision != "exact" else ("conv_kernel",)
    wg_names = ("umma_wgrad_kernel",) if precision != "exact" else ("wgrad_kernel",)

    def agg(names, phases):
        sel = [r for r in rows if r["kernel"] in names and r["phase"] in phases]
        return (sum(r["flop"] for r in sel) / n_steps, sum(r["ms"] for r in sel) / n_steps, sum(r["launches"] for r in sel) // n_steps)
    step_ms = sum(r["ms"] for r in rows) / n_steps
    sustained = float(peaks.get("bf16_tflops_sustained", 1400.0))
    burst = float(peaks.get("bf16_tflops", 1590.0))
    mma_per_product = 3 if precision == "exact_tc" else 1

    def entry(names, phases):
        fl, ms, n = agg(names, phases)
        a = fl / (ms / 1e3) / 1e12 if ms > 0 else 0.0
        return {"launches_per_step": n, "ms_per_step": ms, "algorithmic_flop_per_step": fl, "achieved": a, "frac": a / sustained,
                "frac_of_burst": a / burst, "tensor_pipe_tflops": a * mma_per_product, "share_of_step": ms / step_ms if step_ms else None}
    dom = entry(conv_names, (0, 1))
    fwd_all_ms = sum(r["ms"] for r in rows if r["phase"] == 0) / n_steps
    fwd_flop = 2.0 * MAC_FWD[modality] * frames
    per_kernel = {}
    for r in rows:
        k = "%s:%s" % (r["kernel"], ("fwd", "dgrad", "wgrad", "other")[r["phase"]])
        per_kernel[k] = {"launches": r["launches"] // n_steps, "ms": r["ms"] / n_steps}
    top = dict(sorted(per_kernel.items(), key=lambda kv: -kv[1]["ms"])[:14])
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        tr = traffic.get("umma_conv_v2_kernel:conv2_3x3_fwd:%s" % precision, traffic.get("umma_conv_v2_kernel:conv2_3x3_fwd", {})).get("dram_bytes")
    except Exception:
        tr = None
    return {"bound": "tensor", "kernel": "%s (forward + data gradient, all %d launches of a step)" % (conv_names[0], dom["launches_per_step"]),
            "achieved": dom["achieved"], "peak": sustained, "unit": "TFLOP/s", "frac": dom["frac"], "traffic": tr,
            "tensor_pipe_frac": dom["tensor_pipe_tflops"] / sustained, "mma_per_algorithmic_product": mma_per_product,
            "traffic_unit": "bytes per launch of the largest forward launch (conv2_3x3), ncu --set full dram read+write, profiles/",
            "peak_source": peak_src + " bf16 sustained (kernels timed inside a long step); frac_of_burst uses the burst figure",
            "note": "algorithmic fp32-conv FLOPs (2*F*H*W*Cout*Cin*k*k) / summed per-launch CUDA-event time of two eager steps; "
                    "exact_tc issues 3 tcgen05 MMAs per algorithmic product, tensor_pipe_tflops = achieved x 3",
            "dominant": dom, "forward": entry(conv_names, (0,)), "dgrad": entry(conv_names, (1,)), "wgrad": entry(wg_names, (2,)),
            "forward_pass_all_kernels": {"ms": fwd_all_ms, "achieved": fwd_flop / (fwd_all_ms / 1e3) / 1e12 if fwd_all_ms else None,
                                         "frac": fwd_flop / (fwd_all_ms / 1e3) / 1e12 / sustained if fwd_all_ms else None,
                                         "tensor_pipe_frac": fwd_flop * mma_per_product / (fwd_all_ms / 1e3) / 1e12 / sustained if fwd_all_ms else None},
            "step_ms_sum_of_launches": step_ms, "top_kernels_ms_per_step": top}


def stpp_bandwidth(torch, _lib, dev, l2_flush, peaks):
    """STPP HBM GB/s (the second half of BASELINE.json's metric): the standalone StructuredTemporalPyramidPooling kernels
    (ssnb_stpp_fwd / ssnb_stpp_bwd through the C ABI, L2 flushed before every launch, best of 5) at the bench shape (32
    proposals, 2 MB: launch-latency bound, SURVEY section 8d) and at 16384 proposals (1 GB) where HBM bandwidth is the bound.
    Algorithmic bytes: 61,448 B per proposal each way (9 x 1024 x 4 in, 6 x 1024 x 4 out, 8 B scaling).
    A failure here never costs the bench line."""
    try:
        import ctypes as C
        import ssn_models
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        stpp = ssn_models.SSN(20, 2, 5, 2, "RGB", base_model="BNInception", dropout=0, stpp_cfg=STPP_CFG).stpp
        lo, hi, nm, col = stpp.part_table([2, 7, 9])
        tab = [_lib.int_array(v) for v in (lo, hi, nm, col)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        out = {"hbm_peak_GB/s": hbm}
        for tag, n_prop in (("bench_shape", 32), ("large", 16384)):
            ft = torch.randn(n_prop * SEG, 1024, device=dev)
            sc = torch.rand(n_prop, 2, device=dev)
            course = torch.empty(n_prop, 1024, device=dev)
            pooled = torch.empty(n_prop, len(lo) * 1024, device=dev)
            dft = torch.empty_like(ft)
            best_f, best_b = 1e9, 1e9
            for _ in range(5):
                l2_flush.zero_()
                a.record()
                rc = _lib.lib.ssnb_stpp_fwd(ft.data_ptr(), sc.data_ptr(), n_prop, SEG, 1024, len(lo), *tab, 2, 7, course.data_ptr(), pooled.data_ptr(), stream)
                b.record(); b.synchronize()
                best_f = min(best_f, a.elapsed_time(b))
                l2_flush.zero_()
                a.record()
                rc |= _lib.lib.ssnb_stpp_bwd(course.data_ptr(), pooled.data_ptr(), sc.data_ptr(), n_prop, SEG, 1024, len(lo), *tab, 2, 7, dft.data_ptr(), stream)
                b.record(); b.synchronize()
                best_b = min(best_b, a.elapsed_time(b))
                if rc:
                    raise RuntimeError("ssnb_stpp rc=%d" % rc)
            nbytes = ft.numel() * 4 + sc.numel() * 4 + course.numel() * 4 + pooled.numel() * 4
            out[tag] = {"proposals": n_prop, "bytes": int(nbytes),
                        "fwd": {"us": best_f * 1e3, "GB/s": nbytes / (best_f / 1e3) / 1e9, "frac_of_hbm_peak": nbytes / (best_f / 1e3) / 1e9 / hbm},
                        "bwd": {"us": best_b * 1e3, "GB/s": nbytes / (best_b / 1e3) / 1e9, "frac_of_hbm_peak": nbytes / (best_b / 1e3) / 1e9 / hbm}}
            del ft, sc, course, pooled, dft
        return out
    except Exception as ex:
        return {"error": repr(ex)[:300]}


def fused_gpool_stpp_bw(torch, _lib, model, frames, precision, l2_flush, peaks):
    """the fused 7x7 global-pool + STPP kernel at the bench shape: reads the 5b output once (F x 49 x 1024 elements, fp32 in
    exact / exact_tc, fp16 in fast), writes feat + course + stpp"""
    try:
        import ctypes as C
        dev = l2_flush.device
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        eng = model.base_model.engine_for(frames, True, dev)
        n_prop = frames // SEG
        lo, hi, nm, col = model.stpp.part_table([2, 7, 9])
        feat = torch.empty(frames, 1024, device=dev)
        course = torch.empty(n_prop, 1024, device=dev)
        pooled = torch.empty(n_prop, len(lo) * 1024, device=dev)
        sc = torch.rand(n_prop, 2, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 1e9
        for _ in range(5):
            l2_flush.zero_()
            a.record()
            rc = _lib.lib.ssnb_gpool_stpp_fwd(eng.h, None, C.c_void_p(sc.data_ptr()), SEG, len(lo), _lib.int_array(lo), _lib.int_array(hi),
                                              _lib.int_array(nm), _lib.int_array(col), 2, 7, C.c_void_p(feat.data_ptr()),
                                              C.c_void_p(course.data_ptr()), C.c_void_p(pooled.data_ptr()), stream)
            b.record(); b.synchronize()
            if rc != 0:
                raise RuntimeError("ssnb_gpool_stpp_fwd rc=%d" % rc)
            best = min(best, a.elapsed_time(b))
        nbytes = frames * 49 * 1024 * (2 if precision == "fast" else 4) + feat.numel() * 4 + course.numel() * 4 + pooled.numel() * 4
        return {"proposals": n_prop, "bytes": int(nbytes), "us": best * 1e3, "GB/s": nbytes / (best / 1e3) / 1e9,
                "frac_of_hbm_peak": nbytes / (best / 1e3) / 1e9 / hbm}
    except Exception as ex:
        return {"error": repr(ex)[:300]}


def cpu_baseline_subprocess(args):
    """the reference arm on a bounded sample (1 warm-up + 1 timed step of the same per-GPU batch), in its own process: the
    reference's module names (ssn_models, ops, model_zoo) collide with this repo's drop-in package"""
    try:
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1", "--modality", args.modality,
               "--classes", str(args.classes), "--videos-per-gpu", str(args.videos_per_gpu), "--mode", args.mode,
               "--infer-ticks", str(args.infer_ticks), "--infer-props", str(args.infer_props), "--crops", str(args.crops)]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900).stdout.strip().splitlines()
        return json.loads(out[-1])["cpu_baseline"]
    except Exception as ex:
        return {"error": repr(ex)[:300]}


def run_infer(args, torch, dist, ssn_models, _lib, synth, dev, rank, world, local, bb, PREC, DTYPE, timed_loop, count_launches, barrier,
              max_over_ranks, peaks, peak_src):
    """BASELINE configs[4]: the ssn_test.py loop body (:80-87) for one video per step and GPU — videos are sharded over ranks
    (replicas, no collective)."""
    from ops.ssn_ops import STPPReorgainzed
    in_ch, K = IN_CH[args.modality], args.classes
    T, crops, N, chunk = args.infer_ticks, args.crops, args.infer_props, args.infer_chunk
    hd = synth.synth_heads(K, FEAT_MULT, seed=0)

    def build(precision):
        model = ssn_models.SSN(K, 2, 5, 2, args.modality, base_model="BNInception", dropout=0, test_mode=True, stpp_cfg=STPP_CFG)
        sd = model.state_dict()
        for k, v in bb.items():
            sd["base_model." + k].copy_(v)
        for k, v in hd.items():
            sd[k].copy_(v)
        model.prepare_test_fc()
        model = model.to(dev).eval()
        model.set_precision(PREC[precision], 1.0)
        reorg = STPPReorgainzed(model.test_fc.out_features, K + 1, K, 2 * K, True, stpp_cfg=STPP_CFG)
        return model, reorg

    g = torch.Generator().manual_seed(11 + rank)
    ticks = torch.sort(torch.randint(0, T + 1, (N, 4), generator=g), dim=1)[0].to(dev)
    scaling = torch.rand(N, 2, generator=g).to(dev)
    # one video, crop-major inside each chunk of `chunk` ticks (frames.view(-1, length, H, W) of ssn_test.py:80)
    n_chunks = (T + chunk - 1) // chunk
    video = synth.synth_frames(T * crops, in_ch, seed=50 + rank)                 # [T*crops, C, 224, 224] host
    video_dev = video.to(dev)

    def step_on(model, reorg, src):
        out = torch.empty(T, model.test_fc.out_features, device=dev)
        with torch.no_grad():
            for c in range(n_chunks):
                nt = min(chunk, T - c * chunk)
                frames = src[c * chunk * crops: (c * chunk + nt) * crops]
                out[c * chunk: c * chunk + nt] = model.test_scores(frames, crops)
            return reorg.forward(out, ticks, scaling)

    model, reorg = build(args.precision)
    ms_total, clocks, scores = timed_loop(lambda b: step_on(model, reorg, b), [video_dev], args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("activity", "completeness", "regression"), scores)))
    launches = count_launches(lambda: step_on(model, reorg, video_dev)) * args.steps
    value = N * world * args.steps / (ms_total / 1e3)
    frames_s = T * crops * world * args.steps / (ms_total / 1e3)

    # e2e: the same call from a pinned host video, chunks copied H2D on a copy stream inside the timed region, results read back
    host_video = video.pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()

    def e2e_step():
        out = torch.empty(T, model.test_fc.out_features, device=dev)
        with torch.no_grad():
            def fetch(c):
                nt = min(chunk, T - c * chunk)
                with torch.cuda.stream(copy_stream):
                    d = host_video[c * chunk * crops: (c * chunk + nt) * crops].to(dev, non_blocking=True)
                    e = torch.cuda.Event(); e.record(copy_stream)
                return d, e, nt
            nxt = fetch(0)
            for c in range(n_chunks):
                d, e, nt = nxt
                if c + 1 < n_chunks:
                    nxt = fetch(c + 1)
                main_stream.wait_event(e)
                d.record_stream(main_stream)
                out[c * chunk: c * chunk + nt] = model.test_scores(d, crops)
            a, cpl, rg = reorg.forward(out, ticks, scaling)
        return a.cpu(), cpl.cpu(), rg.cpu()

    e2e_steps = max(2, args.steps // 4)
    e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    d2h = 0
    for _ in range(e2e_steps):
        outs = e2e_step()
        d2h = sum(t.numel() * 4 for t in outs)
    e1.record()
    barrier()
    e2e_value = N * world * e2e_steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
    fwd_flop = 2.0 * MAC_FWD[args.modality] * T * crops
    sustained = float(peaks.get("bf16_tflops_sustained", 1400.0))
    achieved = fwd_flop / (ms_total / args.steps / 1e3) / 1e12
    cpu = cpu_baseline_subprocess(args) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    if rank == 0:
        cfg = config_dict(args, world)
        cfg.update({"precision": args.precision, "l2": "inputs larger than L2 (%.1f GB of frames per step)" % (video.numel() * 4 / 1e9),
                    "ticks_per_forward_call": chunk, "frames_per_forward_call": chunk * crops})
        line = {"metric": metric_name(args), "value": value, "unit": "proposals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE[args.precision], "data": "synthetic", "config": cfg, "clocks": clocks, "gpu_launches": int(launches),
                "frames_per_s": frames_s,
                "e2e": {"value": e2e_value, "unit": "proposals/s", "h2d_bytes_per_step": int(video.numel() * 4), "d2h_bytes_per_step": int(d2h),
                        "steps": e2e_steps, "path": "SSN.test_scores per chunk from a pinned host video (H2D double-buffered on a copy stream) + "
                                                    "STPPReorgainzed.forward + .cpu() of the three score tensors"},
                "roofline": {"bound": "tensor", "kernel": "whole forward step (all kernels)", "achieved": achieved, "peak": sustained, "unit": "TFLOP/s",
                             "frac": achieved / sustained, "traffic": None, "peak_source": peak_src + " bf16 sustained",
                             "note": "algorithmic forward conv FLOPs of the step / step time; exact_tc issues 3 MMAs per product"},
                "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
