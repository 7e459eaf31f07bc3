#!/usr/bin/env python
"""bench.py -- panoptic images/sec of the UPSNet-50 Cityscapes inference hot path (BASELINE.json
configs[1]: synthetic 1x3x1024x2048, batch 1 per GPU) on N B200s, one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python bench.py --dump-outputs DIR ...   # also writes the results of the last timed step as DIR/<name>.npy, so two
                                             # builds can be compared output for output (inputs and weights are seeded)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...   # the CPU port of the path (oracle/cpu_model.py) on the host cores: the reference
                                           # itself has no CPU path for its custom ops, so this arm times torch-CPU convs +
                                           # the C/OpenMP restatements (cpu_baseline.kind = "port")

One "step" = one full per-image forward (backbone -> FPN -> RPN -> proposals -> semantic head (DCN)
-> RCNN -> MaskROI -> mask head x2 -> fused panoptic head).  Images are independent, so ranks are
replicas with no data-path collective ("weak" scaling; DESIGN.md section 6).

JSON line:  value = whole-job images/s with the input image already resident in HBM (CUDA events,
max over ranks); e2e = same metric through the public serving API (upsnet_b200.pipeline.PipelinedEngine) with HOST
buffers: pinned H2D of every image and D2H of its result maps inside the timed region, overlapped across images; roofline = achieved TFLOP/s of the dominant
kernel family measured with CUDA events around its launches, against MEASURED_PEAKS.json;
cpu_baseline = the CPU path (oracle/cpu_model.py) timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "panoptic images/sec at 1024x2048"
H, W = 1024, 2048
WORKLOAD = "UPSNet-50 Cityscapes inference, synthetic 1x3x1024x2048, batch 1 per GPU (BASELINE configs[1])"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class NvmlSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed regions, read in-process through NVML every 50 ms.  Round 1 spawned an
    `nvidia-smi -lms 200` poller on rank 0 only, inside a 70 ms timed region reduced by max-over-ranks: that process made
    rank 0 the straggler of the 1->8 curve (VERDICT r1 weak 10).  An NVML query is a few microseconds of driver time."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev, self.ok = index, [], threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_ev.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.rows.append((sm, mask, util))
            except Exception:
                pass
            self._stop_ev.wait(0.05)

    def stop(self):
        self._stop_ev.set()
        if not self.ok or not self.rows:
            return None
        busy = [r for r in self.rows if r[2] > 0] or self.rows
        reasons = sorted({name for _, m, _ in busy for name, bit in self.REASONS if m & bit})
        return {"sm_mhz": statistics.median([r[0] for r in busy]), "sm_max_mhz": self.mx, "reasons": reasons,
                "samples": len(self.rows), "how": "NVML in-process, 50 ms period, during both timed regions"}


def bind_to_gpu_numa(index):
    """Pin this rank (and the threads it spawns later) to the CPU cores NVML reports as local to its GPU: the host side
    of a replay-bound step is a launch loop, and a rank scheduled on the far socket becomes the straggler."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus = {c for c in cpus if c < ncpu} & set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons (B200_PROFILING.md recipe); fallback when NVML is not importable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        busy = [c for c in sm if c > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


_REAL_STDOUT = None


def _claim_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries print there too (NCCL's version banner on the first
    communicator, oneDNN / OpenMP notices): from here on file descriptor 1 points at stderr and only emit() writes to the
    real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def _best_cpu_threads():
    """The CPU arm uses the thread count that is FASTEST on this box (more threads than ~32 slow the small torch-CPU
    convs down through oversubscription): a one-second probe on a backbone-sized 3x3 convolution picks it."""
    import torch
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | {cores})
    x = torch.randn(1, 256, 128, 256)
    w = torch.randn(256, 256, 3, 3)
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.conv2d(x, w, padding=1)
        t0 = time.perf_counter()
        for _ in range(2):
            torch.nn.functional.conv2d(x, w, padding=1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    os.environ["OMP_NUM_THREADS"] = str(best)     # the C/OpenMP oracle reads it when its library is loaded
    return best


def run_reference(args, rank):
    """--impl reference: the reference's CPU path for the same workload on the host cores."""
    import torch
    if rank != 0:
        return
    cores = _best_cpu_threads()
    from oracle.cpu_model import cpu_ops
    from upsnet_b200.model import UPSNetConfig
    from upsnet_b200.synthetic import synthetic_input, synthetic_model
    model = synthetic_model(UPSNetConfig.cityscapes_r50(), seed=0, device="cpu")
    inputs = [synthetic_input(H, W, seed=s) for s in range(2)]
    budget_s, t_begin = 280.0, time.perf_counter()
    with cpu_ops():
        done_w = 0
        for i in range(args.warmup):
            model(inputs[i % 2]); done_w += 1
            if time.perf_counter() - t_begin > budget_s / 3:
                break
        t0 = time.perf_counter()
        done = 0
        for i in range(args.steps):
            model(inputs[i % 2]); done += 1
            if time.perf_counter() - t_begin > budget_s:
                break
        dt = time.perf_counter() - t0
    val = done / dt
    sample = "%d full 1024x2048 images through torch-CPU fp32 convs + C/OpenMP restated ops (oracle/cpu_model.py)" % done
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": done, "warmup": done_w, "ms_per_step": 1e3 * dt / done, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def cpu_baseline_leg():
    import torch
    cores = _best_cpu_threads()
    from oracle.cpu_model import cpu_ops
    from upsnet_b200.model import UPSNetConfig
    from upsnet_b200.synthetic import synthetic_input, synthetic_model
    model = synthetic_model(UPSNetConfig.cityscapes_r50(), seed=0, device="cpu")
    inp = synthetic_input(H, W, seed=0)
    with cpu_ops():
        model(inp)  # warm-up (thread pools, oneDNN primitive caches)
        t0 = time.perf_counter(); n = 0
        while n < 2 or (time.perf_counter() - t0 < 15.0 and n < 8):
            model(inp); n += 1
        dt = time.perf_counter() - t0
        model.keep_intermediates = True      # one more (untimed) forward that keeps the stage boundaries for the parity block
        out = model(inp)
    return {"value": n / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "%d full 1024x2048 images (after 1 warm-up), torch-CPU fp32 convs + C/OpenMP restated ops, "
                      "%d threads (fastest of a probe over 8..%d)" % (n, cores, os.cpu_count())}, out


def dump_outputs(out, path):
    """--dump-outputs: the result dict resnet_upsnet.forward() builds from one static-engine output (upsnet_b200/model.py),
    one DIR/<name>.npy per tensor: float32 for floating-point tensors, float64 (exact) for integer ones."""
    import numpy as np
    n1, n2, k = (int(v) for v in out["counts"].tolist())
    keep = out["keep"][:k]
    res = {"cls_probs": out["cls_probs"][:n1], "pred_boxes": out["pred_boxes"][:n1], "mask_probs": out["mask_probs"][:n1],
           "cls_inds": out["cls_inds"][:n1], "fcn_outputs": out["fcn_outputs"], "panoptic_cls_inds": out["p_cls"][:n2][keep],
           "panoptic_cls_probs": out["p_scores"][:n2][keep], "panoptic_outputs": out["panoptic_outputs"]}
    arrays = {name: v.cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64) for name, v in res.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "dump exceeds 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def parity_block(gpu_model, cpu_out, dev):
    """The benchmarked configuration against the CPU forward of the same image (seed 0) that the cpu_baseline leg just
    computed: logits within 1e-3 (relative to the tensor's max), label maps on the engine's own head inputs."""
    import numpy as np
    import torch
    from oracle import oracle as O
    from upsnet_b200.synthetic import synthetic_input
    inp = synthetic_input(H, W, seed=0, device=dev)
    gpu_model.keep_intermediates = True
    out = gpu_model(inp)
    gpu_model.keep_intermediates = False
    a, b = out["_intermediates"], cpu_out["_intermediates"]

    def rel(x, y):
        x, y = x.float().cpu(), y.float().cpu()
        return float((x - y).abs().max() / max(1.0, float(y.abs().max())))
    blk = {"against": "CPU fp32 forward of the same synthetic image (oracle/cpu_model.py), same weights",
           "fcn_output_max_rel_diff": rel(a["fcn_output"], b["fcn_output"]),
           "fpn_max_rel_diff": max(rel(x, y) for x, y in zip(a["fpn"], b["fpn"])),
           "semantic_label_agreement": float((out["fcn_outputs"].cpu() == cpu_out["fcn_outputs"]).float().mean()),
           "panoptic_label_agreement_vs_cpu_forward": float((out["panoptic_outputs"].cpu() == cpu_out["panoptic_outputs"]).float().mean())}
    keep, labels = O.panoptic_head(a["fcn_output"][0].float().cpu().numpy(), a["pmask_rois"][:, 1:].cpu().numpy(),
                                   a["pcls_prob"].cpu().numpy(), a["pmask_score"][:, 0].float().cpu().numpy(),
                                   a["pcls_idx"].cpu().numpy(), 11)
    blk["panoptic_labels_bit_exact_on_engine_inputs"] = bool(np.array_equal(out["panoptic_outputs"][0].cpu().numpy(), labels)
                                                             and a["keep_inds"].cpu().tolist() == keep.tolist())
    blk["logits_within_1e-3"] = bool(blk["fcn_output_max_rel_diff"] <= 1e-3 and blk["fpn_max_rel_diff"] <= 1e-3)
    return blk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("UPSNET_PRECISION", "bf16x3"), choices=["fp32", "bf16x3", "bf16"],
                    help="bf16x3 (default, the configuration the parity tests certify at 'fp32 logits within 1e-3'): tcgen05 "
                         "hi/lo split on the hi/lo bf16 pair stream; bf16: tcgen05 single pass + bf16 activation storage "
                         "(secondary figure, bf16-level error); fp32: CUDA-core tiles")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the configs[2] / configs[4] extras of the default run")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("UPSNET_LANES", "2")),
                    help="images in flight per GPU: independent engine instances (CUDA-graph instance + pool + scratch) on their own streams")
    ap.add_argument("--workload", default="cityscapes", choices=["cityscapes", "coco"],
                    help="cityscapes = BASELINE configs[1] (the metric); coco = configs[2] UPSNet-101-DCN 800x1344 (extra)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last one (the tensors forward() returns) to DIR/<name>.npy")
    args = ap.parse_args()
    _claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist
    import upsnet_b200 as U
    from upsnet_b200 import operators as ops
    from upsnet_b200.model import UPSNetConfig
    from upsnet_b200.synthetic import synthetic_input, synthetic_model
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    numa_cpus = 0 if os.environ.get("UPSNET_BENCH_NO_NUMA") else bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # keep stdout to the single JSON line: NCCL's version banner (NCCL_DEBUG=VERSION) would precede it
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    U.set_precision(args.precision)
    global H, W, WORKLOAD
    if args.workload == "coco":
        H, W = 800, 1344
        WORKLOAD = ("UPSNet-101-DCN COCO inference, synthetic 800x1344 (padded from 1333), one image per step "
                    "(BASELINE configs[2]; heads are per-image in the reference, SURVEY F9)")
        model = synthetic_model(UPSNetConfig.coco_r101_dcn(), depth=(3, 4, 23, 3), seed=0, device=dev)
    else:
        model = synthetic_model(UPSNetConfig.cityscapes_r50(), seed=0, device=dev)
    n_img = 4  # rotate distinct images; one step touches >1 GB of activations (>> 126 MB L2)
    host_imgs = [synthetic_input(H, W, seed=100 * rank + s)["data"].pin_memory() for s in range(n_img)]
    dev_imgs = [h.to(dev) for h in host_imgs]
    im_info = synthetic_input(8, 8)["im_info"]; im_info[0, :2] = (H, W)

    def step_resident(i):
        return model({"data": dev_imgs[i % n_img], "im_info": im_info})

    # The resident leg drives the SYNC-FREE engine entry: one CUDA-graph replay per image, the 3-int result-size vector
    # copied to pinned host memory asynchronously (model.forward() would block the host on it every image, which makes the
    # number a measure of host wake-up latency: 101..151 images/s from run to run in round 2).  Everything the forward
    # computes is computed; the sizes are checked after the timed region.
    counts_host = torch.zeros((max(args.steps, 8), 3), dtype=torch.int32).pin_memory()

    # Engine lanes: image i runs on lane i % LANES -- an independent engine instance (own CUDA-graph instance, activation
    # pool, output buffers, scratch) on its own stream -- so the forward passes of LANES consecutive images overlap on the
    # GPU: the single-CTA detection kernels (top-k, NMS sweeps, MaskROI, pan_decide) and the small-grid coarse-level convs
    # of one image hide under the machine-filling convolutions of the other.  Batch stays 1 image per step.
    LANES = max(1, int(args.lanes))
    lane_streams = [torch.cuda.Stream(dev) for _ in range(LANES)]
    last_out = [None]     # engine outputs of the latest step_graph call

    def step_graph(i):
        l = i % LANES
        with torch.cuda.stream(lane_streams[l]):
            out, _ = model._run_static(dev_imgs[i % n_img], im_info[0], lane=l)
            counts_host[i % counts_host.shape[0]].copy_(out["counts"], non_blocking=True)
        last_out[0] = out
        return out

    # end-to-end leg: the pipelined serving front end (upsnet_b200/pipeline.py).  Every step submits one PINNED HOST
    # image (H2D inside the timed region) and reads the previous step's results back to the host (D2H inside the timed
    # region); the copies of neighbouring images overlap the compute of the current one on separate streams.
    from upsnet_b200.pipeline import PipelinedEngine
    # depth = 2 x lanes staging slots: LANES images computing, the next LANES already copied in / the previous being copied out
    E2E_DEPTH = 2 * LANES
    engine = PipelinedEngine(model, im_info, depth=E2E_DEPTH, with_masks=True, lanes=LANES)   # every tensor of the reference's result dict
    pending = []

    def step_e2e(i):
        pending.append(engine.submit(host_imgs[i % n_img]))
        if len(pending) >= E2E_DEPTH:
            return engine.result(pending.pop(0))
        return None

    def drain_e2e():
        res = None
        while pending:
            res = engine.result(pending.pop(0))
        return res

    from upsnet_b200 import replicas

    def sync_all():
        replicas.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.STATS["launches"]
        cur = torch.cuda.current_stream(dev)
        e0.record()
        for ls in lane_streams:
            ls.wait_stream(cur)          # lanes start after e0 ...
        for i in range(steps):
            fn(i)
        if finish is not None:
            finish()          # host-waits for the last results: everything submitted is complete before e1
        for ls in lane_streams:
            cur.wait_stream(ls)          # ... and e1 is recorded after every lane has finished its images
        e1.record()
        sync_all()
        mine = e0.elapsed_time(e1)
        ms = replicas.max_over_ranks(mine, dev)   # slowest rank
        return ms, ops.STATS["launches"] - l0, replicas.all_ranks(mine, dev)

    for i in range(args.warmup):
        step_resident(i)
    for i in range(E2E_DEPTH + 2):
        step_e2e(i)
    drain_e2e()
    sampler = None
    if rank == 0 and not os.environ.get("UPSNET_BENCH_NO_SAMPLER"):
        sampler = NvmlSampler(local)
        if not sampler.ok:
            sampler = ClockSampler(local)
        sampler.start(); time.sleep(0.1)
    if not model._prepared:
        model.prepare()
    for i in range(2):
        step_graph(i)
    counts_host.zero_()
    ms, launches, per_rank = timed(step_graph, args.steps)
    assert int(counts_host[:args.steps, 0].min()) >= 1, "every image must yield at least the dummy detection"
    if args.dump_outputs and rank == 0:      # before the next leg replays the lane's graph over these buffers
        dump_outputs(last_out[0], args.dump_outputs)
    ms_e2e, _, per_rank_e2e = timed(step_e2e, args.steps, finish=drain_e2e)
    clocks = sampler.stop() if sampler else None
    h2d, d2h = engine.bytes_per_image()
    # Serving-format variant of the end-to-end leg (extra information, not the headline): the RAW uint8 HWC image goes up
    # (mean / pad on the device: upsnet_prep_image) and the unified 2-channel panoptic map of base_dataset.py:332-371 comes
    # back next to the detection tensors (upsnet_unified_pan_result) -- 6 + 10 MB over PCIe instead of 25 + 37 MB.
    e2e_compact = None
    if args.workload == "cityscapes" and not args.no_other_configs:
        try:
            raw_imgs = [torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(50 + s_)).pin_memory()
                        for s_ in range(n_img)]
            eng2 = PipelinedEngine(model, im_info, depth=E2E_DEPTH, with_masks=True, with_unified=True, lanes=LANES, label_maps=False)
            pend2 = []

            def step_c(i):
                pend2.append(eng2.submit(raw_imgs[i % n_img]))
                if len(pend2) >= E2E_DEPTH:
                    return eng2.result(pend2.pop(0))

            def drain_c():
                while pend2:
                    eng2.result(pend2.pop(0))
            for i in range(E2E_DEPTH + 2):
                step_c(i)
            drain_c()
            ms_c, _, _ = timed(step_c, args.steps, finish=drain_c)
            hb, db = eng2.bytes_per_image()
            e2e_compact = {"value": world * args.steps / (ms_c * 1e-3), "unit": "images/s", "h2d_bytes_per_step": hb,
                           "d2h_bytes_per_step": db, "api": "PipelinedEngine(raw uint8 HWC image in; with_unified=True, label_maps=False: pan_2ch uint8 map "
                           "(class, instance) + detection tensors + mask probabilities out)"}
            del eng2
        except Exception as exc:
            e2e_compact = {"error": repr(exc)[:200]}

    # ---- roofline leg: CUDA events around every C-ABI call of a few more steps ----
    ops.STATS["trace"] = []
    torch.cuda.synchronize()
    n_trace = min(3, args.steps)
    graph_flag, model.use_cuda_graph = model.use_cuda_graph, False   # per-call events need eager launches
    ovl_flag, model.overlap_heads = model.overlap_heads, False       # ... on ONE stream (no cross-stream contention)
    lvl_flag, model.fcn_head.overlap_levels = model.fcn_head.overlap_levels, False
    for i in range(n_trace):
        # gate: keep the GPU busy while the host enqueues the whole step, so that the event pairs bracket kernels that
        # run back to back (an eager step is host-bound: without the gate small kernels would be timed with launch gaps)
        torch.cuda._sleep(40_000_000)
        step_resident(i)
    torch.cuda.synchronize()
    model.use_cuda_graph = graph_flag
    model.overlap_heads = ovl_flag
    model.fcn_head.overlap_levels = lvl_flag
    trace, ops.STATS["trace"] = ops.STATS["trace"], None
    fam = {}
    for kind, a, b, work in trace:
        f = fam.setdefault(kind, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "calls": 0})
        f["ms"] += a.elapsed_time(b); f["calls"] += 1
        f["flops"] += work.get("flops", 0.0); f["bytes"] += work.get("bytes", 0.0)
    pk = peaks()
    layer_path = os.environ.get("UPSNET_LAYER_TABLE")
    if layer_path and rank == 0:      # per-layer table of the conv family (eager trace, CUDA events per call)
        per = {}
        for kind, a, b, work in trace:
            if "shape" in work:
                e = per.setdefault((kind, work["shape"]), [0, 0.0, work["algo_flops"], work["bytes"]])
                e[0] += 1; e[1] += a.elapsed_time(b)
        with open(layer_path, "w") as fh:
            fh.write("| kernel | layer shape | calls/step | ms/call | TFLOP/s | GB/s |\n|---|---|---:|---:|---:|---:|\n")
            for (kind, shape), (cnt, ms_, fl, by) in sorted(per.items(), key=lambda kv: -kv[1][1]):
                mc = ms_ / cnt
                fh.write("| %s | %s | %.1f | %.4f | %.1f | %.0f |\n" % (kind, shape, cnt / n_trace, mc, fl / mc / 1e9, by / mc / 1e6))
    tot_ms = sum(f["ms"] for f in fam.values())
    # dominant kernel = the dense-conv family (bf16: igemm_tma_kernel for all but a handful of launches)
    conv = {"ms": fam.get("conv2d", {"ms": 0})["ms"], "flops": fam.get("conv2d", {"flops": 0})["flops"],
            "calls": fam.get("conv2d", {"calls": 0})["calls"]}
    algo = sum(w.get("algo_flops", w.get("flops", 0.0)) for k_, _, _, w in trace if k_ == "conv2d")
    achieved = algo / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else 0.0   # ALGORITHMIC flops (x3 MMAs not counted)
    dcn_algo = sum(w.get("algo_flops", 0.0) for k_, _, _, w in trace if k_ == "dcn")
    kname = {"bf16": "igemm_tma_kernel (TMA-fed tcgen05 implicit GEMM; dense conv / FC family incl. stem)",
             "bf16x3": "igemm_tma2_kernel / igemm_tma_kernel on hi/lo bf16 pairs (TMA-fed tcgen05 implicit GEMM, 3 MMAs per "
                       "k-slice: hi*hi + lo*hi + hi*lo; 2-CTA cta_group::2 variant for tiles with >= 8 k-blocks, 1-CTA "
                       "otherwise; dense conv / FC family incl. the RGB stem)",
             "fp32": "igemm_simt_kernel (fp32 CUDA-core tiles)"}[args.precision]
    roofline = {"kernel": kname + ", precision=%s" % args.precision, "bound": "tensor",
                "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["tf_sustained"], "peak_source": pk["source"] + " (sustained bf16)",
                # dram__bytes_read.sum + dram__bytes_write.sum of ONE representative launch of the family under `ncu --set full`
                # (profiles/r2_pair_full.md: FPN / RPN 3x3 256->256 @256x512 on pairs, 136.7 MB read + 93.7 MB written against
                # algorithmic x + y = 268 MB: no re-reads from HBM); null for the other precisions (not captured)
                "traffic": 230.4e6 if args.precision == "bf16x3" else None,
                "traffic_launch": "FPN / RPN 3x3 256->256 @256x512 (154.6 GFLOP algorithmic, 268 MB algorithmic bytes)" if args.precision == "bf16x3" else None,
                "share_of_step": conv["ms"] / tot_ms if tot_ms else None,
                "avg_launch_ms": conv["ms"] / max(conv["calls"], 1),
                "flops_per_step": algo / n_trace, "mma_flops_per_step": conv["flops"] / n_trace,
                # executed tensor-core work (3 passes in bf16x3) against the same peak: how busy the tensor pipe is
                "mma_achieved": conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else 0.0,
                "mma_frac": (conv["flops"] / (conv["ms"] * 1e-3) / 1e12 / pk["tf_sustained"]) if conv["ms"] > 0 else 0.0,
                # `frac` counts ALGORITHMIC flops (2*P*Cout*Cin*k^2, one pass); the fp32-grade product of precision bf16x3 executes
                # three bf16 tensor-core passes per algorithmic flop, so frac <= 1/3 by construction -- mma_frac counts the passes
                "frac_ceiling": (1.0 / 3.0) if args.precision == "bf16x3" else 1.0,
                "families_ms_per_step": {k: round(v["ms"] / n_trace, 4) for k, v in sorted(fam.items())}}
    if "dcn" in fam and fam["dcn"]["ms"] > 0:
        roofline["dcn_tflops"] = dcn_algo / (fam["dcn"]["ms"] * 1e-3) / 1e12
        roofline["timing"] = "CUDA events around every C-ABI call of %d eager single-stream steps, GPU gated so kernels run back to back" % n_trace
    if "panoptic_head" in fam:
        f = fam["panoptic_head"]
        roofline["panoptic_head_gbs"] = f["bytes"] / (f["ms"] * 1e-3) / 1e9
        roofline["panoptic_head_frac_hbm"] = roofline["panoptic_head_gbs"] / pk["hbm_gbs"]

    # secondary figure in the same run: the single-pass bf16 configuration (bf16-level error: NOT the parity mode)
    other = None
    if args.precision == "bf16x3" and args.workload == "cityscapes":
        U.set_precision("bf16")
        for i in range(3):
            step_graph(i)
        ms3, _, _ = timed(step_graph, args.steps)
        other = {"precision": "bf16", "value": world * args.steps / (ms3 * 1e-3), "unit": "images/s",
                 "note": "single tcgen05 pass on bf16 activations: bf16-level error (tests hold it to 4e-2..8e-2), reported "
                         "for reference only -- the headline is the bf16x3 pair stream that meets 'fp32 logits within 1e-3'"}
        U.set_precision(args.precision)
    # The other BASELINE configurations, measured in the same (driver-run) process: configs[2] UPSNet-101-DCN at 800x1344
    # through the same engine entry, and configs[4] -- the panoptic head alone at 19x1024x2048 for n = 100..1000 instances.
    other_cfg = None
    if world == 1 and args.precision == "bf16x3" and args.workload == "cityscapes" and not args.no_other_configs:
        other_cfg = {}
        try:
            import numpy as np
            m3 = synthetic_model(UPSNetConfig.coco_r101_dcn(), depth=(3, 4, 23, 3), seed=0, device=dev)
            H3, W3 = 800, 1344
            imgs3 = [synthetic_input(H3, W3, seed=700 + s_)["data"].to(dev) for s_ in range(n_img)]
            info3 = synthetic_input(8, 8)["im_info"]; info3[0, :2] = (H3, W3)
            cnt3 = torch.zeros((16, 3), dtype=torch.int32).pin_memory()

            def step3(i):
                l = i % LANES
                with torch.cuda.stream(lane_streams[l]):
                    out, _ = m3._run_static(imgs3[i % n_img], info3[0], lane=l)
                    cnt3[i % 16].copy_(out["counts"], non_blocking=True)
            for i in range(2 * LANES):
                step3(i)
            n3 = args.steps
            ms_c3, _, _ = timed(step3, n3)
            other_cfg["configs[2] UPSNet-101-DCN COCO 800x1344 (padded from 1333), one image per step"] = {
                "value": n3 / (ms_c3 * 1e-3), "unit": "images/s", "ms_per_step": ms_c3 / n3, "precision": args.precision, "lanes": LANES,
                "detections_per_image": float(cnt3[:n3, 0].float().mean()),
                "parity": "tests/test_gpu_fullsize.py: res2-5, FPN, fcn_output <= 6e-5 relative vs the literal model at this size"}
            del m3, imgs3
            rng5 = np.random.default_rng(5)
            fcn5 = torch.randn(1, 19, 1024, 2048, device=dev) * 3
            sweep = {}
            for n5 in (100, 200, 500, 1000):
                c5 = np.stack([rng5.uniform(0, 2048, n5), rng5.uniform(0, 1024, n5)], 1)
                s5 = np.exp(rng5.uniform(np.log(16), np.log(512), (n5, 2)))
                b5 = np.concatenate([c5 - s5 / 2, c5 + s5 / 2], 1).astype(np.float32)
                b5[:, 0::2] = np.clip(b5[:, 0::2], 0, 2047); b5[:, 1::2] = np.clip(b5[:, 1::2], 0, 1023)
                a5 = [torch.from_numpy(v).to(dev) for v in (b5, (0.6 + 0.4 * (rng5.permutation(n5) + 1) / (n5 + 1)).astype(np.float32),
                                                             (rng5.standard_normal((n5, 1, 28, 28)) * 2).astype(np.float32),
                                                             rng5.integers(1, 9, n5).astype(np.int64))]
                nd5 = torch.tensor([n5], dtype=torch.int32, device=dev)
                run5 = lambda: U.panoptic_fuse(fcn5, a5[0], a5[1], a5[2], a5[3], 11, n_dev=nd5)
                run5(); run5(); torch.cuda.synchronize()
                e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0_.record()
                for _ in range(10):
                    run5()
                e1_.record(); torch.cuda.synchronize()
                sweep["n=%d" % n5] = round(e0_.elapsed_time(e1_) / 10, 4)
            other_cfg["configs[4] panoptic head (MaskRemoval + SegTerm + void/argmax) at 19x1024x2048, fp32 logits in HBM"] = {
                "ms_per_call": sweep, "unit": "ms", "parity": "tests/test_gpu_parity.py: bit-exact vs the oracle for n = 100..1000 at this size"}
            del fcn5
        except Exception as exc:      # the extra configurations must never cost the headline line
            other_cfg["error"] = repr(exc)[:300]
    if rank == 0:
        cpu, parity = None, None
        if world == 1 and not args.no_cpu_baseline and args.workload == "cityscapes":
            cpu, cpu_out = cpu_baseline_leg()
            parity = parity_block(model, cpu_out, dev)
        line = {"metric": METRIC if args.workload == "cityscapes" else "panoptic images/sec at 800x1344 (COCO, UPSNet-101-DCN)",
                "value": world * args.steps / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "fp32", "bf16x3": "bf16x3", "bf16": "bf16"}[args.precision],
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "parallelism": "replicas x%d (one image per GPU, no collective)" % world,
                           "l2": "no flush: each step streams >1 GB of activations (>> 126 MB L2) and rotates %d images" % n_img,
                           "weights": "random-init (upsnet_b200/synthetic.py), frozen BN folded",
                           "engine": "static shapes, device-side counts, CUDA graph replay=%s; value = sync-free engine entry "
                                     "(result sizes read back asynchronously), e2e = public PipelinedEngine API; %d engine lane(s): consecutive images "
                                     "run on independent graph instances / streams and overlap on the GPU, one image per step" % (bool(model.use_cuda_graph), LANES),
                           "lanes": LANES,
                           "detections_per_image": {"n_det": float(counts_host[:args.steps, 0].float().mean()),
                                                    "n_panoptic_candidates": float(counts_host[:args.steps, 1].float().mean()),
                                                    "n_kept": float(counts_host[:args.steps, 2].float().mean())}},
                "clocks": clocks,
                "e2e": {"value": world * args.steps / (ms_e2e * 1e-3), "unit": "images/s",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "upsnet_b200.pipeline.PipelinedEngine: pinned-host image in, host results out; H2D / "
                               "compute / D2H of neighbouring images overlap (%d staging slots, %d engine lanes)" % (E2E_DEPTH, LANES)},
                "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
                "secondary_mode": other, "other_configs": other_cfg, "e2e_raw_image_in": e2e_compact, "per_rank_ms": {"value": per_rank, "e2e": per_rank_e2e},
                "numa_cpus_bound": numa_cpus}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# --ops: per-operator table (BASELINE.md section 4): new kernel vs the reference's own CUDA kernel
# (oracle/_ref, when shipped) vs the CPU oracle, with achieved GB/s / TFLOP/s against the peaks.
# ------------------------------------------------------------------------------------------------
def run_ops(args):
    import numpy as np
    import torch
    import upsnet_b200 as U
    from oracle import oracle as O
    dev = torch.device("cuda", 0)
    torch.set_grad_enabled(False)       # operator table = inference kernels (modules switch to the autograd path otherwise)
    pk = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    try:
        ref = O.RefKernels()
    except Exception:
        ref = None

    def gpu_ms(fn, iters=20, warm=3):
        for _ in range(warm):
            fn()
        tot = 0.0
        for _ in range(iters):
            flush.zero_()                                   # L2 flush (256 MB > 126 MB L2)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        return tot / iters

    def cpu_ms(fn, reps=3):
        fn(); best = 1e30
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); best = min(best, time.perf_counter() - t0)
        return best * 1e3

    rows = []

    def row(op, cfg, ms, by=None, fl=None, ref_ms=None, cpu=None, err=None):
        r = {"op": op, "config": cfg, "b200_ms": round(ms, 5)}
        if by is not None:
            r["gbs"] = round(by / ms / 1e6, 1); r["frac_hbm"] = round(by / ms / 1e6 / pk["hbm_gbs"], 4)
        if fl is not None:
            r["tflops"] = round(fl / ms / 1e9, 2); r["frac_tensor"] = round(fl / ms / 1e9 / pk["tf_burst"], 4)
        if ref_ms is not None:
            r["ref_kernel_ms"] = round(ref_ms, 5)
        if cpu is not None:
            r["cpu_ms"] = round(cpu, 3); r["cpu_cores"] = os.cpu_count()
        if err is not None:
            r["max_abs_diff"] = float(err)
        rows.append(r); print(json.dumps(r), flush=True)

    rng = np.random.default_rng(0)
    torch.manual_seed(0)

    def rois_for(n, extent, smin, smax):
        c = rng.uniform(0, extent, (n, 2)); s = np.exp(rng.uniform(np.log(smin), np.log(smax), (n, 2)))
        return np.concatenate([np.zeros((n, 1)), np.clip(c - s / 2, 0, extent - 1), np.clip(c + s / 2, 0, extent - 1)], 1).astype(np.float32)

    # ---- config 1: ROIAlign 1x256x256x256, 32 boxes ----
    feat = torch.randn(1, 256, 256, 256, device=dev)
    feat_nhwc = feat.permute(0, 2, 3, 1).contiguous()
    r32 = rois_for(32, 1024, 16, 512); r32d = torch.from_numpy(r32).to(dev)
    for ph in (7, 14):
        want = O.roi_align(feat.cpu().numpy(), r32, ph, ph, 0.25)
        cpu = cpu_ms(lambda: O.roi_align(feat.cpu().numpy(), r32, ph, ph, 0.25))
        by = 4.0 * 32 * 256 * ph * ph * 2 + 20 * 32   # out + (<=) same amount of unique feature reads
        got = U.roi_align(feat, r32d, ph, ph, 0.25)
        rm = gpu_ms(lambda: ref.roi_align(feat, r32d, ph, ph, 0.25)) if ref else None
        row("roi_align nchw", "1x256x256x256, 32 rois, %dx%d" % (ph, ph), gpu_ms(lambda: U.roi_align(feat, r32d, ph, ph, 0.25)),
            by, None, rm, cpu, np.abs(got.cpu().numpy() - want).max())
        row("roi_align nhwc", "1x256x256x256, 32 rois, %dx%d" % (ph, ph),
            gpu_ms(lambda: U.roi_align(feat_nhwc, r32d, ph, ph, 0.25, layout="nhwc")), by)
    # RCNN case: 1000 rois over the 4 FPN levels of a 1024x2048 image
    feats = [torch.randn(1, 256, 256 >> l, 512 >> l, device=dev) for l in range(4)]
    feats_cl = [f.permute(0, 2, 3, 1).contiguous() for f in feats]
    r1k = rois_for(1000, 2048, 16, 600); r1k[:, 2::2] = np.clip(r1k[:, 2::2], 0, 1023); r1kd = torch.from_numpy(r1k).to(dev)
    by = 4.0 * 1000 * 256 * 49 * 2
    sc = [1 / 4., 1 / 8., 1 / 16., 1 / 32.]
    row("fpn_roi_align nchw", "P2..P5 of 1024x2048, 1000 rois, 7x7", gpu_ms(lambda: U.fpn_roi_align(feats, r1kd, 7, 7, sc)), by)
    row("fpn_roi_align nhwc", "P2..P5 of 1024x2048, 1000 rois, 7x7",
        gpu_ms(lambda: U.fpn_roi_align(feats_cl, r1kd, 7, 7, sc, layout="nhwc")), by)

    # ---- NMS ----
    def dets(n, extent):
        c = rng.uniform(0, extent, (n, 2)); s = np.exp(rng.uniform(np.log(16), np.log(256), (n, 2)))
        sc_ = np.sort((rng.permutation(n) + 1.0) / (n + 1))[::-1]
        return np.concatenate([c - s / 2, c + s / 2, sc_[:, None]], 1).astype(np.float32)
    for n, extent, thr in ((1000, 600, 0.7), (8000, 2048, 0.5)):
        d = dets(n, extent); bx = torch.from_numpy(d[:, :4].copy()).to(dev)
        seg = torch.tensor([0, n], dtype=torch.int32, device=dev)
        by = 20.0 * n + 8.0 * n * ((n + 63) // 64) / 2 + 4 * n
        cpu = cpu_ms(lambda: O.nms(d, thr))
        rm = None
        if ref:
            t0 = time.perf_counter(); ref.nms(d, thr); rm = (time.perf_counter() - t0) * 1e3
        row("nms (device resident)", "N=%d thresh %.1f" % (n, thr), gpu_ms(lambda: U.nms_segmented(bx, seg, n, thr)), by, None, rm, cpu)
    d5 = [dets(1000, 600) for _ in range(5)]
    bx5 = torch.from_numpy(np.concatenate(d5)[:, :4].copy()).to(dev)
    seg5 = torch.tensor([0, 1000, 2000, 3000, 4000, 5000], dtype=torch.int32, device=dev)
    row("nms segmented", "5 RPN levels x 1000, one launch pair", gpu_ms(lambda: U.nms_segmented(bx5, seg5, 1000, 0.7)),
        5 * (20.0 * 1000 + 8.0 * 1000 * 16 / 2 + 4000))

    # ---- DCN: semantic-head layer 1 at P2 (SURVEY a12) and the op-level v2 config ----
    x = torch.randn(1, 256, 256, 512, device=dev)
    w = torch.randn(128, 256, 3, 3, device=dev) / 48
    b = torch.randn(128, device=dev)
    off = torch.randn(1, 18, 256, 512, device=dev) * 2
    fl = 2.0 * 256 * 512 * 128 * 256 * 9
    by = 4.0 * (x.numel() + off.numel() + w.numel() + 128 * 256 * 512)
    rm = gpu_ms(lambda: ref.deform_conv(x, off, w, b, pad=1), iters=5) if ref else None
    base = U.deform_conv(x, off, w, b, 1, 1, 1, precision=0)
    row("dcn v1 fp32 simt", "FCN L1@P2 256->128 3x3, 256x512", gpu_ms(lambda: U.deform_conv(x, off, w, b, 1, 1, 1, precision=0), iters=5), by, fl, rm)
    for name, prec in (("bf16x3", 1), ("bf16", 2)):
        got = U.deform_conv(x, off, w, b, 1, 1, 1, precision=prec)
        row("dcn v1 tcgen05 " + name, "FCN L1@P2 256->128 3x3, 256x512",
            gpu_ms(lambda: U.deform_conv(x, off, w, b, 1, 1, 1, precision=prec)), by, fl, None, None,
            (got.float() - base).abs().max().item())
    x2 = torch.randn(2, 256, 50, 84, device=dev); om = torch.randn(2, 27, 50, 84, device=dev)
    m2 = U.ModulatedDeformConv(256, 256, 3, padding=1).to(dev)
    fl2 = 2.0 * 2 * 50 * 84 * 256 * 256 * 9
    for name in ("fp32", "bf16x3", "bf16"):
        U.set_precision(name)
        row("ModulatedDeformConv " + name, "x[2,256,50,84] offset_mask[2,27,50,84] w[256,256,3,3]", gpu_ms(lambda: m2(x2, om)), None, fl2)
    U.set_precision("fp32")

    # ---- dense conv: FPN output conv 3x3 256->256 at P2, and a res4 1x1 ----
    wc = torch.randn(256, 256, 3, 3, device=dev) / 48
    flc = 2.0 * 256 * 512 * 256 * 256 * 9
    basec = U.conv2d(x, wc, None, 1, 1, 1, precision=0)
    row("conv3x3 fp32 simt", "256->256 @256x512", gpu_ms(lambda: U.conv2d(x, wc, None, 1, 1, 1, precision=0), iters=5), None, flc)
    xcl = x.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    for name, prec in (("bf16x3", 1), ("bf16", 2)):
        got = U.conv2d(xcl, wc, None, 1, 1, 1, precision=prec)
        row("conv3x3 tcgen05 " + name, "256->256 @256x512", gpu_ms(lambda: U.conv2d(xcl, wc, None, 1, 1, 1, precision=prec)),
            None, flc, None, None, (got.float() - basec).abs().max().item())

    # ---- config 5: panoptic-head sweep at 1024x2048 ----
    fcn = (torch.randn(1, 19, H, W, device=dev) * 3)
    for n in (100, 200, 500, 1000):
        c = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n)], 1); s = np.exp(rng.uniform(np.log(16), np.log(512), (n, 2)))
        bxs = np.concatenate([c - s / 2, c + s / 2], 1).astype(np.float32)
        bxs[:, 0::2] = np.clip(bxs[:, 0::2], 0, W - 1); bxs[:, 1::2] = np.clip(bxs[:, 1::2], 0, H - 1)
        prob = (0.6 + 0.4 * (rng.permutation(n) + 1) / (n + 1)).astype(np.float32)
        ml = (rng.standard_normal((n, 1, 28, 28)) * 2).astype(np.float32)
        cls = rng.integers(1, 9, n).astype(np.int64)
        a = [torch.from_numpy(v).to(dev) for v in (bxs, prob, ml, cls)]
        by = 4.0 * 19 * H * W + 8.0 * H * W + n * (4 * 784 + 24)
        cpu = None
        if n == 100:
            fc = fcn[0].cpu().numpy()
            cpu = cpu_ms(lambda: O.panoptic_head(fc, bxs, prob, ml, cls, 11), reps=2)
        keep, _ = U.panoptic_fuse(fcn, a[0], a[1], a[2], a[3], 11)
        row("panoptic_head", "19x1024x2048, n=%d (kept %d)" % (n, keep.numel()),
            gpu_ms(lambda: U.panoptic_fuse(fcn, a[0], a[1], a[2], a[3], 11)), by, None, None, cpu)
    print(json.dumps({"ops_table": rows, "peaks": pk}), flush=True)


if __name__ == "__main__":
    if "--ops" in sys.argv:
        run_ops(None)
    else:
        main()
