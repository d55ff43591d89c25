#!/usr/bin/env python
"""Headline benchmark: pruned-INT8 ResNet-18 images/s at per-GPU batch 256 on N B200s
(BASELINE.json `metric`), one process per GPU, batch sharded data-parallel, weights replicated.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference's CPU fbgemm path on the host cores
    python bench.py ... --dump-outputs DIR   # also write the last timed step's logits to DIR/logits.npy

A step is one forward pass of the hot path over one synthetic batch per rank.  `value` is timed with
the inputs already resident in HBM; `e2e` goes through the reference-facing call with HOST buffers
(pinned), H2D and D2H copies inside the timed region.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

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

METRIC = "pruned-INT8 ResNet-18 images/s @bs256 per GPU (synthetic 3x224x224)"
WORKLOADS = {
    # name: (description, dtype tag)
    "int8_r18_pruned": ("distilled+pruned ResNet-18 [57,115,230,460] static INT8 PTQ (fbgemm) forward", "u8"),
    "fp16_r18_pruned": ("distilled+pruned ResNet-18 [57,115,230,460] FP16-cast forward", "f16"),
    "fp16_r50_teacher": ("ResNet-50 teacher FP16 forward", "f16"),
}


# ------------------------------------------------------------------------------------------ sharding helpers
def shard_bounds(total: int, rank: int, world: int):
    """Contiguous batch shard of `rank`: the path has no cross-sample op, so ranks never exchange data."""
    base, extra = divmod(total, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def gather_logits(local: torch.Tensor, total: int, rank: int, world: int):
    """Reporting-only collective: all ranks' logits on rank 0, in batch order."""
    import torch.distributed as dist
    if world == 1:
        return local
    sizes = [shard_bounds(total, r, world) for r in range(world)]
    biggest = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros((biggest,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad)
    return torch.cat([out[r][:hi - lo] for r, (lo, hi) in enumerate(sizes)])


def max_over_ranks(value: float, device) -> float:
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML poll every ~2 ms on a thread;
    falls back to `nvidia-smi -lms` when NVML is unavailable)."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index: int):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop, self._thread, self._proc, self._rows = threading.Event(), None, None, []

    def _poll_nvml(self, nv, handle):
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(handle))
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll_nvml, args=(nv, handle), daemon=True)
            self._thread.start()
            return
        except Exception:
            self._thread = None
        try:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            self._proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                           "--format=csv,noheader,nounits", "-lms", "20"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self._rows.append(l.strip()) for l in self._proc.stdout], daemon=True).start()
        except OSError:
            self._proc = None

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1.0)
        elif self._proc is not None:
            time.sleep(0.05)
            self._proc.terminate()
            for r in self._rows:
                f = [c.strip() for c in r.split(",")]
                try:
                    self.sm.append(float(f[0]))
                    self.max_mhz = float(f[1])
                except (ValueError, IndexError):
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ workloads
def build_reference_module(workload: str):
    """The artefact the reference hands to `model(images)` (synthetic weights: ievm_b200/synthetic.py)."""
    from ievm_b200 import synthetic as mf
    if workload == "int8_r18_pruned":
        return mf.static_quantize_fbgemm(mf.make_student(mf.PRUNED_WIDTHS))
    if workload == "fp16_r18_pruned":
        return mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS))
    return mf.cast_fp16(mf.make_teacher())


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """`--dump-outputs`: each array as <out_dir>/<name>.npy in float32, so that two builds (or the two arms) run with the
    same arguments can be compared output for output.  The inputs are seeded, hence identical from run to run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.detach().float().cpu().numpy())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic(workload: str):
    """DRAM bytes per launch of the dominant kernel from the newest committed ncu --set full capture of this workload
    (profiles/r0N_ncu_full_<workload>.json, written by scripts/ncu_traffic.py); None when no capture exists."""
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r0*_ncu_full_{workload}.json")))
    if not cands:
        return None, None
    d = json.load(open(cands[-1]))
    return d.get("conv_tc_dram_bytes_per_launch"), os.path.relpath(cands[-1], ROOT)


def network_roofline_ms(rows, tensor_tops: float, hbm_gbs: float) -> float:
    """SURVEY 8(d): sum over the engine's launches of max(2*MAC / tensor peak, compulsory bytes / HBM peak)."""
    return 1e3 * sum(max(2 * macs / (tensor_tops * 1e12), byt / (hbm_gbs * 1e9)) for _, macs, byt in rows)


def layer_table(net, n, fused_front=True):
    """Per LAUNCH of the engine: (name, algorithmic MACs, compulsory HBM bytes), real channels, every tensor read /
    written once.  With the fused front end (the product configuration) quantize + stem + max-pool are ONE row: the
    f32 / f16 input in, the pooled tensor out (SURVEY 8(d)'s 4.80 MB/img denominator); the residual is read once by
    the conv that fuses the add."""
    shape = {0: (net.in_h, net.in_w, net.in_c)}
    elem = 1 if net.dtype == 0 else 2
    in_elem = 4 if net.dtype == 0 else 2
    rows = []
    layers = list(net.layers)
    i = 0
    if fused_front and len(layers) >= 2 and layers[0].op == 0 and layers[0].in_tensor == 0 and layers[1].op == 1:
        st, mp = layers[0], layers[1]
        oh, ow = (net.in_h + 2 * st.pad - st.ksize) // st.stride + 1, (net.in_w + 2 * st.pad - st.ksize) // st.stride + 1
        ph, pw = (oh - 1) // 2 + 1, (ow - 1) // 2 + 1
        macs = n * oh * ow * st.cout * st.cin * st.ksize * st.ksize
        byt = n * (net.in_h * net.in_w * net.in_c * in_elem + ph * pw * st.cout * elem) + st.cout * st.cin * st.ksize ** 2 * elem
        shape[st.out_tensor] = (oh, ow, st.cout)
        shape[mp.out_tensor] = (ph, pw, st.cout)
        rows.append((st.name, macs, byt))
        i = 2
    elif net.dtype == 0:
        rows.append(("quantize_input", 0, n * net.in_h * net.in_w * net.in_c * (4 + 1)))
    for L in layers[i:]:
        ih, iw, ic = shape[L.in_tensor]
        if L.op == 0:
            oh = (ih + 2 * L.pad - L.ksize) // L.stride + 1
            ow = (iw + 2 * L.pad - L.ksize) // L.stride + 1
            macs = n * oh * ow * L.cout * L.cin * L.ksize * L.ksize
            byt = n * (ih * iw * ic + oh * ow * L.cout * (2 if L.res_tensor >= 0 else 1)) * elem + L.cout * L.cin * L.ksize ** 2 * elem
            if L.in_tensor == 0 and net.dtype == 1:
                byt = n * (ih * iw * ic + oh * ow * L.cout) * elem
            shape[L.out_tensor] = (oh, ow, L.cout)
        elif L.op == 1:
            oh, ow = (ih - 1) // 2 + 1, (iw - 1) // 2 + 1
            macs, byt = 0, n * (ih * iw + oh * ow) * ic * elem
            shape[L.out_tensor] = (oh, ow, ic)
        elif L.op == 3:
            macs, byt = 0, 3 * n * ih * iw * ic * elem
            shape[L.out_tensor] = (ih, iw, ic)
        else:
            macs, byt = n * L.cin * L.cout, n * (ih * iw * ic * elem + L.cout * 4) + L.cin * L.cout * elem
        rows.append((L.name, macs, byt))
    return rows


def _reference_forward_times(workload: str, bs: int, warmup: int, steps: int):
    """Seconds per forward of the reference's own CPU path (torch fbgemm / CPU half) on all host threads, and the logits
    of the last forward."""
    from ievm_b200 import synthetic as mf
    torch.set_num_threads(os.cpu_count() or 1)
    gm = build_reference_module(workload)
    if workload == "int8_r18_pruned":
        torch.backends.quantized.engine = "fbgemm"
    x = mf.synthetic_images(bs)
    if workload != "int8_r18_pruned":
        x = x.half()
    times = []
    with torch.no_grad():
        for _ in range(max(warmup, 1)):
            gm(x)
        for _ in range(steps):
            t0 = time.perf_counter()
            y = gm(x)
            times.append(time.perf_counter() - t0)
    return times, y


def cpu_baseline_sample(workload: str, bs: int):
    """The reference's own CPU path on the host cores, bounded sample: 1 warm-up + 5 forwards of the headline batch
    (about 1-2 s of CPU work at ~1.6 k img/s), median step."""
    times = sorted(_reference_forward_times(workload, bs, 1, 5)[0])
    med = times[len(times) // 2]
    return {"value": bs / med, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"median of {len(times)} forwards of batch {bs} through torch's fbgemm/ATen CPU path (the module "
                      f"quantization/engines.py:118 builds and :60 calls), {torch.get_num_threads()} threads"}


# ------------------------------------------------------------------------------------------ arms
def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, on the headline
    config (per-GPU batch).  Rank 0 alone runs it; no process group is created, the other ranks exit at once."""
    if rank != 0:
        return
    bs = args.ref_batch or args.batch
    times, y = _reference_forward_times(args.workload, bs, args.warmup, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": y})
    med = sorted(times)[len(times) // 2]
    val = bs / med
    desc, dtype = WORKLOADS[args.workload]
    cb = {"value": val, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
          "sample": f"median of {args.steps} forwards of batch {bs} through torch's fbgemm CPU operators -- the module "
                    f"quantization/engines.py:118 builds and :60 calls (mean {bs * len(times) / sum(times):.0f} img/s)"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * med, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": args.workload, "description": desc, "per_gpu_batch": args.batch,
                   "sample_batch": bs, "device": "host CPU", "torch_threads": torch.get_num_threads()},
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def _timed_steps(fn, steps, barrier, dev):
    """ms per call of fn over `steps` calls between CUDA events (barrier + synchronize on both sides, max over ranks)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1), dev) / steps


def _copy_ceiling(host_tensor, dev, barrier):
    """Raw cudaMemcpyAsync of the very pinned batch the end-to-end loop hands over, on this rank while every rank
    copies: the ceiling of the host-buffer path (GB/s, best of 5 after one warm-up, CUDA events, max over ranks)."""
    d = torch.empty_like(host_tensor, device=dev)
    best = None
    for rep in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        d.copy_(host_tensor, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = max_over_ranks(e0.elapsed_time(e1), dev)
        if rep:
            best = ms if best is None else min(best, ms)
    return host_tensor.numel() * host_tensor.element_size() / (best / 1e3) / 1e9


def run_b200(args, rank, world, local_rank):
    import ievm_b200
    from ievm_b200 import synthetic as mf

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    # stdout carries exactly one JSON line: whatever libraries print on file descriptor 1 (NCCL's version banner
    # among them) is sent to stderr for the duration of the run; the line itself goes to the saved descriptor
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    i8 = args.workload == "int8_r18_pruned"
    n = args.batch
    # the CPU baseline (rank 0, N = 1 only) runs BEFORE any GPU work exists, so nothing spins on a GPU while the host
    # cores are being timed
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_sample(args.workload, n)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    ref_mod = build_reference_module(args.workload)
    if i8:
        eng = ievm_b200.B200QuantizedResNet.from_converted(ref_mod, device=local_rank, max_batch=n)
    else:
        eng = ievm_b200.B200HalfResNet.from_half_module(ref_mod, device=local_rank, max_batch=n)
    x_host = mf.synthetic_images(n, seed=7 + rank)
    if not i8:
        x_host = x_host.half()
    x_host = x_host.pin_memory()
    x = x_host.to(dev)
    if args.graph:
        eng.set_option("use_graph", 1)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput -------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        y = eng(x)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        y = eng(x)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop() if rank == 0 else None
    value = world * n * args.steps / (ms / 1e3)
    ms_step = ms / args.steps

    # ---- end to end: the reference's evaluation loop (engines.py:52-63) over HOST batches -------------------
    # evaluate_accuracy(model, loader) hands one pinned CPU batch per iteration; the engine pipelines H2D, forward and the
    # D2H read of the logits (ievm_submit_*_host / ievm_wait).  Timed on the host clock around the whole loop.
    e2e_steps = max(4, min(args.steps, 12))
    labels_host = torch.randint(0, 6, (n,), generator=torch.Generator().manual_seed(5 + rank))
    loader = [(x_host, labels_host)] * e2e_steps

    def timed_eval(batches):
        ievm_b200.evaluate_accuracy(eng, batches[:2])
        barrier()
        t0 = time.perf_counter()
        ievm_b200.evaluate_accuracy(eng, batches)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        barrier()
        return max_over_ranks(dt, dev)

    e2e_s = timed_eval(loader)
    in_bytes = x_host.numel() * x_host.element_size()
    out_bytes = n * eng.net.num_classes * (4 if i8 else 2)
    h2d_gbs = _copy_ceiling(x_host, dev, barrier)
    e2e = {"value": world * n * e2e_steps / e2e_s, "unit": "images/s", "h2d_bytes_per_step": in_bytes,
           "d2h_bytes_per_step": out_bytes, "steps": e2e_steps,
           "how": "ievm_b200.evaluate_accuracy(engine, loader of pinned CPU batches) = the reference's loop "
                  "quantization/engines.py:52-63: per batch pinned H2D + forward + D2H of the logits, two batches in flight",
           "h2d_copy_gbs_per_rank": h2d_gbs,
           "copy_ceiling_images_per_s": world * h2d_gbs * 1e9 / (in_bytes / n),
           "frac_of_copy_ceiling": (world * n * e2e_steps / e2e_s) / (world * h2d_gbs * 1e9 / (in_bytes / n))}
    # the plain synchronous call y = model(cpu_tensor) (engines.py:60), one call at a time
    for _ in range(2):
        eng(x_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        y_host = eng(x_host)
    barrier()
    e2e["sync_call_images_per_s"] = world * n * e2e_steps / max_over_ranks(time.perf_counter() - t0, dev)

    # ---- the same loop fed with decoded 8-bit images (SURVEY 8(f)-1: ToTensor+Normalize+quantize fused) ----
    e2e_u8 = None
    if i8:
        xu8 = torch.randint(0, 256, (n, 224, 224, 3), dtype=torch.uint8,
                            generator=torch.Generator().manual_seed(11 + rank)).pin_memory()
        u8_s = timed_eval([(xu8, labels_host)] * e2e_steps)
        u8_gbs = _copy_ceiling(xu8, dev, barrier)
        u8_rate = world * n * e2e_steps / u8_s
        u8_ceiling = min(world * u8_gbs * 1e9 / (xu8.numel() / n), value)
        e2e_u8 = {"value": u8_rate, "unit": "images/s", "h2d_bytes_per_step": xu8.numel(), "d2h_bytes_per_step": out_bytes,
                  "steps": e2e_steps, "h2d_copy_gbs_per_rank": u8_gbs,
                  "ceiling_images_per_s": u8_ceiling, "frac_of_ceiling": u8_rate / u8_ceiling,
                  "how": "evaluate_accuracy over pinned uint8 NHWC batches -> ievm_submit_u8_host: the reference's ToTensor + "
                         "Normalize (dataset.py:16-18) + quantize_per_tensor fused into the front-end kernel via a 3x256 LUT; "
                         "ceiling = min(copy bandwidth, device-resident rate)"}
        # ... and with the dataset's native 200 x 200 images: Resize (Pillow bilinear) runs on the GPU as well
        x200 = torch.randint(0, 256, (n, 200, 200, 3), dtype=torch.uint8,
                             generator=torch.Generator().manual_seed(13 + rank)).pin_memory()
        r_s = timed_eval([(x200, labels_host)] * e2e_steps)
        e2e_u8["with_resize_from_200x200"] = {"value": world * n * e2e_steps / r_s, "unit": "images/s",
                                              "h2d_bytes_per_step": x200.numel(), "d2h_bytes_per_step": out_bytes}

    # ---- bs-1 latency (BASELINE.json: "p50 bs1 latency ms"; protocol of engines.py:26-34, synchronised) ----
    latency = None
    if rank == 0 and not args.no_latency:
        cls = ievm_b200.B200QuantizedResNet if i8 else ievm_b200.B200HalfResNet
        eng1 = (cls.from_converted if i8 else cls.from_half_module)(ref_mod, device=local_rank, max_batch=1)
        eng1.set_option("use_graph", 1)
        x1 = x[:1].contiguous()
        for _ in range(10):
            eng1(x1)
        torch.cuda.synchronize(dev)
        wall, devt = [], []
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.latency_runs):
            t0 = time.perf_counter()
            a.record()
            eng1(x1)
            b.record()
            torch.cuda.synchronize(dev)
            wall.append(1e3 * (time.perf_counter() - t0))
            devt.append(a.elapsed_time(b))
        wall.sort()
        devt.sort()
        launches1 = eng1.launches_per_forward
        w_bytes = sum(L.cout * L.cin * max(L.ksize, 1) ** 2 for L in eng1.net.layers if L.op in (0, 2)) * (1 if i8 else 2)
        hbm = peaks()["hbm_gbs"] * 1e9
        latency = {"p50_ms": wall[len(wall) // 2], "mean_ms": sum(wall) / len(wall), "p99_ms": wall[int(len(wall) * 0.99)],
                   "device_p50_ms": devt[len(devt) // 2], "runs": len(wall), "warmup": 10, "batch": 1,
                   "launches": launches1,
                   "floor_ms": 1e3 * w_bytes / hbm + launches1 * 0.0025,
                   "floor_how": f"weights {w_bytes / 1e6:.1f} MB / HBM peak + {launches1} dependent launches x 2.5 us "
                                f"(programmatic-dependent-launch gap between graph nodes)",
                   "how": "host wall clock around model(x1) + synchronize, input resident on device, CUDA graph replay"}
        eng1.close()

    # ---- logits gathered over NVLink for reporting; the gather must equal a single-GPU run of the same images ----
    gathered = gather_logits(y.float(), world * n, rank, world)
    if rank == 0 and args.dump_outputs:
        # the logits of the last timed step, every rank's shard in batch order (24 bytes per image)
        dump_outputs(args.dump_outputs, {"logits": gathered})
    gather_bitexact = None
    if world > 1:
        ok = True
        if rank == 0:
            for r in range(world):
                xr = mf.synthetic_images(n, seed=7 + r)
                if not i8:
                    xr = xr.half()
                yr = eng(xr.to(dev)).float()
                ok = ok and bool(torch.equal(yr, gathered[r * n:(r + 1) * n]))
        gather_bitexact = {"ok": ok, "how": "rank 0 recomputed every rank's shard (seed 7 + r) on its own GPU and compared "
                                            "with the all-gathered logits bit for bit (SURVEY 8(e))"}

    # ---- strong scaling (BASELINE.json configs[2]: batch sharded N/G per GPU) ----------------------------
    strong = None
    if i8 and not args.no_extra:
        strong = {}
        for gb in (256, 4096):
            per = gb // world
            if per < 1:
                continue
            e = eng if per <= n else ievm_b200.B200QuantizedResNet.from_converted(ref_mod, device=local_rank, max_batch=per)
            if e is not eng:
                e.set_option("use_graph", 1)
            lo, hi = shard_bounds(gb, rank, world)
            xs = mf.synthetic_images(hi - lo, seed=7).to(dev) if hi - lo <= 512 else \
                torch.randn(hi - lo, 3, 224, 224, generator=torch.Generator(device=dev).manual_seed(7), device=dev)
            for _ in range(3):
                e(xs)
            t_ms = _timed_steps(lambda: e(xs), 10, barrier, dev)
            strong[f"global_batch_{gb}"] = {"per_gpu_batch": hi - lo, "ms_per_step": t_ms, "images_per_s": gb / (t_ms / 1e3)}
            if e is not eng:
                e.close()
            del xs

    # ---- secondary workloads of BASELINE.json (configs[1], [3], [4]), a few steps each -------------------------------
    secondary = None
    if i8 and not args.no_extra:
        pk = peaks()
        secondary = {}

        def fp16_workload(name, module16, batch):
            e = ievm_b200.B200HalfResNet.from_half_module(module16, device=local_rank, max_batch=batch)
            e.set_option("use_graph", 1)
            xs = mf.synthetic_images(min(batch, 256), seed=7 + rank).half().to(dev)
            if batch > 256:
                xs = xs.repeat(batch // 256, 1, 1, 1)
            for _ in range(3):
                e(xs)
            t_ms = _timed_steps(lambda: e(xs), 6, barrier, dev)
            roof = network_roofline_ms(layer_table(e.net, batch), pk["bf16_tflops"], pk["hbm_gbs"])
            secondary[name] = {"per_gpu_batch": batch, "ms_per_step": t_ms, "images_per_s": world * batch / (t_ms / 1e3),
                               "network_roofline_ms": roof, "network_roofline_frac": roof / t_ms,
                               "launches": e.launches_per_forward}
            return e, xs

        es, xs16 = fp16_workload("fp16_r18_pruned_bs256", mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS)), 256)
        es.close()
        et, xt = fp16_workload("fp16_r50_teacher_bs256", mf.cast_fp16(mf.make_teacher()), 256)
        et.close()
        del xs16, xt
        # KD evaluation step: teacher + (unpruned) student forwards + the soft-target loss, global batch 512
        kb = max(512 // world, 1)
        teacher = ievm_b200.B200HalfResNet.from_half_module(mf.cast_fp16(mf.make_teacher()), device=local_rank, max_batch=kb)
        student = ievm_b200.B200HalfResNet.from_half_module(mf.cast_fp16(mf.make_student(mf.UNPRUNED_WIDTHS)),
                                                            device=local_rank, max_batch=kb)
        for e in (teacher, student):
            e.set_option("use_graph", 1)
        xk = mf.synthetic_images(min(kb, 256), seed=7 + rank).half().to(dev)
        if kb > 256:
            xk = xk.repeat(kb // 256, 1, 1, 1)
        yk = torch.randint(0, 6, (kb,), generator=torch.Generator().manual_seed(3 + rank)).to(dev)

        def kd_step():
            return ievm_b200.kd_eval_loss(student(xk), teacher(xk), yk, alpha=0.5, temperature=4.0)

        for _ in range(3):
            out4 = kd_step()
        t_ms = _timed_steps(kd_step, 6, barrier, dev)
        secondary["kd_eval_global_bs512"] = {"per_gpu_batch": kb, "ms_per_step": t_ms,
                                            "images_per_s": world * kb / (t_ms / 1e3), "loss": float(out4[0]),
                                            "how": "ResNet-50 teacher + unpruned ResNet-18 student FP16 forwards + "
                                                   "knowledge_distillation/train.py:47-57 loss kernel per step"}
        teacher.close()
        student.close()

    line = None
    if rank == 0:
        # ---- per-launch timing for the roofline of the dominant kernel ----------------------
        eng.set_option("use_graph", 0)
        eng.set_option("profile", 1)
        for _ in range(args.steps):
            eng(x)
        prof = eng.profile_read()
        eng.set_option("profile", 0)
        rows = layer_table(eng.net, n)
        table = {name: (macs, byt) for name, macs, byt in rows}
        pk = peaks()
        per_launch = {nm: t / c for nm, t, c in prof if c and t > 0}
        serial_ms = sum(per_launch.values())
        # per-launch CUDA events serialise the launches (no overlap between dependent kernels); inside the timed step the
        # CUDA graph overlaps prologues and tails, so the per-launch times are rescaled to sum to the measured step
        scale = ms_step / serial_ms if serial_ms else 1.0
        front = eng.net.layers[0].name
        tc = [nm for nm in per_launch if nm in table and table[nm][0] > 0 and nm != front and nm != "fc"]
        tc_ms = sum(per_launch[nm] for nm in tc) * scale
        tc_macs = sum(table[nm][0] for nm in tc)
        # a block's 1x1 downsample conv runs inside its first 3x3 conv's launch (conv_dual.cuh): its MACs and bytes are in
        # the sums above, its time is in that launch's
        index_of = {L.name: i for i, L in enumerate(eng.net.layers)}
        tc_launches = len({eng.layer_launch(index_of[nm]) for nm in tc})
        try:
            mma_peak = ievm_b200.measure_mma_peak("i8" if i8 else "f16", local_rank)
            peak_src = f"tcgen05.mma kind::{'i8' if i8 else 'f16'} M128xN256 instruction stream on all SMs, measured in this run " \
                       f"(ievm_probe_mma_peak, CUDA events)"
        except RuntimeError:
            mma_peak = None
        burst = (2 if i8 else 1) * pk["bf16_tflops"]
        tensor_peak = mma_peak or burst
        if mma_peak is None:
            peak_src = ("2 x " if i8 else "") + f"{pk['source']} burst cuBLAS bf16 (MEASURED_PEAKS.json)"
        achieved = 2 * tc_macs / (tc_ms / 1e3) / 1e12 if tc_ms else 0.0
        traffic, traffic_src = ncu_traffic(args.workload)
        roof_burst = network_roofline_ms(rows, burst, pk["hbm_gbs"])
        roof_meas = network_roofline_ms(rows, tensor_peak, pk["hbm_gbs"])
        roofline = {
            "kernel": "conv_tc_kernel / conv_dual_kernel / conv_s2_kernel (tcgen05 implicit GEMM, %d convs in %d launches/step)" % (len(tc), tc_launches),
            "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
            "frac": achieved / tensor_peak if tensor_peak else None, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src,
            "frac_of_2x_burst_bf16" if i8 else "frac_of_burst_bf16": achieved / burst,
            "algorithmic_flops_per_launch": 2 * tc_macs / max(tc_launches, 1),
            "algorithmic_bytes_per_launch": sum(table[nm][1] for nm in tc) / max(tc_launches, 1),
            "time_basis": "per-launch CUDA events (serialised, sum %.3f ms) rescaled by %.3f to the timed graph step "
                          "(%.3f ms)" % (serial_ms, scale, ms_step),
            "share_of_step": tc_ms / ms_step if ms_step else None,
            "per_launch_ms": {nm: round(t, 5) for nm, t in per_launch.items()},
            "per_launch_ms_in_step": {nm: round(t * scale, 5) for nm, t in per_launch.items()},
            "network_bytes_per_image": sum(b for _, _, b in rows) / n,
            "network_roofline_ms": roof_burst,
            "network_roofline_frac": roof_burst / ms_step,
            "network_roofline_how": "sum over the engine's launches of max(2*MAC / tensor peak, compulsory bytes / HBM "
                                    "peak) with the fused front end as ONE row (SURVEY 8(d)); tensor peak = "
                                    + ("2 x " if i8 else "") + "burst cuBLAS bf16, HBM = measured copy bandwidth",
            "network_roofline_ms_measured_mma_peak": roof_meas,
            "network_roofline_frac_measured_mma_peak": roof_meas / ms_step,
            "network_hbm_gbs": sum(b for _, _, b in rows) / (ms_step / 1e3) / 1e9,
        }
        desc, dtype = WORKLOADS[args.workload]
        line = {
            "metric": METRIC if i8 else f"{args.workload} images/s @bs{n} per GPU",
            "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": {"workload": args.workload, "description": desc, "per_gpu_batch": n, "global_batch": world * n,
                       "parallelism": f"dp{world} (batch sharded, weights replicated, no data-path collective)",
                       "l2_policy": "inputs larger than L2 (154 MB f32 batch vs 126 MB L2)" if i8 else
                                    "input batch 77 MB f16; activations stream through L2",
                       "cuda_graph": bool(args.graph)},
            "clocks": clocks, "e2e": e2e, "e2e_u8_pipeline": e2e_u8, "gpu_launches": eng.launches_per_forward * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "latency_bs1": latency,
            "strong_scaling": strong, "secondary": secondary, "gather_bitexact": gather_bitexact,
            "logits_checksum": float(gathered.double().sum().item()),
        }
    barrier()
    eng.close()
    if dist is not None:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    os.close(real_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="int8_r18_pruned", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch")
    ap.add_argument("--ref-batch", type=int, default=0, help="reference arm: images per CPU step (0 = the per-GPU batch)")
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip strong scaling and the secondary workloads")
    ap.add_argument("--latency-runs", type=int, default=300)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the logits of the last one to DIR/logits.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1 and args.impl == "b200":
            # convenience: re-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", str(29400 + os.getpid() % 500)] + sys.argv
            sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
