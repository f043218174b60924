#!/usr/bin/env python
"""bench.py -- KITTI-shape scenes/sec of the full 3DSSD SA backbone (BASELINE.json metric, configs[1]).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (the reference arm, see below)

A "step" is one pass of the whole path -- backbone (layer1..layer4 of configs/kitti/3dssd/3dssd.yaml incl. the vote
layer) + detection head + decode + BEV NMS -- over one batch of 8 synthetic KITTI-shaped scenes [8,16384,4] per GPU
(weak scaling: the batch is sharded by scene, no data-path collective; ONE exchange of the per-scene detection blocks
ends a step, inside the step's CUDA graph: this library's peer-memory kernel, `--exchange nccl` for ncclAllGather).

value  : scenes/s, inputs resident in HBM.  Every step is one CUDA-graph replay; `--pipeline` (default 24) steps are in
         flight on separate streams with their own graphs and buffers (a step chains latency-bound sampling stages that
         keep a few SMs busy for milliseconds and short throughput-bound stages, so steps overlap).  Timing: after
         max(W, 2*pipeline) warm-up steps, `--brackets` (5) brackets of exactly K steps each, one CUDA-event pair per
         bracket, barrier + synchronize on both sides, L2 flushed before every step, max over ranks per bracket, MEDIAN
         bracket reported; ms_per_step = that bracket / K.
e2e    : the same brackets through the public API with HOST buffers: pinned H2D copy of the batch into the graph's
         input + the step + D2H read of the gathered detection blocks inside the timed region.
config.latency_ms_single_step: one step at a time (sync after each), the library's latency mode (SABackbone
         latency_mode=True: layer-1 FPS cut into resumable launches whose samples are consumed while it continues).
roofline: time-weighted tensor-pipe figure over ALL grouped-MLP kernels of one step (the kernels that dominate the
         step's SM-time), each timed live with CUDA events; roofline_fps: the layer-1 D-FPS chain (ns per round).
cpu_baseline: the CPU restatement (oracle/, fp32 BLAS MLP) on a bounded sample of the same workload.
--dump-outputs DIR: after the timed brackets, what the last timed step returned to its caller is written as DIR/<name>.npy
         (float32; integer outputs as float64): the per-layer points, features and sample indices of rank 0 and the
         detections of all ranks.  Inputs and weights are seeded, so two builds can be compared output for output.
clocks : sampled in-process through NVML from before the first bracket to after the last one (no nvidia-smi start-up
         inside a bracket); median / reasons are over the samples that fall inside timed brackets.

--impl reference: the reference's implementation of this path is CUDA (lib/utils/tf_ops/*_g.cu) -- it has no
CPU code for sampling/grouping (SURVEY.md finding 4).  The arm therefore runs the reference's OWN kernels,
compiled unmodified into oracle/_ref/libref_ops.so, on the same GPU, with PyTorch fp32 ops standing in
one-for-one for the TF stock ops (oracle/ref_layers.py) and the NMS on the CPU like tf.image.non_max_suppression;
if that library is absent it falls back to the CPU port.  Its cpu_baseline object carries the CPU port timing.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "KITTI-shape scenes/sec (B×16384 pts) full SA backbone, 1/2/4/8×B200"
UNIT = "scenes/s"
SCENES_PER_GPU = 8
NPOINTS = 16384
# the SAME string in both arms (the driver compares them)
WORKLOAD = ("configs[1]: full 3DSSD SA backbone (3dssd.yaml layer1-4 + vote) + detection head, decode and BEV NMS, "
            "synthetic KITTI 16384x4 clouds, batch 8 per GPU")
DTYPE = "bf16x3-split/f32-acc"   # fp32 operands split in two bf16 terms, 3 tcgen05 MMAs per product, fp32 accumulation


# ----------------------------------------------------------------------------------------------------------
# clocks: in-process NVML sampling thread (falls back to one long-lived nvidia-smi started at program start)
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index=0, period=0.05):
        self.index, self.period = index, period
        self.samples = []          # (t, sm_mhz, max_mhz, reason bits)
        self.windows = []          # (t0, t1) of timed brackets
        self.stop_flag = threading.Event()
        self.mode = None
        self.proc = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            try:
                q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                              "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                             stderr=subprocess.DEVNULL, text=True)
                self.mode = "nvidia-smi"
                self.thread = threading.Thread(target=self._poll_smi, daemon=True)
                self.thread.start()
            except OSError:
                self.mode = None
        return self

    def _poll_nvml(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = int(get_reasons(self.h))
                self.samples.append((time.perf_counter(), sm, self.max_mhz, bits))
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(self.period)

    def _poll_smi(self):
        names = [0x8, 0x40, 0x20, 0x4]
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm, mx = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            bits = 0
            for bit, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    bits |= bit
            self.samples.append((time.perf_counter(), sm, mx, bits))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        time.sleep(2.5 * self.period)
        self.stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in self.windows)]
        use = inside if inside else self.samples
        bits = 0
        for s in use:
            bits |= s[3]
        return {"sm_mhz": float(np.median([s[1] for s in use])) if use else None,
                "sm_max_mhz": max(s[2] for s in use) if use else None,
                "reasons": sorted(v for k, v in self.REASONS.items() if bits & k),
                "samples": len(use), "samples_total": len(self.samples), "source": self.mode,
                "note": "median over the samples taken inside the timed brackets (value and e2e)"}


# ----------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port on a bounded sample
# ----------------------------------------------------------------------------------------------------------
def cpu_baseline(arch, params, head_params, pts_np, max_scenes=2):
    """Times the CPU restatement of the whole step (oracle/, all host threads; MLP through numpy's fp32 BLAS instead of
    the double-precision checker loop; head + decode + NMS included) on the first `max_scenes` scenes of the workload."""
    from oracle import head as ohead
    from oracle import layers as olayers
    from oracle import ops as oops
    oops.build()
    cores = oops.get_threads()
    saved = oops.linear_bn_relu

    def fast_linear(x, w, bias=None, bn=None, relu=True):
        y = x.reshape(-1, x.shape[-1]) @ w
        if bias is not None:
            y = y + bias
        if bn is not None:
            g, be, mu, var = bn
            inv = g / np.sqrt(var + np.float32(1e-3))
            y = y * inv + (be - mu * inv)
        if relu:
            np.maximum(y, 0, out=y)
        return y.reshape(x.shape[:-1] + (w.shape[1],)).astype(np.float32, copy=False)

    oops.linear_bn_relu = fast_linear
    try:
        sample = np.ascontiguousarray(pts_np[:max_scenes])
        t0 = time.perf_counter()
        xyz_l, feat_l = olayers.backbone_forward(arch, sample, params, ffps_mode="matrix")[:2]
        boxes, score, _ = ohead.head_forward(xyz_l[-1], feat_l[-1], head_params)
        oops.bev_nms(boxes, score, 0.1, 100)
        dt = time.perf_counter() - t0
    finally:
        oops.linear_bn_relu = saved
    return {"value": sample.shape[0] / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d of the %d scenes of one step, backbone + head + decode + NMS, oracle/ C restatement + numpy fp32 BLAS MLP, %.1f s"
                      % (sample.shape[0], pts_np.shape[0], dt)}


def ncu_dram_bytes(name):
    """dram read+write bytes per launch from a committed ncu export (profiles/<name>), or None."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, seen = 0.0, 0
    for line in open(path):
        parts = line.split()
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and parts[2] in unit:
            tot += float(parts[1]) * unit[parts[2]]
            seen += 1
    return tot if seen == 2 else None


def nominal_mlp_flops(arch, in_channels, scenes, cfg):
    """2*B*M*K*sum(Cin*Cout) with UNPADDED channel counts over the grouped MLPs + aggregation convs of the SA layers
    (SURVEY.md 8d: what the reference computes, first conv in the grouped domain)."""
    ch = cfg.layer_channels(arch, in_channels)
    total = 0
    npts = [NPOINTS]
    for li, spec in enumerate(arch):
        radius, nsample, mlps, npoint, ltype, vote_idx, agg = spec[2], spec[3], spec[4], spec[8], spec[11], spec[14], spec[15]
        if ltype != "SA_Layer":
            npts.append(npts[spec[0][0]])
            continue
        cin = ch[spec[1][0]]
        if vote_idx != -1:
            m = npts[vote_idx]
        else:
            m = sum(2 * p if meth == "FS" else p for p, meth in zip(npoint, spec[7]))
        npts.append(m)
        if not isinstance(radius, list) or not radius:
            continue
        for k, mlp in zip(nsample, mlps):
            c = cin + 3
            for co in mlp:
                total += 2 * m * k * c * co
                c = co
        if agg not in (None, -1):
            total += 2 * m * sum(x[-1] for x in mlps) * agg
    return total * scenes


class MlpTimer:
    """Wraps the tensor-core MLP entry points of tf_ops for ONE eager step: a CUDA-event pair around every call and the
    bf16 MMA flops the call issues (3 per logical MMA, padded K/N as the kernel runs them)."""
    NAMES = ("linear_tc", "linear_tc_hoisted", "linear_tc_gather", "sa_mlp_fused", "sa_mlp_fused_hoisted")

    def __init__(self, torch, tf_ops):
        self.torch, self.tf_ops, self.rec, self.saved = torch, tf_ops, [], {}

    @staticmethod
    def _r16(x):
        return (int(x) + 15) // 16 * 16

    def _flops(self, name, a, kw):
        """Called from summary(), after the step has drained (a unit count is read back from the device)."""
        r16 = self._r16
        urows = None
        if kw.get("units") is not None:                 # unit-list route: 128-row tiles of 16 listed 8-row units
            urows = (int(kw["units"][0].item()) + 15) // 16 * 128
        if name == "linear_tc":
            hi, f = a[0], a[2]
            return 2.0 * (urows if urows is not None else hi.numel() // hi.shape[-1]) * f.kp * r16(f.cout)
        if name == "linear_tc_hoisted":
            idx, f = a[5], a[6]
            return 2.0 * (urows if urows is not None else idx.numel()) * f.kp * r16(f.cout)
        if name == "linear_tc_gather":
            idx, f = a[3], a[4]
            return 2.0 * idx.numel() * f.kp * r16(f.cout)
        stack = a[5] if name == "sa_mlp_fused" else a[7]
        idx = a[3] if name == "sa_mlp_fused" else a[5]
        rows = urows if urows is not None else idx.numel()
        k, tot = r16(stack.cin), 0.0
        for n in stack.nout:
            tot += 2.0 * rows * k * r16(n)
            k = r16(n)
        return tot

    def __enter__(self):
        for n in self.NAMES:
            fn = getattr(self.tf_ops, n)
            self.saved[n] = fn

            def wrap(*a, _fn=fn, _n=n, **kw):
                e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
                e0.record()
                r = _fn(*a, **kw)
                e1.record()
                self.rec.append((_n, e0, e1, a, kw))
                return r
            setattr(self.tf_ops, n, wrap)
        return self

    def __exit__(self, *exc):
        for n, fn in self.saved.items():
            setattr(self.tf_ops, n, fn)

    def summary(self):
        self.torch.cuda.synchronize()
        per = {}
        tot_ms = tot_fl = 0.0
        for n, e0, e1, a, kw in self.rec:
            fl = 3.0 * self._flops(n, a, kw)
            ms = e0.elapsed_time(e1)
            tot_ms += ms; tot_fl += fl
            d = per.setdefault(n, [0, 0.0, 0.0])
            d[0] += 1; d[1] += ms; d[2] += fl
        return tot_ms, tot_fl, {n: {"launches": d[0], "ms": d[1], "tflops_bf16_issued": d[2] / (d[1] * 1e-3) / 1e12 if d[1] else 0.0}
                                for n, d in per.items()}


# ----------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--brackets", type=int, default=5, help="timed brackets per leg; the median is reported")
    ap.add_argument("--ffps-mode", default="direct", choices=["direct", "matrix", "fused"])
    ap.add_argument("--mlp-mode", default="tc", choices=["tc", "fp32"])
    ap.add_argument("--gather-in-kernel", type=int, default=1, help="1: first conv of unfused SA scales gathers its operand itself")
    ap.add_argument("--hoist-first", type=int, default=2, help="first conv of an SA scale evaluated per point (hoisted), not per grouped row: 0 off, 1 layer-by-layer scales, 2 all")
    ap.add_argument("--no-graph", action="store_true", help="eager launches (for ncu captures)")
    ap.add_argument("--latency-mode", action="store_true", help="with --no-graph: run the latency-mode network (for ncu captures)")
    ap.add_argument("--pipeline", type=int, default=24, help="steps in flight (independent CUDA graphs on separate streams)")
    ap.add_argument("--fps-cluster", type=int, default=None,
                    help="CTAs per scene of the D-FPS kernels: 0 heuristic, >0 exact, <0 cap; default -4 when steps are pipelined (frees SMs), else 0")
    ap.add_argument("--fps-packet", action="store_true", help="experiment: lone D-FPS with the coordinates-in-packet kernel (small shared-memory footprint)")
    ap.add_argument("--fps-bucket", default="auto", choices=["auto", "on", "off"],
                    help="layer-1 D-FPS of the throughput step: auto/on = single-CTA kernel with spatial pruning, off = cluster kernel")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: the per-step all-gather as this library's peer-memory kernel (default) or as ncclAllGather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-scenes", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference" and int(os.environ.get("RANK", "0")) != 0:
        return                                   # under torchrun rank 0 alone runs the reference arm

    import torch
    pkg = importlib.import_module("3dssd_b200")
    synth = importlib.import_module("3dssd_b200.synth")
    if args.impl == "reference":
        rank, world, local = 0, int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    else:
        rank, world, local = pkg.dist.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local).start() if rank == 0 else None      # runs from here to the end of the last bracket
    arch = pkg.config.ARCH_3DSSD
    params = pkg.params.init_params(arch, 1, seed=0)
    head_params = pkg.params.init_head_params(pkg.config.layer_channels(arch, 1)[-1], seed=1)
    pts_np = synth.kitti_like(SCENES_PER_GPU, NPOINTS, seed=1000 + rank * SCENES_PER_GPU)

    if args.impl == "reference":
        return run_reference(args, torch, pkg, arch, params, head_params, pts_np, rank, world, dev, sampler)

    import torch.distributed as dist
    P = 1 if args.no_graph else max(1, args.pipeline)
    if args.fps_cluster is None:
        args.fps_cluster = -4 if P > 1 else 0
    # detection head + decode + GPU BEV-NMS produce the per-scene detection block that is gathered / copied to the host
    head = pkg.DetectionHead(params=head_params, device=dev)
    mk = dict(in_channels=1, device=dev, ffps_mode=args.ffps_mode, mlp_mode=args.mlp_mode, head=head,
              gather_in_kernel=bool(args.gather_in_kernel), hoist_first=args.hoist_first)
    net = pkg.SABackbone(arch, params, fps_cluster=args.fps_cluster, latency_mode=bool(args.no_graph and args.latency_mode),
                         fps_packet=args.fps_packet, fps_bucket={"auto": None, "on": True, "off": False}[args.fps_bucket], **mk)
    net_lat = pkg.SABackbone(arch, params, fps_cluster=0, latency_mode=True, **mk)
    pts = torch.from_numpy(pts_np).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    total_scenes = SCENES_PER_GPU * world

    # ---- one eager step: launches per step (counted at the ctypes boundary: every C-ABI call below launches exactly
    # one kernel) and the per-call times / issued flops of the tensor-core MLP kernels (roofline) -------------------
    counter = {"n": 0}
    L = pkg.lib()
    queries = ("ssd3d_version", "ssd3d_last_error", "ssd3d_fps_needs_temp", "ssd3d_fps_supports_rounds", "ssd3d_ffps_supported",
               "ssd3d_sa_fused_smem", "ssd3d_query_ball_point_workspace", "ssd3d_bn_train_workspace")   # host-only, no launch
    counted = [n for n in pkg.EXPORTS if n not in queries]
    originals = {n: getattr(L, n) for n in counted}

    class Counting:
        def __init__(self, name, fn):
            self.name, self.fn = name, fn

        def __call__(self, *a):
            n = 1
            if self.name == "ssd3d_query_ball_point_multi_ws" and (getattr(a[13], "value", None) or getattr(a[12], "value", None)):
                n = 2                                   # culled ball query: grid build + search; exhaustive + unit lists: search + list
            elif self.name == "ssd3d_bn_train":
                n = 3
            counter["n"] += n
            return self.fn(*a)

    gather0 = pkg.dist.DetectionGather(total_scenes, dev)
    for _ in range(2):
        out = net.forward(pts)
        net.detections(out[0], out[1], out=gather0.out())
    torch.cuda.synchronize()
    for n in counted:
        setattr(L, n, Counting(n, originals[n]))
    # the GPU is held busy while the host enqueues the whole step, so that each event pair brackets kernel time only (an
    # idle GPU would add the host's launch preparation -- tensor-map encoding, ctypes -- to every short kernel)
    torch.cuda._sleep(int(0.08 * 1.9e9))
    with MlpTimer(torch, pkg.tf_ops) as mt:
        out = net.forward(pts)
        net.detections(out[0], out[1], out=gather0.out())
    mlp_ms, mlp_flops, mlp_per = mt.summary()
    launches_per_step = counter["n"] + (1 if world > 1 else 0)                 # + the exchange (peer_allgather_kernel / ncclAllGather)
    for n in counted:
        setattr(L, n, originals[n])

    # ---- steps in flight: P independent step pipelines (own CUDA graph + static buffers + stream + communicator).
    streams = [torch.cuda.Stream(device=dev) for _ in range(P)]
    exchange = "none" if world == 1 else args.exchange
    gathers = None
    if exchange == "peer":
        # one symmetric allocation for all pipelines (+ the latency-mode graph), the exchange itself is a kernel of libssd3d
        try:
            probe = pkg.dist.DetectionGather(total_scenes, dev)
            arena = pkg.dist.PeerArena((P + 2) * pkg.dist.PeerArena.share_bytes(world, probe.slice_bytes), dev)
            gathers = [pkg.dist.PeerGather(total_scenes, dev, arena) for _ in range(P)]
            # cross-check against ncclAllGather once, eagerly: same bytes on every rank
            chk_p, chk_n = pkg.dist.PeerGather(total_scenes, dev, arena), pkg.dist.DetectionGather(total_scenes, dev)
            o = net.forward(pts)
            for g in (chk_p, chk_n):
                net.detections(o[0], o[1], out=g.out())
                g.gather()
            torch.cuda.synchronize()
            same = torch.tensor([int(torch.equal(chk_p.raw, chk_n.raw) and chk_p.timeouts() == 0)], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            if int(same.item()) != 1:
                raise RuntimeError("peer exchange disagrees with ncclAllGather")
        except Exception as e:  # noqa: BLE001 -- no symmetric memory on this box: fall back to NCCL, and say so
            sys.stderr.write("bench.py: peer-memory exchange unavailable (%s); using ncclAllGather\n" % str(e).splitlines()[0])
            exchange, gathers = "nccl", None
    groups = [dist.new_group(ranks=list(range(world))) if exchange == "nccl" else None for _ in range(P)]
    if gathers is None:
        gathers = [pkg.dist.DetectionGather(total_scenes, dev, group=groups[k]) for k in range(P)]
    runners = []
    gather_in_graph = True
    for k in range(P):
        if args.no_graph:
            static_in = pts.clone()

            def replay(points=None, static_in=static_in, g=gathers[k]):
                if points is not None:
                    static_in.copy_(points, non_blocking=True)
                o = net.forward(static_in)
                r = net.detections(o[0], o[1], out=g.out())
                g.gather()
                return o, r
            runners.append(replay)
        else:
            try:
                runners.append(net.capture(pts, gather=gathers[k]))
            except RuntimeError as e:                      # NCCL refused capture: gather eagerly after the replay instead
                if world == 1 or not gather_in_graph:
                    raise
                gather_in_graph = False
                sys.stderr.write("bench.py: all-gather could not be captured (%s); running it eagerly per step\n" % str(e).splitlines()[0])
                torch.cuda.synchronize()
                break
    if not gather_in_graph and not args.no_graph:
        runners = []
        for k in range(P):
            inner = net.capture(pts, gather=None)
            g = gathers[k]

            def replay(points=None, inner=inner, g=g):
                o, (blk, cnt) = inner(points)
                ob, oc = g.out()
                ob.copy_(blk, non_blocking=True); oc.copy_(cnt, non_blocking=True)
                g.gather()
                return o, (blk, cnt)
            runners.append(replay)
    main_s = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_in = torch.from_numpy(pts_np).pin_memory()
    host_out = [torch.empty((gathers[k].raw.numel(),), dtype=torch.uint8).pin_memory() for k in range(P)]

    last = {}

    def one_step(i, e2e):
        k = i % P
        last["k"], last["out"] = k, runners[k](host_in if e2e else None)      # e2e: pinned H2D into the graph's static input first
        if e2e:
            host_out[k].copy_(gathers[k].raw, non_blocking=True)   # all ranks' detection blocks + counts

    def bracket(nsteps, e2e, timed=True):
        """nsteps pipelined steps inside one CUDA-event pair; returns device ms (max over ranks)."""
        barrier()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        start.record(main_s)
        for s_ in streams:
            s_.wait_event(start)
        for i in range(nsteps):
            s_ = streams[i % P]
            with torch.cuda.stream(s_):
                flush.zero_()                                      # L2 flush before every step (inside the bracket)
                one_step(i, e2e)
        for s_ in streams:
            main_s.wait_stream(s_)
        end.record(main_s)
        barrier()
        t1 = time.perf_counter()
        ms = start.elapsed_time(end)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        if timed and sampler is not None:
            sampler.window(t0, t1)
        return ms

    warm = max(args.warmup, 2 * P)
    bracket(warm, False, timed=False)
    nsteps = args.steps
    val_ms = sorted(bracket(nsteps, False) for _ in range(max(1, args.brackets)))
    total_ms = val_ms[len(val_ms) // 2]

    # ---- e2e: host buffers through the public API ---------------------------------------------------------
    bracket(warm, True, timed=False)
    e2e_all = sorted(bracket(nsteps, True) for _ in range(max(1, args.brackets)))
    e2e_ms = e2e_all[len(e2e_all) // 2]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["out"][0], gathers[last["k"]].result())

    # ---- single-step latency: one step at a time, sync after each, latency-mode network --------------------
    lat_runner = None
    if not args.no_graph:
        lat_gather = None
        if gather_in_graph:
            lat_gather = pkg.dist.PeerGather(total_scenes, dev, arena) if exchange == "peer" else pkg.dist.DetectionGather(total_scenes, dev, group=groups[0])
        lat_runner = net_lat.capture(pts, gather=lat_gather)
    thr_runner = runners[0]

    def serial_latency(run, nrep):
        lat = []
        for _ in range(nrep):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            lat.append(e0.elapsed_time(e1))
        return float(np.median(lat[2:])) if len(lat) > 4 else float(np.median(lat))
    nlat = max(12, min(args.steps, 30))
    latency_thr_ms = serial_latency(thr_runner, nlat)
    latency_ms = serial_latency(lat_runner, nlat) if lat_runner is not None else latency_thr_ms

    # ---- the layer-1 D-FPS chain timed alone with events on its stream -------------------------------------
    xyz = pts[..., :3].contiguous()

    def time_fps(bucket):
        for _ in range(3):
            pkg.farthest_point_sample(4096, xyz, bucket_kernel=bucket)
        torch.cuda.synchronize()
        kev = []
        for _ in range(max(5, min(args.steps, 20))):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pkg.farthest_point_sample(4096, xyz, bucket_kernel=bucket)
            e1.record()
            kev.append((e0, e1))
        torch.cuda.synchronize()
        return float(np.mean([a.elapsed_time(b) for a, b in kev]))
    k_ms = time_fps(False)            # 8-CTA cluster kernel: the latency-mode step
    kb_ms = time_fps(True)            # single-CTA kernel with spatial pruning: the throughput step
    # the two kernels must pick the same samples on the bench's own scenes (reported, not assumed)
    fps_agree = bool(torch.equal(pkg.farthest_point_sample(4096, xyz, bucket_kernel=True),
                                 pkg.farthest_point_sample(4096, xyz, bucket_kernel=False)))

    if world > 1:
        t = torch.tensor([k_ms, mlp_ms, latency_ms, latency_thr_ms, kb_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        k_ms, mlp_ms, latency_ms, latency_thr_ms, kb_ms = (float(v) for v in t.tolist())

    if rank == 0:
        peaks = {}
        ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(ppath):
            peaks = json.load(open(ppath))
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        tc_peak = float(peaks.get("bf16_tflops", 1700.0))
        fps_bytes = SCENES_PER_GPU * (4096 - 1) * NPOINTS * 16          # B*(M-1)*N*(4c+4), SURVEY.md 8d
        scenes = SCENES_PER_GPU * world * nsteps
        nominal = nominal_mlp_flops(arch, 1, SCENES_PER_GPU, pkg.config)
        ach_tc = mlp_flops / (mlp_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": scenes / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / nsteps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": WORKLOAD, "scenes_per_gpu": SCENES_PER_GPU,
                       "global_batch": SCENES_PER_GPU * world, "points": NPOINTS, "parallelism": "scene-sharded dp%d" % world,
                       "ffps": args.ffps_mode, "mlp": args.mlp_mode, "cuda_graph": not args.no_graph,
                       "l2": "flushed (256 MiB write) before every timed step",
                       "steps_in_flight": P, "hbm_peak_allocated_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "fps_cluster": args.fps_cluster, "fps_l1_kernel": "cluster" if net.fps_bucket is False else "bucket (1 CTA per scene)", "fps_l1_kernels_agree": fps_agree, "allgather_in_graph": bool(gather_in_graph and not args.no_graph),
                       "exchange": {"peer": "libssd3d peer_allgather_kernel over NVLink peer memory (symmetric buffers), inside the step graph",
                                    "nccl": "ncclAllGather, one communicator per pipeline", "none": "single GPU"}[exchange],
                       "exchange_timeouts": sum(g.timeouts() for g in gathers) if exchange == "peer" else 0,
                       "latency_ms_single_step": latency_ms,
                       "latency_ms_single_step_throughput_graph": latency_thr_ms,
                       "latency_note": "one step at a time with a sync after each (as the reference arm runs): latency-mode "
                                       "graph (SABackbone latency_mode=True) / the throughput graph used for `value`",
                       "brackets": len(val_ms), "steps_per_bracket": nsteps, "warmup_effective": warm,
                       "bracket_ms": val_ms, "e2e_bracket_ms": e2e_all,
                       "timing": "median of %d brackets of %d steps; one CUDA-event pair per bracket "
                                 "(L2 flushes included), barrier + synchronize on both sides, max over ranks per bracket; every step is "
                                 "one CUDA-graph replay incl. the ncclAllGather, %d step pipelines on separate streams"
                                 % (len(val_ms), nsteps, P)},
            "e2e": {"value": scenes / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(host_in.numel() * 4), "d2h_bytes_per_step": int(host_out[0].numel())},
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": ach_tc, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach_tc / tc_peak,
                         "traffic": ncu_dram_bytes("r02_ncu_mlp_top.txt"),
                         "kernel": "time-weighted over ALL tensor-core MLP kernels of one step (%d launches: %s)"
                                   % (len(mt.rec), ", ".join("%s x%d" % (n, d["launches"]) for n, d in sorted(mlp_per.items()))),
                         "kernel_ms": mlp_ms, "per_kernel": mlp_per,
                         "algorithmic_gflop_per_step": nominal / 1e9,
                         "algorithmic_tflops_fp32_grade": nominal / (mlp_ms * 1e-3) / 1e12,
                         "note": "achieved = bf16 tcgen05 flops ISSUED (3 MMAs per fp32-grade product, padded K/N) summed over the step's "
                                 "MLP launches / the sum of their CUDA-event times (one eager step, each launch timed on its stream); "
                                 "peak = MEASURED_PEAKS.json bf16_tflops (burst: kernels timed one at a time)"
                                 + ("" if peaks else " [fallback 1700: file absent]")
                                 + "; algorithmic = 2*B*M*K*sum(Cin*Cout) unpadded incl. the hoisted first convs (SURVEY 8d), fp32-grade"},
            "roofline_fps": {"bound": "latency", "kernel": "fps3_direct_kernel (D-FPS layer 1, 16384->4096, B=8, 8 CTAs per scene: the latency-mode step), timed alone",
                             "throughput_kernel": {"kernel": "fps3_bucket_kernel (same sampling, ONE CTA per scene, spatial pruning: the throughput step)",
                                                   "kernel_ms": kb_ms, "ns_per_round": kb_ms * 1e6 / 4095, "sm_ms_per_batch": 8 * kb_ms,
                                                   "cluster_kernel_sm_ms_per_batch": 64 * k_ms},
                             "kernel_ms": k_ms, "rounds": 4095, "ns_per_round": k_ms * 1e6 / 4095,
                             "floor_ns_per_round": 271.0,
                             "floor_note": "critical path of one round at 1.965 GHz: 4 packed distance updates + compare chain (~60 cyc) "
                                           "+ 2 redux.sync (~50) + st.async DSMEM one-way + mbarrier wake-up (~180, B300_MICROARCH DSMEM "
                                           "latency) + LDS + 2 redux + LDS of the winner (~90) = ~533 cyc = 271 ns",
                             "effective_stream_gbs": fps_bytes / (k_ms * 1e-3) / 1e9, "hbm_peak_gbs": hbm_peak,
                             "effective_stream_frac": fps_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
                             "traffic": ncu_dram_bytes("r01_ncu_fps_l1.txt"),
                             "note": "effective-stream bytes B*(M-1)*N*16 = what the reference streams per round (SURVEY 8d); the kernel "
                                     "keeps them on chip (DRAM traffic ~1.6 MB), so this is a latency chain, not an HBM-bound kernel"},
        }
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(arch, params, head_params, pts_np, args.cpu_scenes)
        print(json.dumps(line))
    if world > 1:
        # Every number is out.  The captured step graphs hold NCCL kernels of their pipelines' communicators and NCCL's
        # communicator teardown waits for the graphs that captured it (destroy_process_group() hung here for the full time limit
        # of a 2-GPU run, after the JSON line was printed): meet at a barrier, then leave without the teardown.
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def dump_outputs(out_dir, forward_out, detections, limit_bytes=64 * 10 ** 6):
    """Writes a step's outputs as <out_dir>/<name>.npy: xyz_<l>, features_<l>, fps_idx_<l> per layer of the backbone
    (None entries skipped), detection_boxes [B,100,9] and detection_counts [B].  Floating outputs are float32, integer
    ones float64 (exact)."""
    arrays = {}
    for prefix, tensors in zip(("xyz", "features", "fps_idx"), forward_out):
        for i, t in enumerate(tensors):
            if t is not None:
                arrays["%s_%d" % (prefix, i)] = t
    arrays["detection_boxes"], arrays["detection_counts"] = detections
    arrays = {k: t.detach().cpu().numpy() for k, t in arrays.items()}
    arrays = {k: a.astype(np.float32 if a.dtype.kind == "f" else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit_bytes:
        raise SystemExit("bench.py: the step's outputs take %d bytes, more than the %d a dump may hold" % (total, limit_bytes))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_reference(args, torch, pkg, arch, params, head_params, pts_np, rank, world, dev, sampler):
    """Reference arm (see module docstring).  Under torchrun only rank 0 works."""
    if rank != 0:
        return
    from oracle import ref_ops
    cpu = cpu_baseline(arch, params, head_params, pts_np, args.cpu_scenes)
    if not ref_ops.available():
        line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": world,
                "steps": 1, "warmup": 0, "ms_per_step": 1e3 * SCENES_PER_GPU / cpu["value"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "reference_device": "CPU port (oracle/_ref not built)"},
                "cpu_baseline": cpu,
                "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    from oracle import ref_layers
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    pts = torch.from_numpy(pts_np).to(dev)
    cache = {}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def step():
        xyz_l, feat_l = ref_layers.backbone_forward(arch, pts, params, cache)
        return ref_layers.head_forward(xyz_l[-1], feat_l[-1], head_params, cache)   # ends with the CPU NMS (D2H sync)

    for _ in range(max(1, min(args.warmup, 3))):
        step()
    torch.cuda.synchronize()
    steps = args.steps
    tot = 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        step()
        torch.cuda.synchronize()
        tot += (time.perf_counter() - w0) * 1e3          # the step ends on the host (CPU NMS): wall clock around it
    if sampler is not None:
        sampler.window(t0, time.perf_counter())
    clocks = sampler.stop() if sampler else None
    val = SCENES_PER_GPU * steps / (tot * 1e-3)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": 1, "steps": steps,
            "warmup": args.warmup, "ms_per_step": tot / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "reference_device": "B200: the reference's own CUDA kernels (oracle/_ref/libref_ops.so, unmodified "
                                           "sources, nvcc -O2 sm_100) + PyTorch fp32 ops one-for-one for the TF stock ops + "
                                           "CPU NMS like tf.image.non_max_suppression; the reference has no CPU "
                                           "implementation of this path",
                       "l2": "flushed between timed steps",
                       "timing": "one step at a time; host wall clock around each step with a synchronize on both sides "
                                 "(the step ends on the host, in the NMS)"},
            "clocks": clocks,
            "cpu_baseline": cpu,
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
