#!/usr/bin/env python
"""bench.py -- rays/sec of NeuRAD's volumetric-rendering hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one synthetic PandaSet-shaped time step (BASELINE config 2): 6 x 1920x1080
pinhole cameras traced at NeuRAD's render stride ([1::3,1::3] -> 6 x 230 400 rays) and one 64-beam x 1800-azimuth lidar
sweep (115 200 rays) = 1 497 600 traced rays, reference default grids / MLPs (random-init, tables U(-1,1), 0 actors).
Metric as the reference defines it: rays / time between device synchronisations (nerfstudio/pipelines/ad_pipeline.py:
198-208, 296-304); only TRACED rays are counted (the reference counts the 9x larger full-resolution pixel grid).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Two timed arms per run:
  value  device-resident inputs: ray generation + ONE `get_nff_outputs` launch pair over the whole time step.
  e2e    the metric through the reference-facing entry points with HOST buffers: per sensor
         `Cameras.generate_rays` -> `NeuRADModel.get_outputs_for_camera_ray_bundle` (render + lidar head + rgb CNN decoder),
         `NeuRADModel.get_outputs_for_lidar` for the sweep (points from pinned host memory), every output image / point
         cloud copied to pinned host memory by the copy engine on a second stream.  `NeuRADModel._bind()`, the Python of
         the API mirror and all host<->device copies are inside the timed region.

N > 1 (torchrun, one rank per GPU): rays shard with no data-path collective -- every rank renders its own time step
(weak scaling); the per-step gather of {features, depth, accumulation} is fused into the render epilogue (peer stores over
NVLink) and verified against an NCCL all-gather after the timed loops (`gather_verified`).  `config5_strong` adds one
strong-scaling point (8 388 608 rays split N ways).

Secondary keys of the N = 1 line: config3_actors (16 actors), config4_lidar_grid (128 x 2048 sweep with rolling shutter),
with_rgb_decoder, train_step (child process), gpu_torch_baseline (the reference's torch path = oracle port on CUDA),
cpu_baseline.
"""
from __future__ import annotations

import argparse
import contextlib
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def bind_to_gpu_numa_node(local_rank: int) -> dict:
    """Pin this process (and therefore its pinned-memory allocations: first touch, local policy) to the CPUs of the NUMA
    node the rank's GPU hangs off.  Must run BEFORE torch allocates pinned buffers.  Uses only sysfs + nvidia-smi."""
    info = {"node": None, "cpus": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=20).stdout
        bus = {int(a): b.strip().lower() for a, b in (ln.split(",") for ln in out.strip().splitlines())}
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[local_rank]) if visible and visible.split(",")[local_rank].isdigit() else local_rank
        bdf = bus[phys]
        bdf = bdf[-12:] if len(bdf) > 12 else bdf  # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return info
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"node": node, "cpus": len(allowed)}
    except Exception as e:  # no sysfs / not permitted: run unbound and say so
        info["error"] = f"{type(e).__name__}: {e}"[:120]
    return info


import torch  # noqa: E402

ALGO_BYTES_PER_RAY = 69_900  # SURVEY.md section 8(d) / BASELINE.md section 2: fp32 tables, no actor hits
CAM_RAYS = 640 * 360
WORKLOAD = "neurad-default config2: 6x1920x1080 pinhole @stride3 (6x230400 rays) + 64x1800 lidar (115200 rays), 0 actors"
STRONG_RAYS = 8_388_608  # BASELINE configs[4]
DUMP_ROWS = 131_072  # --dump-outputs keeps at most this many rows of an output (48-wide features: 25 MB)


def sample_rows(t: torch.Tensor):
    """`t` as [rows, channels] float32 numpy; above DUMP_ROWS rows, a fixed seeded sample of them (in order)."""
    t = t.reshape(-1, t.shape[-1])
    if t.shape[0] > DUMP_ROWS:
        keep = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
        t = t[keep.to(t.device)]
    return t.float().cpu().numpy()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


RENDER_KERNEL_SOURCES = ("b200nerf.cu", "nff_device.h", "nff_lane.h", "nff_params.h", "simt.h", "tc_mlp.cuh")


def kernel_sources_sha() -> str:
    """Hash of the CUDA sources the two timed render kernels are built from (the entry-point file and the headers they
    include; the decoder / training-operator headers are not part of them): profiles/traffic.json records the one it was
    captured at, and a capture of a different binary is not reported as this run's traffic."""
    h = hashlib.sha256()
    for name in RENDER_KERNEL_SOURCES:
        h.update(name.encode())
        h.update(open(os.path.join(ROOT, "neurad-studio_b200", "csrc", name), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- workload
def build_workload(cfg, frame: int):
    """Host-side description of one time step: 6 cameras + 1 lidar sweep at t = 1 + 0.5*frame seconds."""
    from neurad_studio_b200 import scene

    t = 1.0 + 0.5 * (frame % 12)
    return scene.pandaset_rig(time=t), scene.pandar64_scan(time=t, seed=frame)


class Step:
    """One time step on one rank: the device-resident arm (one fused launch pair) and the API / host-buffer arm."""

    def __init__(self, model, cfg, cams, scan, world, rank, gather="p2p"):
        from neurad_studio_b200.nerfstudio_api import Cameras, Lidars

        self.model, self.be, self.cfg, self.cams, self.scan = model, model._bind(), cfg, cams, scan
        be = self.be
        self.n_cam = len(cams) * CAM_RAYS
        self.n = self.n_cam + scan.points.shape[0]
        dev = be.device
        self.dev = dev
        self.world, self.rank = world, rank
        fdim = cfg.feature_dim
        # the gather buffers [world, n, w]: every rank's slice is written directly by the render kernel; with
        # gather="p2p" they live in symmetric memory and the kernel also stores each row into the peers' copies
        self.p2p = world > 1 and gather == "p2p"
        if self.p2p:
            from neurad_studio_b200.dist import PeerGatherBuffers

            self.pg = PeerGatherBuffers(self.n, fdim, dev)
            self.pg.bind(be)
            self.gather = self.pg.buf
            keys = ("features", "depth", "accumulation")
            self._dev_peers = {k: [int(p) for p in self.pg.hdl[k].buffer_ptrs] for k in keys}
        else:
            self.gather = {k: torch.empty(world, self.n, w, device=dev) for k, w in (("features", fdim), ("depth", 1), ("accumulation", 1))}
            self._dev_peers = None
        self.local = {k: torch.empty(self.n, 1, device=dev) for k in ("prop_depth_0", "prop_depth_1")}
        self.sensor = torch.cat([torch.full((CAM_RAYS,), c.sensor_idx, dtype=torch.long) for c in cams] +
                                [torch.full((scan.points.shape[0],), scan.sensor_idx, dtype=torch.long)]).to(dev)
        self.is_lidar = torch.cat([torch.zeros(self.n_cam, dtype=torch.uint8), torch.ones(scan.points.shape[0], dtype=torch.uint8)]).to(dev)
        self.rays = {k: torch.empty(self.n, w, device=dev) for k, w in (("origins", 3), ("directions", 3), ("pixel_area", 1), ("times", 1))}
        self.points_dev = scan.points.to(dev)
        self.kernel_events = []
        self.launches = 0
        # ---- API arm: the reference-facing objects and the pinned host buffers its outputs land in
        self.cameras = Cameras(cams, dev)
        self.lidars = Lidars([scan], dev)
        self.points_pinned = scan.points.clone().pin_memory()
        n_l = scan.points.shape[0]
        self.host_cam = [{"rgb": torch.empty(1080, 1920, 3).pin_memory(), "depth": torch.empty(360, 640, 1).pin_memory(),
                          "accumulation": torch.empty(360, 640, 1).pin_memory()} for _ in cams]
        self.host_lidar = {k: torch.empty(n_l, w).pin_memory() for k, w in (("depth", 1), ("intensity", 1), ("ray_drop_prob", 1), ("points", 3))}
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.e2e_launches = 0

    # ------------------------------------------------------------------------------------------ device-resident arm
    def _raygen(self, points):
        be = self.be
        off = 0
        for cam in self.cams:
            be.raygen_pinhole(cam, 1, 3, 1, 3, out={k: v[off:off + CAM_RAYS] for k, v in self.rays.items()})
            off += CAM_RAYS
            self.launches += 1
        be.raygen_lidar_points(self.scan, points, out={k: v[off:] for k, v in self.rays.items()})
        self.launches += 1

    def run_device(self, time_kernel: bool):
        """inputs already resident in HBM; one launch pair for the whole time step"""
        self._raygen(self.points_dev)
        rays = dict(self.rays, sensor_idx=self.sensor, is_lidar=self.is_lidar)
        out = {k: self.gather[k][self.rank] for k in self.gather}
        out.update(self.local)
        if self.p2p:
            self.be.set_peer_outputs(self._dev_peers, self_rank=self.rank, row_offset=self.rank * self.n)
        if time_kernel:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        self.be.render(rays, out=out, image_width=640)
        self.launches += 2  # nff_sample_lane_kernel + nff_shade_lane_kernel
        if time_kernel:
            e1.record()
            self.kernel_events.append((e0, e1))
        self._finish_gather()
        return out

    def _finish_gather(self):
        if self.world == 1:
            return
        if self.p2p:
            self.pg.barrier()  # rows were stored into every peer by the render kernel; only a barrier is left
        else:
            import torch.distributed as dist

            for k, buf in self.gather.items():
                dist.all_gather_into_tensor(buf.view(-1), buf[self.rank].reshape(-1))

    # ------------------------------------------------------------------------------------- API / host-buffer arm
    def _to_host(self, pairs, keep, ready=None):
        """D2H on the copy stream (copy engine) once the main stream (and, with a decoder stream, the image's decoder) has
        produced the tensors."""
        ev = torch.cuda.Event()
        ev.record()
        self.copy_stream.wait_event(ev)
        if ready is not None:
            self.copy_stream.wait_event(ready)
        with torch.cuda.stream(self.copy_stream):
            for dst, src in pairs:
                dst.copy_(src.reshape(dst.shape), non_blocking=True)
        keep.extend(src for _, src in pairs)  # alive until the step's final synchronisation

    def run_e2e(self):
        """The metric's own call sequence (ad_pipeline.py:198-208, 296-304), host buffers in and out."""
        model, be = self.model, self.be
        keep = []
        row = 0
        for i, host in enumerate(self.host_cam):
            if self.p2p:  # the image's rows also go to every peer's gather buffer from inside the render kernel
                be.set_peer_outputs(self._dev_peers, self_rank=self.rank, row_offset=self.rank * self.n + row)
            rb = self.cameras.generate_rays(camera_indices=i, keep_shape=True)
            out = model.get_outputs_for_camera_ray_bundle(rb)
            self._to_host([(host[k], out[k]) for k in host], keep, ready=out.get("rgb_ready"))
            row += CAM_RAYS
            self.e2e_launches += 1 + 5 + 3 + 10  # raygen, subsample copies, render pair + lidar head, decoder
        if self.p2p:
            be.set_peer_outputs(self._dev_peers, self_rank=self.rank, row_offset=self.rank * self.n + row)
        out, _ = model.get_outputs_for_lidar(self.lidars, {"lidar": self.points_pinned, "lidar_idx": 0})
        self._to_host([(self.host_lidar[k], out[k]) for k in self.host_lidar], keep)
        self.e2e_launches += 1 + 3
        self._finish_gather()
        if getattr(model, "decoder_stream", None) is not None:
            model.decoder_stream.synchronize()
        self.copy_stream.synchronize()
        torch.cuda.current_stream(self.dev).synchronize()
        return out

    @property
    def h2d_bytes(self):
        cam_desc = len(self.cams) * (12 + 4 + 3 + 4) * 4
        return self.points_pinned.numel() * 4 + cam_desc

    @property
    def d2h_bytes(self):
        return sum(t.numel() * 4 for h in self.host_cam for t in h.values()) + sum(t.numel() * 4 for t in self.host_lidar.values())


# ------------------------------------------------------------------------------------------ CPU / torch baselines
_BEST_THREADS = None
_ORACLE_PARAMS: dict = {}


def pick_cpu_threads(cfg):
    """The torch CPU path is made of small ops and stops scaling (or regresses) on many-core hosts: probe a few
    thread counts on a tiny sample and keep the fastest, so the baseline is the reference at its best."""
    global _BEST_THREADS
    if _BEST_THREADS is not None:
        return _BEST_THREADS
    ncpu = len(os.sched_getaffinity(0)) or 1
    cands = sorted({c for c in (ncpu, 64, 32, 16, 8) if c <= ncpu})
    best, best_v = cands[0], -1.0
    for c in cands:
        torch.set_num_threads(c)
        v, _, _ = oracle_rays_per_sec(cfg, 1024, _threads_fixed=True)
        if v > best_v:
            best, best_v = c, v
    _BEST_THREADS = best
    torch.set_num_threads(best)
    return best


def oracle_rays_per_sec(cfg, n_sample: int, repeats: int = 1, _threads_fixed: bool = False, device: str = "cpu", decoders: bool = True):
    """The reference's PyTorch path (oracle port) on a bounded sample of the same workload: ray generation,
    get_nff_outputs and -- like the metric's entry points -- the lidar head on all rays and the rgb CNN decoder on the camera
    rays (arranged as one image patch).  device="cpu": the host cores (the reference arm / cpu_baseline); device="cuda": the
    same torch code on the GPU (gpu_torch_baseline: the reference's own GPU path when tiny-cuda-nn is absent)."""
    from neurad_studio_b200 import scene
    from oracle import decoder_oracle as D
    from oracle import neurad_oracle as O
    from oracle.convert import to_oracle_cfg

    if device == "cpu" and not _threads_fixed:
        pick_cpu_threads(cfg)
    key = (str(device), cfg.n_actors)
    if key not in _ORACLE_PARAMS:  # parameters are built once, outside every timed region
        _ORACLE_PARAMS.clear()
        _ORACLE_PARAMS[key] = (scene.make_params(cfg, seed=1, beta=3.0, sdf_bias=0.6, device=device),
                               scene.make_rgb_decoder_params(seed=2, device=device))
    params, dec = _ORACLE_PARAMS[key]
    cams, scan = build_workload(cfg, 0)
    n_l = n_sample // 13  # same camera : lidar proportion as the workload (12 : 1)
    ph = 32
    pw = max(1, (n_sample - n_l) // ph)
    n_c = ph * pw  # the camera sample is one ph x pw patch of the stride-3 pixel grid
    cam = cams[0]
    ys, xs = torch.meshgrid(torch.arange(1, 1 + 3 * ph, 3), torch.arange(1, 1 + 3 * pw, 3), indexing="ij")
    coords = (torch.stack([ys, xs], -1).reshape(-1, 2) + 0.5).float().to(device)
    ocfg = to_oracle_cfg(cfg)
    best = None
    mv = lambda t: t.to(device) if torch.is_tensor(t) else t  # noqa: E731
    for _ in range(repeats):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        # torch.device(...) as a context: the oracle's factory calls (torch.linspace / zeros / full ...) land on `device`
        with torch.no_grad(), (torch.device(device) if device != "cpu" else contextlib.nullcontext()):
            rc = O.generate_rays_pinhole(mv(cam.c2w), cam.fx, cam.fy, cam.cx, cam.cy, cam.height, cam.width, coords, cam.time,
                                         mv(cam.velocity), cam.rolling_shutter_time, cam.time_to_center_pixel)
            rl = O.generate_rays_lidar_points(mv(scan.l2w), mv(scan.points[:n_l]), scan.time, mv(scan.velocity))
            rays = {k: torch.cat([rc[k], rl[k]]) for k in ("origins", "directions", "pixel_area", "times")}
            n = rays["origins"].shape[0]
            sensor = torch.cat([torch.zeros(n_c, 1, dtype=torch.long), torch.full((n_l, 1), 6)]).to(device)
            is_lidar = torch.cat([torch.zeros(n_c, 1, dtype=torch.bool), torch.ones(n_l, 1, dtype=torch.bool)]).to(device)
            out = O.nff_outputs(params, ocfg, rays["origins"], rays["directions"], rays["pixel_area"], rays["times"], sensor, is_lidar)
            if decoders:
                f = out["features"]
                h = f
                for i in range(3):  # lidar_decoder on every ray (intensity_for_cam=True, neurad.py:663-665)
                    h = torch.nn.functional.linear(h, params[f"lidar_decoder.layers.{i}.weight"], params[f"lidar_decoder.layers.{i}.bias"])
                    h = torch.relu(h) if i < 2 else h
                D.rgb_decoder(dec, f[:n_c].view(1, ph, pw, -1))
        if device != "cpu":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return n / best, n, best


_SAVED_STDOUT = None


def train_step_probe(timeout_s: float = 240.0) -> dict:
    """Secondary figure for SURVEY 8(f) row f2: one NFF TRAINING step (NeuRAD's 40 960 camera + 16 384 lidar ray batch
    through the module walk, both regularisers, loss.backward() through the hand-written backward operators), timed
    with CUDA events by tools/train_probe.py in a CHILD process after every headline measurement is finished."""
    cmd = [sys.executable, os.path.join(ROOT, "tools", "train_probe.py"), "--steps", "5", "--warmup", "2"]
    try:
        res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout_s)
        lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
        if res.returncode != 0 or not lines:
            tail = (res.stderr or res.stdout).strip().splitlines()[-3:]
            return {"error": f"tools/train_probe.py rc={res.returncode}: " + " | ".join(tail)[:400]}
        out = json.loads(lines[-1])
        out["note"] = "secondary figure (not the headline metric); measured in a child process after the timed arms"
        return out
    except Exception as e:  # time-out, missing file, malformed output ...
        return {"error": f"{type(e).__name__}: {e}"[:400]}


def _emit(line: dict):
    sys.stdout.flush()
    if _SAVED_STDOUT is not None:
        os.dup2(_SAVED_STDOUT, 1)
    print(json.dumps(line), flush=True)


def roofline_block(n_rays, kern_ms, kernel):
    peak, peak_src = measured_peaks()
    achieved = n_rays * ALGO_BYTES_PER_RAY / (kern_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "kernel": kernel, "kernel_ms": kern_ms, "peak_source": peak_src, "algorithmic_bytes_per_ray": ALGO_BYTES_PER_RAY}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=16384)
    ap.add_argument("--no-decoder", action="store_true", help="skip the extra 'with_rgb_decoder' measurement (N = 1)")
    ap.add_argument("--no-train", action="store_true", help="skip the extra 'train_step' measurement (N = 1, child process)")
    ap.add_argument("--no-extras", action="store_true", help="skip config3 / config4 / strong-scaling / torch-GPU baseline legs")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: p2p = render epilogue stores rows into every peer's buffer over NVLink (default); "
                         "nccl = all_gather_into_tensor after the render")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned to DIR/<name>.npy (float32): render_* the "
                         "device-resident arm's outputs, camera_* / lidar_* the API arm's host buffers (a fixed sample of "
                         f"{DUMP_ROWS} rows where an output has more); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3)
    # every rank (also the single one at N = 1: the API arm's pinned buffers and launch latencies otherwise depend on which
    # socket the scheduler happened to start the process on -- 38.7 vs 44.4 ms per e2e step between two fresh boxes)
    numa = bind_to_gpu_numa_node(local_rank) if args.impl == "b200" else {"node": None, "cpus": None}

    import neurad_studio_b200 as nsb

    cfg = nsb.NeuRADConfig(n_actors=0)
    base = {
        "metric": "rays/sec (camera+lidar)", "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_step_per_gpu": 6 * CAM_RAYS + 115200, "tables": "fp32, main 8x2^22x4 + proposal 6x2^20x1 (U(-1,1))",
                   "l2": "inputs larger than L2 (560 MB of tables, 300 MB of outputs per step); no explicit flush", "kernel": "ray-per-lane, 2-D tile walk (image_width=640), tcgen05 3xTF32 MLPs", "parallelism": f"ray-shard dp{world}" + ("" if world == 1 else f", gather={args.gather}")},
    }

    if args.impl == "reference":
        # the reference's own (PyTorch, CPU) implementation of the path = the oracle port, on the host cores, doing what the
        # b200 arm's e2e does per ray: ray generation, get_nff_outputs, lidar head, rgb decoder on the camera rays
        if rank != 0:
            return
        n_sample = max(2048, args.cpu_sample // 4)
        for _ in range(min(args.warmup, 1)):
            oracle_rays_per_sec(cfg, n_sample)
        t0 = time.perf_counter()
        tot = 0
        for _ in range(args.steps):
            _, n, _ = oracle_rays_per_sec(cfg, n_sample)
            tot += n
        dt = time.perf_counter() - t0
        v = tot / dt
        line = dict(base, impl="reference", value=v, ms_per_step=dt / args.steps * 1e3, n_gpus=world,
                    cpu_baseline={"value": v, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
                                  "sample": f"{n_sample} rays/step of the same workload (12:1 camera:lidar; render + lidar head + rgb decoder), oracle port of the reference torch path"},
                    e2e={"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, gpu_launches=0)
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        # NCCL / c10d print a version banner on stdout at first use; rank 0 must print ONE JSON line, so stdout is
        # pointed at stderr until the result line is written (restored in _emit)
        sys.stdout.flush()
        global _SAVED_STDOUT
        _SAVED_STDOUT = os.dup(1)
        os.dup2(2, 1)
        import datetime

        # a mis-ordered collective or a wedged kernel should cost minutes, not NCCL's 10-minute default plus its debug dump
        os.environ.setdefault("TORCH_NCCL_DUMP_ON_TIMEOUT", "0")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    from neurad_studio_b200 import scene
    from neurad_studio_b200.nerfstudio_api import NeuRADModel

    # the model as a user holds it: the API mirror's NeuRADModel with the reference's parameter names on the device
    params = scene.make_params(cfg, seed=1, beta=3.0, sdf_bias=0.6, device=dev)
    model = NeuRADModel(cfg)
    model.load_reference_state_dict(params)
    model.rgb_decoder.load_state_dict({k[len("rgb_decoder."):]: v for k, v in scene.make_rgb_decoder_params(seed=2).items()}, strict=False)
    model = model.to(dev).eval()
    del params
    be = model._bind()
    cams, scan = build_workload(cfg, rank)
    step = Step(model, cfg, cams, scan, world, rank, args.gather)

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        step.run_device(False)
        step.run_e2e()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    step.launches = 0
    ms = timed(lambda: step.run_device(True), args.steps)
    dump = {}
    if args.dump_outputs and rank == 0:
        dump = {f"render_{k}": sample_rows(v) for k, v in dict({k: b[rank] for k, b in step.gather.items()}, **step.local).items()}
    launches = step.launches // args.steps
    kern_ms = sorted(a.elapsed_time(b) for a, b in step.kernel_events)
    kern_ms = sum(kern_ms) / len(kern_ms)
    step.e2e_launches = 0
    # B200_E2E_DECODER_STREAM=1: the API arm pipelines image i's rgb decoder (side stream) under image i + 1's render
    # (NeuRADModel.set_decoder_stream; +2 % in back-to-back A/B runs).  Off by default: two of three full bench runs with it
    # showed a much slower e2e arm (44 / 61 ms per step instead of 38; the single-stream arm never did), not understood yet.
    dec_stream = os.environ.get("B200_E2E_DECODER_STREAM", "0") != "0"
    if dec_stream:
        model.set_decoder_stream(torch.cuda.Stream(device=dev))
    ms_e2e = timed(step.run_e2e, args.steps)
    if args.dump_outputs and rank == 0:
        dump.update({f"camera_{k}": sample_rows(torch.stack([h[k] for h in step.host_cam])) for k in step.host_cam[0]})
        dump.update({f"lidar_{k}": sample_rows(v) for k, v in step.host_lidar.items()})
    e2e_launches = step.e2e_launches // args.steps
    # the host buffers the e2e arm filled must hold what the API returns on the device (last image + the sweep re-rendered)
    if step.p2p:
        be.set_peer_outputs(None)  # the check re-renders locally only (run_device / run_e2e bind their own row offsets)
    with torch.no_grad():
        chk = model.get_outputs_for_camera_ray_bundle(step.cameras.generate_rays(len(cams) - 1))
        chk_l, _ = model.get_outputs_for_lidar(step.lidars, {"lidar": step.points_pinned, "lidar_idx": 0})
    torch.cuda.synchronize()
    model.set_decoder_stream(None)
    e2e_ok = all(torch.equal(step.host_cam[-1][k], chk[k].cpu().reshape(step.host_cam[-1][k].shape)) for k in step.host_cam[-1]) and \
        all(torch.equal(step.host_lidar[k], chk_l[k].cpu().reshape(step.host_lidar[k].shape)) for k in step.host_lidar)
    # multi-GPU: every peer's slice of the fused gather against an NCCL all-gather of the local slices
    gather_ok = None
    if world > 1 and step.p2p:
        import torch.distributed as dist

        step.run_device(False)
        barrier()
        gather_ok = True
        for k, buf in step.gather.items():
            ref = torch.empty_like(buf)
            dist.all_gather_into_tensor(ref.view(-1), buf[rank].reshape(-1).clone())
            gather_ok = gather_ok and bool(torch.equal(ref, buf))
        t = torch.tensor([1.0 if gather_ok else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        gather_ok = bool(t.item() == 1.0)
    # strong-scaling point (BASELINE configs[4]): one 8 388 608-ray batch, contiguous 1/N shards, fused gather
    strong = None
    if not args.no_extras:
        per = STRONG_RAYS // world
        reps = -(-per // step.n)
        big = {k: torch.cat([v] * reps)[:per].contiguous() for k, v in dict(step.rays, sensor_idx=step.sensor[:, None], is_lidar=step.is_lidar[:, None]).items()}
        big["sensor_idx"], big["is_lidar"] = big["sensor_idx"].reshape(-1), big["is_lidar"].reshape(-1)
        if world > 1 and step.p2p:
            from neurad_studio_b200.dist import PeerGatherBuffers

            del step.pg, step.gather  # symmetric memory of the weak-scaling arm
            pg = PeerGatherBuffers(per, cfg.feature_dim, dev)
            pg.bind(be)
            ptrs = {k: [int(p) for p in pg.hdl[k].buffer_ptrs] for k in ("features", "depth", "accumulation")}
            be.set_peer_outputs(ptrs, self_rank=rank, row_offset=rank * per)
            sout = {k: pg.buf[k][rank] for k in pg.buf}
        else:
            be.set_peer_outputs(None)
            pg = None
            sout = {k: torch.empty(per, w, device=dev) for k, w in (("features", cfg.feature_dim), ("depth", 1), ("accumulation", 1))}
        sout.update({k: torch.empty(per, 1, device=dev) for k in ("prop_depth_0", "prop_depth_1")})

        def run_strong():
            be.render(big, out=sout)
            if pg is not None:
                pg.barrier()

        for _ in range(2):
            run_strong()
        ms_s = timed(run_strong, args.steps)
        strong = {"rays_total": per * world, "rays_per_gpu": per, "ms_per_batch": ms_s / args.steps, "value": per * world / (ms_s / args.steps * 1e-3),
                  "unit": "rays/s", "scaling": "strong", "what": "BASELINE configs[4]: one 8 388 608-ray batch (config-2 rays repeated), contiguous 1/N shards, fused peer-store gather"}
        be.set_peer_outputs(None)
        del big, sout
    # (ii) of SURVEY 8(d): the device-resident step followed by the camera rgb decoder on the six rendered feature images
    dec_line = None
    if world == 1 and not args.no_decoder:
        n_cams = len(cams)
        rgb = torch.empty(n_cams, 1080, 1920, 3, device=dev)
        dec_events = []
        be.set_rgb_decoder(model.rgb_decoder.state_dict(), prefix="", bn_eps=model.rgb_decoder[2].main_branch[1].eps)

        def run_with_decoder():
            out = step.run_device(False)
            feats = out["features"][: step.n_cam].view(n_cams, 360, 640, -1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            be.rgb_decode(feats, out=rgb)
            e1.record()
            dec_events.append((e0, e1))

        for _ in range(2):
            run_with_decoder()
        dec_events.clear()
        ms_dec = timed(run_with_decoder, args.steps)
        be.check_status()
        d_ms = sorted(a.elapsed_time(b) for a, b in dec_events)
        d_ms = sum(d_ms) / len(d_ms)
        mac_per_ray = 48 * 32 + 4 * 50176 + 32 * 288 + 9 * (4 * 50176 + 3 * 32)
        tf = 2.0 * mac_per_ray * step.n_cam / (d_ms * 1e-3) / 1e12
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        tpeak = float(peaks.get("bf16_tflops_sustained", 1443.2))
        dec_line = {"value": step.n * args.steps / (ms_dec * 1e-3), "unit": "rays/s", "ms_per_step": ms_dec / args.steps,
                    "decoder_ms": d_ms, "decoder_camera_rays_per_s": step.n_cam / (d_ms * 1e-3), "gpu_launches_decoder": 10,
                    "roofline": {"bound": "tensor", "achieved": tf, "executed": 3 * tf, "peak": tpeak, "unit": "TFLOP/s",
                                 "frac": tf / tpeak, "frac_executed": 3 * tf / tpeak,
                                 "note": "achieved = algorithmic 4.04 MFLOP/camera ray; executed = 3x (bf16 hi/lo split: three MMAs per product for fp32-level accuracy); peak = measured sustained dense bf16"},
                    "what": "render step + NeuRADModel.rgb_decoder on the 6 feature images (6x360x640x48 -> 6x1080x1920x3 rgb)"}
    # BASELINE configs[2] / configs[3]: secondary legs with the same roofline block, N = 1
    extras = {}
    if world == 1 and not args.no_extras:
        extras = secondary_legs(be, cfg, dev, args.steps, timed)
    clocks = sampler.stop() if rank == 0 else None
    rays_total = step.n * world * args.steps
    value = rays_total / (ms * 1e-3)
    e2e_value = rays_total / (ms_e2e * 1e-3)
    if rank != 0:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()
        return
    roof = roofline_block(step.n, kern_ms, "nff_sample_lane_kernel + nff_shade_lane_kernel (one render)")
    roof["bound_note"] = ("HBM is the CONTRACTUAL bound (algorithmic gather bytes / measured copy bandwidth); physically the pair is "
                          "issue-bound: L1/L2 absorb ~94 % of the gathers (traffic << algorithmic bytes), see `limiter`")
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        tj = json.load(open(traffic_file))
        if tj.get("kernel_sources_sha") == kernel_sources_sha():
            roof["traffic"] = tj.get("dram_bytes_per_launch")
            roof["limiter"] = tj.get("limiter")
            roof["traffic_source"] = tj.get("source")
        else:
            roof["traffic_source"] = "profiles/traffic.json was captured for other kernel sources (sha mismatch): not reported"
    line = dict(base, value=value, ms_per_step=ms / args.steps, clocks=clocks, gpu_launches=launches,
                e2e={"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": step.h2d_bytes, "d2h_bytes_per_step": step.d2h_bytes,
                     "ms_per_step": ms_e2e / args.steps, "host_buffers_verified": bool(e2e_ok), "gpu_launches": e2e_launches,
                     "decoder_stream": dec_stream,
                     "how": "per sensor through the API mirror, as pipelines/ad_pipeline.py:198-208,296-304 does: Cameras.generate_rays -> "
                            "NeuRADModel.get_outputs_for_camera_ray_bundle (render + lidar head + rgb CNN decoder), NeuRADModel.get_outputs_for_lidar "
                            "(sweep points from pinned host memory); rgb / depth / accumulation images and the lidar outputs copied to pinned host "
                            "memory by the copy engine on a second stream; with decoder_stream the rgb decoder of image i runs on a side stream under the render "
                            "of image i + 1 (NeuRADModel.set_decoder_stream); _bind() and all Python inside the timed region"},
                roofline=roof, numa=numa)
    if gather_ok is not None:
        line["gather_verified"] = gather_ok
    if strong is not None:
        line["config5_strong"] = strong
    if dec_line is not None:
        line["with_rgb_decoder"] = dec_line
    line.update(extras)
    if world == 1 and not args.no_train:
        torch.cuda.synchronize()
        del step, model
        torch.cuda.empty_cache()  # the child process needs ~3 GB of its own
        line["train_step"] = train_step_probe()
    if world == 1 and args.cpu_sample > 0:
        v, n, dt = oracle_rays_per_sec(cfg, args.cpu_sample)
        line["cpu_baseline"] = {"value": v, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"{n} rays (12:1 camera:lidar; render + lidar head + rgb decoder) of the same workload in {dt:.1f} s, oracle port of the reference torch path, best of thread counts probed, host has {os.cpu_count()} cpus"}
    if args.dump_outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    _emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


def secondary_legs(be, cfg, dev, steps, timed) -> dict:
    """configs[2] (16 actors), configs[3] (128 x 2048 lidar grid with rolling shutter) and the torch-GPU comparator."""
    import neurad_studio_b200 as nsb
    from neurad_studio_b200 import scene

    out = {}
    # ---- config 3: config 2's time step with 16 rigid actors crossing the cameras' frusta (default table sizes)
    try:
        cfg3 = nsb.NeuRADConfig(n_actors=16)
        trajs = scene.make_trajectories(16, cfg3.duration)
        p3 = scene.make_params(cfg3, seed=1, beta=3.0, sdf_bias=0.6, device=dev, trajectories=trajs)
        be.load_params(cfg3, p3)
        cams, scan = build_workload(cfg3, 0)
        n = 6 * CAM_RAYS + scan.points.shape[0]
        rays = {k: torch.empty(n, w, device=dev) for k, w in (("origins", 3), ("directions", 3), ("pixel_area", 1), ("times", 1))}
        sensor = torch.cat([torch.full((CAM_RAYS,), c.sensor_idx, dtype=torch.long) for c in cams] + [torch.full((scan.points.shape[0],), 6, dtype=torch.long)]).to(dev)
        is_lidar = torch.cat([torch.zeros(6 * CAM_RAYS, dtype=torch.uint8), torch.ones(scan.points.shape[0], dtype=torch.uint8)]).to(dev)
        pts = scan.points.to(dev)
        res = {k: torch.empty(n, w, device=dev) for k, w in (("features", cfg3.feature_dim), ("depth", 1), ("accumulation", 1), ("prop_depth_0", 1), ("prop_depth_1", 1))}
        ev = []

        def run3():
            off = 0
            for cam in cams:
                be.raygen_pinhole(cam, 1, 3, 1, 3, out={k: v[off:off + CAM_RAYS] for k, v in rays.items()})
                off += CAM_RAYS
            be.raygen_lidar_points(scan, pts, out={k: v[off:] for k, v in rays.items()})
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            be.render(dict(rays, sensor_idx=sensor, is_lidar=is_lidar), out=res, image_width=640)
            e1.record()
            ev.append((e0, e1))

        for _ in range(3):
            run3()
        ev.clear()
        ms3 = timed(run3, steps)
        be.check_status()
        k3 = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
        out["config3_actors"] = {"value": n * steps / (ms3 * 1e-3), "unit": "rays/s", "ms_per_step": ms3 / steps, "rays_per_step": n,
                                 "roofline": roofline_block(n, k3, "nff_sample_lane_kernel + nff_shade_lane_kernel, 16 actors"),
                                 "what": "BASELINE configs[2]: config 2's time step + 16 dynamic rigid actors (per-ray candidate lists, per-actor 4-level grids), default table sizes"}
        del p3, rays, res
    except Exception as e:
        out["config3_actors"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    # ---- config 4: one 128-beam x 2048-azimuth sweep with rolling shutter through the volumetric path (config-2 parameters)
    try:
        p2 = scene.make_params(cfg, seed=1, beta=3.0, sdf_bias=0.6, device=dev)
        be.load_params(cfg, p2)
        l2w = torch.zeros(3, 4)
        l2w[:, :3] = torch.eye(3)
        l2w[:, 3] = torch.tensor([0.0, 0.0, 2.0])
        n4 = 128 * 2048
        rays = {k: torch.empty(n4, w, device=dev) for k, w in (("origins", 3), ("directions", 3), ("pixel_area", 1), ("times", 1))}
        sensor = torch.full((n4,), 6, dtype=torch.long, device=dev)
        is_lidar = torch.ones(n4, dtype=torch.uint8, device=dev)
        res = {k: torch.empty(n4, w, device=dev) for k, w in (("features", cfg.feature_dim), ("depth", 1), ("accumulation", 1), ("prop_depth_0", 1),
                                                               ("prop_depth_1", 1), ("intensity", 1), ("ray_drop_logits", 1))}
        ev = []

        def run4():
            r = be.raygen_lidar_grid(l2w, -25.0, 15.0, 128, 360.0 / 2048, 4.0, 0.1, torch.tensor([10.0, 0.0, 0.0]), out=rays)
            assert r["shape"] == (128, 2048)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            be.render(dict(rays, sensor_idx=sensor, is_lidar=is_lidar), out=res, want_intensity=True, image_width=2048)
            e1.record()
            ev.append((e0, e1))

        for _ in range(3):
            run4()
        ev.clear()
        ms4 = timed(run4, steps)
        be.check_status()
        k4 = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
        out["config4_lidar_grid"] = {"value": n4 * steps / (ms4 * 1e-3), "unit": "rays/s", "ms_per_sweep": ms4 / steps, "rays_per_sweep": n4,
                                     "roofline": roofline_block(n4, k4, "nff_sample_lane_kernel + nff_shade_lane_kernel + lidar_decode_kernel, 262 144 rays"),
                                     "what": "BASELINE configs[3] (SURVEY 8d reading): 128-beam x 2048-azimuth sweep, per-ray time offset over the 0.1 s revolution, origin + velocity * dt, rendered through the volumetric path + lidar head"}
        del rays, res
        # ---- the reference's torch path on the GPU (oracle port with device=cuda): BASELINE.md section 3's comparator
        try:
            from oracle import neurad_oracle  # noqa: F401  (bench's baseline legs may execute the oracle)

            oracle_rays_per_sec(cfg, 32768, device="cuda")
            v, n_t, dt = oracle_rays_per_sec(cfg, 32768, repeats=3, device="cuda")
            out["gpu_torch_baseline"] = {"value": v, "unit": "rays/s", "sample": f"{n_t} rays (one eval_num_rays_per_chunk; render + lidar head + rgb decoder) in {dt * 1e3:.0f} ms",
                                         "what": "the reference's own PyTorch path (implementation='torch', oracle port) on this GPU -- the GPU comparator when tiny-cuda-nn / nerfacc are absent (BASELINE.md section 3); NOT tiny-cuda-nn"}
        except Exception as e:
            out["gpu_torch_baseline"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        del p2
    except Exception as e:
        out["config4_lidar_grid"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
