#!/usr/bin/env python3
"""bench.py -- measures the colour-conversion hot path on B200 (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--workload c2|c3|c4|c5] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic frame (or batch) of the workload.  Default workload c2 is
the configuration BASELINE.json quotes its metric on: 7680x4320 RGB32f -> 12-bit Rec.2100 PQ YCbCr 4:2:0.

  value      whole-job Gpixels/s with inputs already resident in HBM, K steps between two CUDA events on the
             launching stream, barrier + synchronize on both sides, max over ranks.
  e2e        the same metric through the host-pointer C-ABI call the plug-in binds (avifgpu_encode_rows /
             avifgpu_decode_rows): pinned host rows -> PCIe -> kernel -> PCIe -> pinned host planes, every step.
  roofline   algorithmic bytes per launch / mean launch duration (CUDA events around every launch) against the
             measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the reference's CPU loop (oracle/_ref where the reference has the stage, the C restatement for
             the libheif stage) on this box's host cores, on a bounded sample -- reported, not a target.

With --impl reference only the CPU arm runs (rank 0 under torchrun; other ranks exit 0).
--dump-outputs DIR writes what the last timed step computed to DIR/<name>.npy (see dump_outputs): the inputs are seeded,
so two builds run with the same arguments can be compared output for output.
Multi-GPU (torchrun, one rank per GPU): frames / tiles are independent, so ranks share nothing on the data path
("scaling": "weak": every rank converts its own frame; --mode tile splits ONE frame into row blocks and gathers
the planes over NCCL, reported separately in `gather`).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "avif-format_b200", "python"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

from avifgpu import abi  # noqa: E402

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only when MEASURED_PEAKS.json is absent


# ---- workloads ------------------------------------------------------------------------------------------------------

def nclx_2020(transfer):
    return abi.Nclx(1, abi.PRIMARIES_BT2020, transfer, abi.MATRIX_BT2020_NCL, 1)


class Workload:
    """Describes one BASELINE.json configuration: geometry, descriptions, byte counts, synthetic data."""

    def __init__(self, key, rows=None, batch=None):
        """rows / batch: a smaller instance of the same configuration (a row block of c4, a share of c5's batch)."""
        self.key = key
        if key == "c2":
            self.name = "7680x4320 RGB32f -> 12-bit Rec.2100 PQ YCbCr 4:2:0 (BT.2020 NCL, full range, box down-filter, peak 80 nit)"
            self.direction, self.w, self.h, self.batch = "encode", 7680, 4320, 1
            self.enc = abi.EncodeDesc(self.w, self.h, 32, 3, abi.ALPHA_NONE, 12, abi.TRANSFER_PQ, 80, abi.LAYOUT_PLANAR_YCBCR,
                                      abi.CHROMA_420, abi.DOWN_FILTER_BOX, abi.GRAY16_LUT, nclx_2020(abi.TRANSFER_CHAR_PQ))
            self.bytes_per_pixel = 12 + 3  # SURVEY.md 8(d): in 12 B/px, out Y 2 + CbCr 2*2/4
            self.dtype = "f32"
        elif key == "c3":
            self.name = "7680x4320 10-bit HLG YCbCr 4:2:0 -> RGB32f (BT.2020 NCL, full range, OOTF gamma 1.2 @ 1000 nit)"
            self.direction, self.w, self.h, self.batch = "decode", 7680, 4320, 1
            self.dec = abi.DecodeDesc(self.w, self.h, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32,
                                      nclx_2020(abi.TRANSFER_CHAR_HLG), 1, 1.2, 1000, 80)
            self.bytes_per_pixel = 3 + 12
            self.dtype = "f32"
        elif key == "c3pq":
            self.name = "7680x4320 10-bit PQ YCbCr 4:2:0 -> RGB32f (BT.2020 NCL, full range, peak 80 nit)"
            self.direction, self.w, self.h, self.batch = "decode", 7680, 4320, 1
            self.dec = abi.DecodeDesc(self.w, self.h, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32,
                                      nclx_2020(abi.TRANSFER_CHAR_PQ), 1, 1.2, 1000, 80)
            self.bytes_per_pixel = 3 + 12
            self.dtype = "f32"
        elif key == "c4":
            self.name = "16384x16384 RGBA16 -> 10-bit YCbCr 4:2:2 + alpha plane (BT.601, straight alpha)"
            self.direction, self.w, self.h, self.batch = "encode", 16384, 16384, 1
            self.enc = abi.EncodeDesc(self.w, self.h, 16, 4, abi.ALPHA_STRAIGHT, 10, abi.TRANSFER_CLIP, 80, abi.LAYOUT_PLANAR_YCBCR,
                                      abi.CHROMA_422, abi.DOWN_FILTER_BOX, abi.GRAY16_LUT, None)
            self.bytes_per_pixel = 8 + 6
            self.dtype = "f32"
        elif key == "c5":
            self.name = "batch of 4096x4096 Gray16 -> 12-bit monochrome SMPTE 428-1 (32 images per GPU)"
            self.direction, self.w, self.h, self.batch = "encode", 4096, 4096, 32
            self.enc = abi.EncodeDesc(self.w, self.h * self.batch, 16, 1, abi.ALPHA_NONE, 12, gray16_curve=abi.GRAY16_SMPTE428)
            self.bytes_per_pixel = 2 + 2
            self.dtype = "f32"
        else:
            raise SystemExit(f"unknown workload {key}")
        if rows is not None:
            self.h = rows
            if self.direction == "encode":
                self.enc = self.enc.copy(height=rows)
            else:
                self.dec = self.dec.copy(height=rows)
        if batch is not None:
            self.batch = batch
            self.enc = self.enc.copy(height=self.h * batch)
        self.rows_total = self.h * self.batch
        self.pixels = self.w * self.rows_total
        self.algorithmic_bytes = self.pixels * self.bytes_per_pixel

    # -- descriptions for a row block presented as an image (CPU sample, multi-GPU tiles)
    def encode_desc(self, rows):
        return self.enc.copy(height=rows)

    def decode_desc(self, rows):
        return self.dec.copy(height=rows)

    # -- synthetic data (SURVEY.md 8(d)), generated on the device with a seeded generator
    def make_device_input(self, torch, device, seed):
        g = torch.Generator(device=device)
        g.manual_seed(seed)
        if self.key == "c2" and getattr(self, "smooth", False):
            # A smooth frame (supplementary, --data smooth): horizontal ramps per channel with 0.1 % noise, so that
            # neighbouring pixels fall into the same step-table buckets the way natural images do.
            x = torch.linspace(0.0, 1.0, self.w, device=device).repeat_interleave(3)
            phase = torch.tensor([0.05, 0.35, 0.65], device=device).repeat(self.w)
            base = 0.02 + 0.9 * torch.remainder(x + phase, 1.0)
            noise = 1.0 + 1.0e-3 * (torch.rand((self.h, self.w * 3), generator=g, device=device) - 0.5)
            return [(base[None, :] * noise).contiguous()]
        if self.key == "c2":
            n = (self.h, self.w * 3)
            kind = torch.rand(n, generator=g, device=device)
            v = torch.rand(n, generator=g, device=device)
            lo, hi = float(np.log(1e-4)), float(np.log(4.0))
            logu = torch.exp(torch.rand(n, generator=g, device=device) * (hi - lo) + lo)
            v = torch.where(kind < 0.20, logu, v)
            v = torch.where((kind >= 0.20) & (kind < 0.25), -torch.rand(n, generator=g, device=device), v)
            v = torch.where((kind >= 0.25) & (kind < 0.30), torch.round(torch.rand(n, generator=g, device=device)), v)
            return [v.contiguous()]
        if self.key in ("c3", "c3pq"):
            cw, ch = (self.w + 1) // 2, (self.h + 1) // 2
            y = torch.randint(0, 1024, (self.h, self.w), generator=g, device=device, dtype=torch.int16)
            cb = torch.randint(0, 1024, (ch, cw), generator=g, device=device, dtype=torch.int16)
            cr = torch.randint(0, 1024, (ch, cw), generator=g, device=device, dtype=torch.int16)
            return [y, cb, cr]
        if self.key == "c4":
            v = torch.randint(0, 32769, (self.h, self.w * 4), generator=g, device=device, dtype=torch.int32).to(torch.int16)
            return [v]
        v = torch.randint(0, 32769, (self.rows_total, self.w), generator=g, device=device, dtype=torch.int32).to(torch.int16)
        return [v]

    def make_device_output(self, torch, device):
        if self.direction == "decode":
            return [torch.empty((self.h, self.w * 3), dtype=torch.float32, device=device)]
        shapes = abi.encode_plane_shapes(self.enc)
        dt = torch.int16 if self.enc.image_bit_depth > 8 else torch.uint8
        return [None if s is None else torch.empty(s, dtype=dt, device=device) for s in shapes]


# ---- helpers ----------------------------------------------------------------------------------------------------------

class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md 'clocks line'), polled through NVML
    from a thread (nvidia-smi -lms cannot resolve a region of a few milliseconds); nvidia-smi is the fallback."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.running = False
        self.nvml = None
        self.thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            physical = self.index
            if visible:
                ids = [v.strip() for v in visible.split(",") if v.strip()]
                if self.index < len(ids) and ids[self.index].isdigit():
                    physical = int(ids[self.index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(physical)
            self.nvml = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
            return
        self.running = True
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        n = self.nvml
        while self.running:
            try:
                mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    reasons = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.0005)

    def _smi_once(self):
        try:
            out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            return float(out[0]), float(out[1])
        except Exception:
            return None, None

    def stop(self, t0, t1):
        if self.nvml is None:
            sm, smax = self._smi_once()
            return {"sm_mhz": sm, "sm_max_mhz": smax, "reasons": ["nvml unavailable: one nvidia-smi sample taken after the timed region"], "samples": 0}
        self.running = False
        self.thread.join(timeout=1.0)
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:
            inside = self.samples[-1:]
        mask = 0
        for s in inside:
            mask |= s[2]
        return {"sm_mhz": statistics.median([s[1] for s in inside]) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": [name for name, bit in self.REASONS if mask & bit], "samples": len(inside)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(workload_key):
    """dram bytes per launch from the committed ncu capture of the same command, if one has been recorded."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload_key)
    except Exception:
        return None


def common_config(workload):
    """The `config` object both arms print, key for key (the driver compares them)."""
    return {"workload": workload.name, "width": workload.w, "height": workload.rows_total, "pixels_per_step_per_gpu": workload.pixels,
            "algorithmic_bytes_per_pixel": workload.bytes_per_pixel}


# ---- the CPU arm (reference's CPU loop; the only place bench.py touches oracle/) -------------------------------------------

class CpuArm:
    def __init__(self, workload):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle  # noqa: E402  (checker / CPU baseline only)
        self.oracle = oracle
        self.port = oracle.load_restatement()
        self.ref = oracle.load_reference()
        self.w = workload
        self.threads = os.cpu_count() or 1

    def kind(self):
        """"reference": the reference's own translation units (oracle/_ref) run the stage the reference owns; "port": the C
        restatement does.  c5 is this project's composition (no reference path), the PQ/HLG decodes and c2/c4's in-tree
        stage go through the compiled reference when it is present; the libheif stage of c2/c4 is always the restatement
        (libheif is not in the reference tree) -- `stages` spells that out."""
        if self.w.key == "c5":
            return "port"
        return "reference" if self.ref is not None else "port"

    def stages(self):
        wl = self.w
        own = "oracle/_ref (reference TUs compiled in place)" if self.ref is not None else "oracle/liboracle.so (C restatement)"
        if wl.key in ("c2", "c4"):
            return {"plug-in stage (WriteHeifImage.cpp)": own, "libheif stage (matrix + down-filter)": "oracle/liboracle.so (C restatement)"}
        if wl.key == "c5":
            return {"Gray16 -> SMPTE 428 (this project's composition)": "oracle/liboracle.so (C restatement)"}
        return {"plug-in stage (ReadHeifImage.cpp / YuvDecode.cpp)": own}

    def describe(self, rows):
        wl = self.w
        if wl.key == "c2":
            stage = ("CreateHeifImageRGBThirtyTwoBit via the compiled reference TUs, then the libheif stage (matrix + 4:2:0 box; not in "
                     "the reference tree) via the C restatement") if self.ref is not None else "C restatement (fused)"
        elif wl.key in ("c3", "c3pq"):
            stage = "ReadHeifImageRGBThirtyTwoBit via the compiled reference TUs" if self.ref is not None else "C restatement"
        elif wl.key == "c4":
            stage = ("CreateHeifImageRGBSixteenBit via the compiled reference TUs + C restatement of the libheif stage"
                     if self.ref is not None else "C restatement (fused)")
        else:
            stage = "C restatement (Gray16 -> SMPTE 428 is this project's composition; the reference has no such path)"
        return f"{rows} rows x {wl.w} px of the workload ({rows * wl.w / 1e6:.2f} Mpx), {self.threads} threads, row-block parallel; {stage}"

    def _input(self, rows, seed):
        rng = np.random.default_rng(seed)
        wl = self.w
        if wl.key == "c2":
            import cases
            return cases.float_host_rows(rng, rows, wl.w, 3)
        if wl.key in ("c3", "c3pq"):
            cw, ch = (wl.w + 1) // 2, (rows + 1) // 2
            return [rng.integers(0, 1024, (rows, wl.w)).astype(np.uint16), rng.integers(0, 1024, (ch, cw)).astype(np.uint16),
                    rng.integers(0, 1024, (ch, cw)).astype(np.uint16), None]
        if wl.key == "c4":
            return rng.integers(0, 32769, (rows, wl.w * 4)).astype(np.uint16)
        return rng.integers(0, 32769, (rows, wl.w)).astype(np.uint16)

    def run_once(self, rows, data):
        """Converts `rows` rows; returns seconds."""
        wl, t = self.w, self.threads
        t0 = time.perf_counter()
        if wl.direction == "decode":
            (self.ref or self.port).decode(wl.decode_desc(rows), data, threads=t)
        elif wl.key in ("c2", "c4") and self.ref is not None:
            desc = wl.encode_desc(rows)
            inter = self.ref.encode(desc.copy(layout=abi.LAYOUT_REFERENCE), data, threads=t)[0]
            self.port.rgb_codes_to_ycbcr(desc, inter, threads=t)
        else:
            self.port.encode(wl.encode_desc(rows), data, threads=t)
        return time.perf_counter() - t0

    def sample(self, target_seconds, seed=99):
        """Sizes a row block so one conversion takes about target_seconds; returns (rows, seconds)."""
        wl = self.w
        probe_rows = min(wl.rows_total, max(2 * self.threads, 16)) & ~1
        probe_rows = max(probe_rows, 2)
        data = self._input(probe_rows, seed)
        self.run_once(probe_rows, data)
        t_probe = max(self.run_once(probe_rows, data), 1e-4)
        rows = int(probe_rows * target_seconds / t_probe) & ~1
        rows = max(min(rows, wl.rows_total), probe_rows)
        data = self._input(rows, seed + 1)
        return rows, data


def run_reference_impl(args, workload, rank, world):
    if rank != 0:
        return
    arm = CpuArm(workload)
    budget = float(os.environ.get("AVIFGPU_BENCH_REFERENCE_BUDGET_S", "150"))  # seconds for the whole run (tests shrink it)
    per_step = min(max(budget / (args.steps + args.warmup + 1), 0.5), 15.0)
    rows, data = arm.sample(per_step)
    for _ in range(args.warmup):
        arm.run_once(rows, data)
    t = 0.0
    for _ in range(args.steps):
        t += arm.run_once(rows, data)
    value = rows * workload.w * args.steps / t / 1e9
    line = {
        "impl": "reference", "metric": "Gpixels/s", "value": value, "unit": "Gpx/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": workload.dtype, "data": "synthetic",
        "config": common_config(workload),
        "cpu_baseline": {"value": value, "unit": "Gpx/s", "cores": arm.threads, "kind": arm.kind(), "stages": arm.stages(),
                         "sample": arm.describe(rows), "sample_rows_per_step": rows, "libm": arm.port.libm_version()},
        "e2e": {"value": value, "unit": "Gpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---- the GPU arm --------------------------------------------------------------------------------------------------------

class DeviceRun:
    """One workload resident in this rank's HBM: rotating input / output sets (so nothing of a previous step survives in
    the 126 MB L2) and a `launch(i)` that enqueues step i through the device-pointer C-ABI call."""

    def __init__(self, torch, avifgpu, gpu, wl, device, seed, copies=3):
        self.torch, self.wl, self.gpu, self.device = torch, wl, gpu, device
        if wl.direction == "encode":
            gpu.prepare_encode(wl.enc)  # a frame pipeline builds its step tables up front (one-off, ~40 ms; INTEGRATION.md 3)
        self.copies = copies
        self.inputs = [wl.make_device_input(torch, device, seed + 17 * i) for i in range(copies)]
        self.outputs = [wl.make_device_output(torch, device) for _ in range(copies)]
        self.stream = torch.cuda.current_stream(device)
        self.handle = self.stream.cuda_stream
        self._planes = avifgpu.planes_from_tensors

    def launch(self, i):
        wl, gpu = self.wl, self.gpu
        src, dst = self.inputs[i % self.copies], self.outputs[i % self.copies]
        if wl.direction == "encode":
            rows = src[0]
            gpu.encode_device(wl.enc, rows.data_ptr(), rows.stride(0) * rows.element_size(), self._planes(dst), stream=self.handle)
        else:
            out = dst[0]
            gpu.decode_device(wl.dec, self._planes([src[0], src[1], src[2], None]), out.data_ptr(), out.stride(0) * out.element_size(),
                              stream=self.handle)

    def timed(self, steps, warmup, barrier):
        """(elapsed ms over `steps` launches, per-launch ms list) between CUDA events on the launching stream."""
        torch = self.torch
        for i in range(warmup):
            self.launch(i)
        barrier()
        events = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        events[0].record(self.stream)
        for i in range(steps):
            self.launch(i)
            events[i + 1].record(self.stream)
        torch.cuda.synchronize(self.device)
        return events[0].elapsed_time(events[-1]), [events[i].elapsed_time(events[i + 1]) for i in range(steps)]


DUMP_ELEMENTS = 15_000_000  # float32 values in all: a dump stays under 64 MB


def dump_outputs(directory, torch, wl, outputs):
    """Writes the arrays a caller of the timed call receives -- decode: "rgb", the RGB32f rows; encode: the "y", "cb", "cr"
    and "alpha" planes that exist, their codes as float32 -- to directory/<name>.npy.  An array larger than its even share
    of DUMP_ELEMENTS keeps a fixed, seeded choice of whole rows (in ascending order), the same on every run."""
    names = ["rgb"] if wl.direction == "decode" else ["y", "cb", "cr", "alpha"]
    arrays = [(name, t) for name, t in zip(names, outputs) if t is not None]
    share = DUMP_ELEMENTS // len(arrays)
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays:
        keep = min(t.shape[0], max(1, share // t.shape[1]))
        if keep < t.shape[0]:
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(directory, name + ".npy"), t.float().cpu().numpy())


def roofline_block(wl, per_launch_ms, traffic=None):
    peak, peak_source = measured_peak()
    mean_ms = statistics.mean(per_launch_ms)
    achieved = wl.algorithmic_bytes / (mean_ms * 1e-3) / 1e9
    block = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
             "peak_source": peak_source, "algorithmic_bytes_per_launch": wl.algorithmic_bytes, "mean_launch_ms": mean_ms,
             "min_launch_ms": min(per_launch_ms)}
    if traffic is not None:
        block["traffic_source"] = ("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed "
                                   "ncu --set full capture of this command (not re-measured in this run: ncu cannot wrap a timed bench)")
    return block


def measure_e2e(torch, gpu, wl, run, device, barrier, steps):
    """The host-pointer C-ABI call with pinned host buffers on both sides, copies inside the timed region."""
    if wl.direction == "encode":
        host_in = torch.empty(run.inputs[0][0].shape, dtype=run.inputs[0][0].dtype, pin_memory=True)
        host_in.copy_(run.inputs[0][0])
        shapes = abi.encode_plane_shapes(wl.enc)
        dt = torch.int16 if wl.enc.image_bit_depth > 8 else torch.uint8
        host_out = [None if s is None else torch.empty(s, dtype=dt, pin_memory=True) for s in shapes]
        host_planes = abi.Planes()
        for k, t in enumerate(host_out):
            if t is not None:
                host_planes.data[k] = t.data_ptr()
                host_planes.stride[k] = t.stride(0) * t.element_size()
        h2d = host_in.numel() * host_in.element_size()
        d2h = sum(t.numel() * t.element_size() for t in host_out if t is not None)

        def step():
            gpu._check(gpu.lib.avifgpu_encode_rows(gpu.handle, C.byref(wl.enc), host_in.data_ptr(), host_in.stride(0) * host_in.element_size(),
                                                   0, wl.rows_total, C.byref(host_planes)))
    else:
        host_src = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in run.inputs[0]]
        for hs, t in zip(host_src, run.inputs[0]):
            hs.copy_(t)
        host_rows = torch.empty(run.outputs[0][0].shape, dtype=torch.float32, pin_memory=True)
        host_planes = abi.Planes()
        for k, t in enumerate(host_src):
            host_planes.data[k] = t.data_ptr()
            host_planes.stride[k] = t.stride(0) * t.element_size()
        h2d = sum(t.numel() * t.element_size() for t in host_src)
        d2h = host_rows.numel() * 4

        def step():
            gpu._check(gpu.lib.avifgpu_decode_rows(gpu.handle, C.byref(wl.dec), C.byref(host_planes), 0, wl.h, host_rows.data_ptr(),
                                                   host_rows.stride(0) * 4))
    step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize(device)
    return time.perf_counter() - t0, h2d, d2h


def run_shuttle_bench(wl_key, w, h, steps, devices):
    """e2e through the plug-in's OWN entry point: the C++ row shuttle (avif-format_b200/host/GpuRowShuttle.cpp,
    CreateHeifImageRGB*Bit) driven by a mock Photoshop host, planes in pageable heap memory with padded strides like
    libheif's.  Built here with g++ (host code only; the pixels go through libavifgpu.so)."""
    pkg = os.path.join(ROOT, "avif-format_b200")
    exe = os.path.join("/tmp", f"avifgpu_shuttle_bench_{os.getpid()}")
    cmd = ["g++", "-std=c++17", "-O2", "-I", os.path.join(pkg, "host"), os.path.join(pkg, "host", "tools", "shuttle_bench.cpp"),
           os.path.join(pkg, "host", "GpuRowShuttle.cpp"), os.path.join(pkg, "lib", "libavifgpu.so"),
           "-Wl,-rpath," + os.path.join(pkg, "lib"), "-lpthread", "-o", exe]
    try:
        subprocess.run(cmd, check=True, capture_output=True, timeout=300)
        out = {}
        # the read side (c3) has no planes to allocate: its source planes are the decoder's, filled before the clock starts
        variants = (("resident", "warm"), ("copy", "warm")) if wl_key == "c3" else (("resident", "warm"), ("resident", "fresh"), ("copy", "fresh"))
        for host, pages in variants:
            done = subprocess.run([exe, wl_key, str(w), str(h), str(steps), host, pages] + [str(d) for d in devices], capture_output=True, text=True,
                                  timeout=600)
            out[f"host_{host}_planes_{pages}"] = json.loads(done.stdout.strip().splitlines()[-1])
        return out
    except Exception as error:  # the figure is an extra; the line must still print
        return {"unavailable": f"{type(error).__name__}: {error}"}
    finally:
        try:
            os.remove(exe)
        except OSError:
            pass


def nvlink_counters(index):
    """Cumulative NVLink data bytes (tx, rx) of GPU `index` over all links, or None (nvidia-smi nvlink -gt d)."""
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], capture_output=True, text=True, timeout=20).stdout
        tx = rx = 0
        found = False
        for line in out.splitlines():
            line = line.strip()
            if "Data Tx" in line or "Data Rx" in line:
                value = int(line.split(":")[-1].strip().split()[0])
                found = True
                if "Tx" in line:
                    tx += value
                else:
                    rx += value
        return (tx * 1024, rx * 1024) if found else None  # KiB
    except Exception:
        return None


def run_b200(args, workload, rank, world, local_rank):
    import torch
    import avifgpu

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the avifgpu path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)

    def max_over_ranks(values):
        if dist is None:
            return [float(v) for v in values]
        t = torch.tensor([float(v) for v in values], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    gpu = avifgpu.Context(local_rank)
    wl = workload
    seed0 = {"c2": 2, "c3": 3, "c3pq": 6, "c4": 4, "c5": 5}[wl.key] * 1000 + 1234
    run = DeviceRun(torch, avifgpu, gpu, wl, device, seed0 + 101 * rank)

    # -- timed region: K steps, device-resident inputs
    run.timed(0, max(args.warmup, 3), barrier)  # warm-up only
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches_before = gpu.launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    elapsed_ms, per_launch_ms = run.timed(args.steps, 0, lambda: None)
    t_wall1 = time.perf_counter()
    barrier()
    launches = gpu.launch_count() - launches_before
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    elapsed_ms = max_over_ranks([elapsed_ms])[0]
    value = world * wl.pixels * args.steps / (elapsed_ms * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, wl, run.outputs[(args.steps - 1) % run.copies])

    # -- e2e: the host-pointer C-ABI call, pinned host buffers, copies inside the timed region
    e2e_steps = max(1, min(args.steps, 10))
    e2e_s, h2d, d2h = measure_e2e(torch, gpu, wl, run, device, barrier, e2e_steps)
    e2e_s = max_over_ranks([e2e_s])[0]
    e2e_value = world * wl.pixels * e2e_steps / e2e_s / 1e9

    # -- other configurations of BASELINE.json, shorter runs (device-resident): so that the driver's line carries them too
    others = {}
    if world == 1 and not args.no_other_workloads:
        del run
        torch.cuda.empty_cache()
        for key in ("c3", "c3pq", "c4", "c5"):
            if key == wl.key:
                continue
            other = Workload(key)
            other_run = DeviceRun(torch, avifgpu, gpu, other, device, 777 + len(others), copies=2 if key == "c4" else 3)
            ms, per = other_run.timed(12, 3, barrier)
            block = roofline_block(other, per, recorded_traffic(key))
            others[key] = {"workload": other.name, "value": other.pixels * 12 / (ms * 1e-3) / 1e9, "unit": "Gpx/s", "steps": 12,
                           "roofline_frac": block["frac"], "achieved_gbs": block["achieved"], "mean_launch_ms": block["mean_launch_ms"]}
            del other_run
            torch.cuda.empty_cache()
        run = None

    # -- multi-GPU as north_star states it: ONE c4 frame row-tiled over the ranks, planes assembled on the owner;
    #    c5's batch of 256 images shared out
    tile = batch = None
    if dist is not None and not args.no_multi_gpu_blocks:
        run = None
        torch.cuda.empty_cache()
        tile = run_tile_block(torch, dist, gpu, avifgpu, device, rank, world, max(3, min(args.steps, 10)))
        batch = run_batch_block(torch, dist, gpu, avifgpu, device, rank, world, max(3, min(args.steps, 10)), barrier, max_over_ranks)
    elif dist is not None and args.mode == "tile" and wl.direction == "encode":
        tile = run_tile_block(torch, dist, gpu, avifgpu, device, rank, world, max(3, min(args.steps, 10)), workload=wl)

    shuttle = None
    if rank == 0 and not args.no_shuttle and wl.key in ("c2", "c3", "c4"):
        shuttle = {"one_gpu": run_shuttle_bench(wl.key, wl.w, wl.rows_total, 5, [local_rank])}
        if wl.key == "c2" and world == 1:
            # the read side beside it: ReadHeifImageRGBThirtyTwoBit on config 3's image (8K 10-bit HLG 4:2:0 -> RGB32f)
            shuttle["one_gpu_read_side_c3"] = run_shuttle_bench("c3", wl.w, wl.rows_total, 5, [local_rank])
    if dist is not None:
        dist.barrier()
    if rank == 0 and world > 1 and not args.no_shuttle and wl.key in ("c2", "c4"):
        # every GPU of the job behind ONE plug-in call (avifgpu_shard_group); the other ranks idle at the barrier below
        shuttle[f"{world}_gpus_one_process"] = run_shuttle_bench(wl.key, wl.w, wl.rows_total, 5, list(range(world)))
    if dist is not None:
        dist.barrier()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(wl)
            rows, data = arm.sample(12.0)
            seconds = arm.run_once(rows, data)
            cpu = {"value": rows * wl.w / seconds / 1e9, "unit": "Gpx/s", "cores": arm.threads, "kind": arm.kind(), "stages": arm.stages(),
                   "sample": arm.describe(rows), "seconds": seconds, "libm": arm.port.libm_version()}
        config = common_config(wl)
        line = {
            "metric": "Gpixels/s", "value": value, "unit": "Gpx/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": wl.dtype, "data": "synthetic" if not getattr(wl, "smooth", False) else "synthetic (smooth ramps + 0.1 % noise; supplementary)",
            "config": config,
            "details": {"parallelism": f"{world} independent frame(s), one per GPU, no collective on the data path",
                        "l2": f"3 rotating input/output sets of {wl.algorithmic_bytes / 1e6:.0f} MB each (> 126 MB L2)"},
            "roofline": roofline_block(wl, per_launch_ms, recorded_traffic(wl.key)),
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "Gpx/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "ms_per_step": 1e3 * e2e_s / e2e_steps, "buffers": "pinned host memory on both sides (avifgpu_host_alloc-equivalent)"},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if shuttle is not None:
            line["e2e_shuttle"] = shuttle
        if others:
            line["other_workloads"] = others
        if tile is not None:
            line["tile"] = tile
        if batch is not None:
            line["batch"] = batch
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    gpu.close()


def block_seeded_rows(torch, wl, device, y0, n, block_index):
    """Rows [y0, y0 + n) of the synthetic c4 frame: every row block has its own seed, so a rank can make just its part."""
    g = torch.Generator(device=device)
    g.manual_seed(40000 + block_index)
    return torch.randint(0, 32769, (n, wl.w * 4), generator=g, device=device, dtype=torch.int32).to(torch.int16)


def run_tile_block(torch, dist, gpu, avifgpu, device, rank, world, steps, workload=None):
    """SURVEY.md 8(e): ONE frame (default BASELINE config 4, 16384x16384 RGBA16 -> 10-bit 4:2:2 + A), rank r converts row
    block r, the planar image is assembled on the owner (rank 0), two ways:
      fused      the conversion kernels store straight into rank 0's planes over NVLink (CUDA IPC peer mapping): the
                 transfer overlaps the conversion tile by tile, there is no gather pass;
      gather     each rank converts into local planes, then ONE grouped NCCL gather per step sends every plane block to
                 rank 0, received directly into its place in the final plane (no re-stitch copy).
    Device time, max over ranks.  Both assembled images are compared with rank 0 converting the whole frame alone."""
    from avifgpu import sharding
    wl = workload or Workload("c4")
    gpu.prepare_encode(wl.enc)
    blocks = avifgpu.shard_row_blocks(0, wl.rows_total, world)
    y0, n = blocks[rank]
    if wl.key == "c4":
        block = block_seeded_rows(torch, wl, device, y0, n, rank)
    else:
        block = wl.make_device_input(torch, device, 4242)[0][y0:y0 + n].contiguous()  # same seed everywhere: the same frame
    stream = torch.cuda.current_stream(device).cuda_stream
    dt = torch.int16 if wl.enc.image_bit_depth > 8 else torch.uint8
    shapes = abi.encode_plane_shapes(wl.enc)
    block_desc = wl.enc.copy(height=n)
    local = [None if s is None else torch.empty(s, dtype=dt, device=device) for s in abi.encode_plane_shapes(block_desc)]
    full = [None if s is None else torch.empty(s, dtype=dt, device=device) for s in shapes] if rank == 0 else None

    def convert_local():
        if n > 0:
            gpu.encode_device(block_desc, block.data_ptr(), block.stride(0) * block.element_size(), avifgpu.planes_from_tensors(local), stream=stream)

    def gather_to_owner():
        sharding.gather_planes_to_owner(dist, torch, wl.enc, blocks, local, full, rank, owner=0)

    def time_loop(body):
        for _ in range(2):
            body()
        torch.cuda.synchronize(device)
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            body()
        e1.record()
        torch.cuda.synchronize(device)
        t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    convert_ms = time_loop(convert_local)

    def convert_and_gather():
        convert_local()
        gather_to_owner()
    gather_ms = time_loop(convert_and_gather)

    # reference result: rank 0 converts the whole frame alone
    whole = None
    if rank == 0:
        frame = torch.cat([block_seeded_rows(torch, wl, device, by0, bn, r) for r, (by0, bn) in enumerate(blocks)]) if wl.key == "c4" \
            else wl.make_device_input(torch, device, 4242)[0]
        whole = [None if s is None else torch.empty(s, dtype=dt, device=device) for s in shapes]
        gpu.encode_device(wl.enc, frame.data_ptr(), frame.stride(0) * frame.element_size(), avifgpu.planes_from_tensors(whole), stream=stream)
        torch.cuda.synchronize(device)
        one_gpu_ms = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gpu.encode_device(wl.enc, frame.data_ptr(), frame.stride(0) * frame.element_size(), avifgpu.planes_from_tensors(whole), stream=stream)
            e1.record()
            torch.cuda.synchronize(device)
            one_gpu_ms.append(e0.elapsed_time(e1))
        del frame
    gathered_identical = bool(all(torch.equal(a, b) for a, b in zip(full, whole) if a is not None)) if rank == 0 else None

    plane_bytes = sum(s[0] * s[1] * (2 if wl.enc.image_bit_depth > 8 else 1) for s in shapes if s is not None)
    ingress = plane_bytes * (wl.rows_total - blocks[0][1]) / max(wl.rows_total, 1)  # bytes that must reach the owner over NVLink
    report = {
        "workload": wl.name, "mode": f"one frame, {world} even row-block tiles, planes assembled on rank 0",
        "identical_to_single_gpu": gathered_identical,
        "one_gpu_ms": statistics.median(one_gpu_ms) if rank == 0 else None,
        "convert_ms": convert_ms, "convert_gpx_s": wl.pixels / (convert_ms * 1e-3) / 1e9,
        "gather": {"how": "grouped NCCL send/recv to the owner, received in place (torch.distributed.batch_isend_irecv)",
                   "convert_plus_assemble_ms": gather_ms, "gpx_s": wl.pixels / (gather_ms * 1e-3) / 1e9},
        "owner_nvlink_ingress_bytes": ingress,
        "owner_nvlink_ingress_floor_ms": {"at_770_GBs_measured_peer_copy": ingress / 770e9 * 1e3, "at_900_GBs_nominal": ingress / 900e9 * 1e3},
    }

    # fused placement
    try:
        peer = sharding.PeerPlanes(dist, wl.enc, rank, owner=0)
    except Exception as error:  # no peer access on this box: report it, keep the gather numbers
        report["fused"] = {"unavailable": str(error)}
        return report
    peer_planes = peer.planes()
    block_ptr, block_stride = block.data_ptr(), block.stride(0) * block.element_size()

    def convert_place():
        if n > 0:
            gpu.encode_device(wl.enc, block_ptr, block_stride, peer_planes, y0=y0, nrows=n, stream=stream)

    counters_before = nvlink_counters(0) if rank == 0 else None
    fused_ms = time_loop(convert_place)
    torch.cuda.synchronize(device)
    dist.barrier()
    counters_after = nvlink_counters(0) if rank == 0 else None
    placed_identical = None
    if rank == 0:
        placed = peer.owner_tensors(torch, device)
        placed_identical = bool(all(torch.equal(a, b) for a, b in zip(placed, whole) if a is not None))
        del placed
    dist.barrier()
    peer.close()
    fused = {"how": "every rank's conversion kernel stores its block into rank 0's planes (CUDA IPC peer mapping, NVLink / NVSwitch)",
             "identical_to_single_gpu": placed_identical, "convert_plus_assemble_ms": fused_ms, "gpx_s": wl.pixels / (fused_ms * 1e-3) / 1e9,
             "ingress_gbs": ingress / (fused_ms * 1e-3) / 1e9}
    if counters_before and counters_after:
        launches_counted = steps + 2
        fused["owner_nvlink_rx_bytes_per_step_counted"] = (counters_after[1] - counters_before[1]) / launches_counted
    report["fused"] = fused
    if rank == 0 and report["one_gpu_ms"]:
        report["speedup_vs_one_gpu"] = {"fused": report["one_gpu_ms"] / fused_ms, "gather": report["one_gpu_ms"] / gather_ms,
                                        "convert_only": report["one_gpu_ms"] / convert_ms}
    return report


def run_batch_block(torch, dist, gpu, avifgpu, device, rank, world, steps, barrier, max_over_ranks):
    """BASELINE config 5: a batch of 256 4096x4096 Gray16 images -> 12-bit SMPTE 428, images shared out over the ranks
    (256 / world each, no data-path collective).  Each rank's share is compared with the same images converted one by one."""
    total = 256
    mine = total // world + (1 if rank < total % world else 0)
    wl = Workload("c5", batch=mine)
    gpu.prepare_encode(wl.enc)
    g = torch.Generator(device=device)
    g.manual_seed(50000 + rank)
    rows = torch.randint(0, 32769, (wl.rows_total, wl.w), generator=g, device=device, dtype=torch.int32).to(torch.int16)
    out = wl.make_device_output(torch, device)
    stream = torch.cuda.current_stream(device).cuda_stream

    def convert():
        gpu.encode_device(wl.enc, rows.data_ptr(), rows.stride(0) * 2, avifgpu.planes_from_tensors(out), stream=stream)

    for _ in range(2):
        convert()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        convert()
    e1.record()
    torch.cuda.synchronize(device)
    ms = max_over_ranks([e0.elapsed_time(e1)])[0] / steps
    # the batch call must equal image-by-image conversion (the first two images of this rank's share)
    single = Workload("c5", batch=1)
    identical = True
    for i in range(min(mine, 2)):
        one = single.make_device_output(torch, device)
        part = rows[i * wl.h:(i + 1) * wl.h]
        gpu.encode_device(single.enc, part.data_ptr(), part.stride(0) * 2, avifgpu.planes_from_tensors(one), stream=stream)
        torch.cuda.synchronize(device)
        identical = identical and bool(torch.equal(one[0], out[0][i * wl.h:(i + 1) * wl.h]))
    flags = max_over_ranks([0.0 if identical else 1.0])
    pixels = total * wl.w * wl.h
    per_gpu_bytes = mine * wl.w * wl.h * wl.bytes_per_pixel
    peak, _ = measured_peak()
    return {"workload": "batch of 256 x 4096x4096 Gray16 -> 12-bit monochrome SMPTE 428-1, images shared out over the ranks",
            "images_per_gpu": mine, "convert_ms": ms, "gpx_s": pixels / (ms * 1e-3) / 1e9, "identical_to_image_by_image": flags[0] == 0.0,
            "per_gpu_roofline_frac": per_gpu_bytes / (ms * 1e-3) / 1e9 / peak, "collective": "none (results stay on the GPU that made them)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--workload", choices=("c2", "c3", "c3pq", "c4", "c5"), default="c2")
    ap.add_argument("--no-other-workloads", action="store_true", help="N = 1: skip the short c3 / c3pq / c4 / c5 lines")
    ap.add_argument("--no-multi-gpu-blocks", action="store_true", help="N > 1: skip the c4 tile and c5 batch blocks")
    ap.add_argument("--no-shuttle", action="store_true", help="skip e2e_shuttle (the C++ row shuttle under a mock host)")
    ap.add_argument("--mode", choices=("frames", "tile"), default="frames")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--data", choices=("random", "smooth"), default="random",
                    help="c2 only: 'random' (default, SURVEY 8(d): the worst case for the table look-ups) or 'smooth' (supplementary)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, rank 0, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = Workload(args.workload)
    workload.smooth = args.data == "smooth"
    if args.impl == "reference":
        run_reference_impl(args, workload, rank, world)
        return
    run_b200(args, workload, rank, world, local_rank)


if __name__ == "__main__":
    main()
