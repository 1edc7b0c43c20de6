#!/usr/bin/env python
"""bench.py — decoded Mpixel/s of a synthetic 1080p 4:2:0 baseline-JPEG batch (BASELINE.json metric).

One process per GPU (torchrun for N > 1); the batch is sharded by image (weak scaling: every GPU decodes `--images`
images), no collective on the data path.  Prints ONE JSON line.

  value      whole-job Mpixel/s with the JPEG bitstreams already resident in HBM
             (timed: unstuff/RST pre-pass + Huffman decode + IDCT/colour through jpgpu_batch_decode, CUDA events)
  parity     the timed batch itself, checked outside the timed region: coefficients of sampled images against the
             encoder's own, samples against the oracle, every copy of a file byte-identical to the first
  e2e        same metric through the library's host-to-host pipeline (jpgpu_pipeline_*): files in one pinned buffer in,
             pixels in one pinned buffer out, single-copy transfers overlapped with the kernels; next to it the plain
             cudaMemcpyAsync ceiling for the same bytes, measured in the same run at the same N
  roofline   the IDCT+colour kernel: algorithmic bytes (blocks*128 B in + W*H*3 B out) / its CUDA-event time, against
             MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline  the oracle (restatement of the reference decoder, O(N^4) cosf IDCT) on the host cores
  extra      short runs of BASELINE configs[3] (64 x 4K 4:4:4, restart interval 16), configs[4] (16 384 images sharded
             over the N GPUs, decoded in waves: strong scaling), a corpus at the density of the reference's fixtures
             (~2.7 bit/pixel), and - rank 0, N > 1 - the same job through the single-process multi-device handle

--impl reference times the reference's own CPU algorithm (the oracle port; the Rust crate cannot be built here) on the
same workload, bounded to a sample that finishes in minutes.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "decoded_mpixel_per_s_1080p_420_batch"
UNIT = "Mpixel/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--images", type=int, default=1024, help="images per GPU (BASELINE configs[2]: 1024 on 1 B200)")
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthetic images cycled to fill the batch")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--subsampling", default="420")
    ap.add_argument("--quality", type=int, default=85)
    ap.add_argument("--noise", type=float, default=6.0, help="sigma of the generator's noise (6: ~1.2 bit/pixel; 17.5: ~2.7)")
    ap.add_argument("--restart-interval", type=int, default=0, help="MCUs per restart interval (0 = none; needs the DRI "
                    "extension the reference panics on: BASELINE configs[3], e.g. 3840x2160 444 with 480/16/1)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="images in the CPU baseline sample (0 = 2 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra configurations (configs[3], configs[4], dense corpus, multi-device arm)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--job-images", type=int, default=16384, help="images of the configs[4] job, sharded over the N GPUs")
    ap.add_argument("--e2e-chunk", type=int, default=64, help="images per chunk of the host-to-host pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed decode returned as DIR/<name>.npy "
                    "(float32 / float64, at most 64 MB; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    return args


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_source_sha():
    h = hashlib.sha256()
    for f in ("jpgpu_kernels.cu", "jpgpu_core.h"):
        h.update(open(os.path.join(ROOT, "jpeg_rust_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def recorded_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per image of one `ncu --set full` capture of the IDCT/colour kernel
    (profiles/idct_traffic.json, written by profiles/summarize_ncu.py).  Only handed out while the kernel source is the
    one that was profiled; otherwise None - a stale constant is worse than none."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "idct_traffic.json")))
        e = t.get(key)
        if e and e.get("kernel_source_sha") == kernel_source_sha():
            return e["dram_bytes_per_image"], e.get("profile")
    except Exception:
        pass
    return None, None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.

    Through NVML in-process (pynvml: two light queries every 10 ms from a thread) where that is available; the
    `nvidia-smi -lms` loop it replaces is kept as the fallback.  Eight ranks each running their own nvidia-smi poller
    cost the slowest rank 3 % at N = 8 (6.94 against 6.72 ms per step with the pollers running; the same GPUs driven
    from one process after the pollers had stopped: 6.71-6.72 ms each, profiles/r02t)."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []          # nvidia-smi fallback: raw lines; NVML: (sm_mhz, reasons bitmask) tuples
        self.nvml = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(self.index)
            bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.lines.append((mhz, mask))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            n = self.nvml
            bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
            sm = sorted(x[0] for x in self.lines)
            reasons = sorted(k for k, b in bits.items() if any(x[1] & b for x in self.lines))
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "NVML, 10 ms period, in-process"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(self.NAMES, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


def cpu_reference_throughput(files, width, height, nthreads, sample):
    """The reference's algorithm (oracle port, cosf per term like transform.rs:79-81) on `nthreads` host threads,
    one image per thread at a time. Returns (Mpixel/s, seconds, images)."""
    import oracle_ffi as O
    from concurrent.futures import ThreadPoolExecutor
    O.lib()
    todo = [files[i % len(files)] for i in range(sample)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(nthreads) as ex:
        secs = list(ex.map(lambda f: O.time_decode(f, O.LAYOUT_REF, O.EXT_NONE, O.COS_CALL, 1), todo))
    dt = time.perf_counter() - t0
    if any(s < 0 for s in secs):
        raise RuntimeError("oracle failed on a benchmark image")
    return sample * width * height / dt / 1e6, dt, sample


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from jpeg_rust_b200 import synth
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or max(cores, 8)
    files = synth.synth_corpus(min(sample, args.distinct), args.width, args.height, args.subsampling, args.quality,
                               noise_sigma=args.noise)
    vals = []
    for _ in range(args.warmup):
        cpu_reference_throughput(files[:cores], args.width, args.height, cores, min(cores, len(files)))
    t_total = 0.0
    for _ in range(args.steps):
        v, dt, n = cpu_reference_throughput(files, args.width, args.height, cores, sample)
        vals.append(v)
        t_total += dt
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"synthetic {args.width}x{args.height} {args.subsampling} q{args.quality} baseline JPEG; "
                               f"each step decodes a bounded sample of {sample} images on the host CPU",
                   "images_per_step": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} images per step, one image per thread, oracle (C restatement of the "
                                   "reference: linear-search Huffman, O(N^4) f32 IDCT with cosf per term); the Rust "
                                   "crate itself cannot be built in this image (no rustc/cargo)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
class Workload:
    """`n` images (the `files` cycled), packed into one pinned host buffer, parsed, planned as one batch on `device`."""

    def __init__(self, files, n, ext, device, ctx=None):
        import numpy as np
        from jpeg_rust_b200 import LAYOUT_SPEC, Batch, pack_files, parse_packed
        self.files, self.n, self.distinct = files, n, len(files)
        cycled = [files[i % len(files)] for i in range(n)]
        self.sizes = [len(f) for f in cycled]
        self.buf, self.offs, self.owner = pack_files(cycled)
        self.descs, pst = parse_packed(self.buf, self.offs, self.sizes, ext, LAYOUT_SPEC)
        assert not any(pst), pst
        self.batch = Batch(descs=self.descs, device=device, keepalive=self.owner, ctx=ctx)
        self.stats = self.batch.stats()
        self.np = np

    def close(self):
        self.batch.close()


def time_decode(batch, stream, steps, barrier, max_over_ranks):
    import torch
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        batch.decode()            # the call a user makes: image groups pipelined over auxiliary streams inside the library
    e1.record(stream)
    barrier()
    time_decode.last_local_ms = e0.elapsed_time(e1) / steps
    return max_over_ranks(e0.elapsed_time(e1)) / steps


def stage_times(batch, stream, steps):
    """Entropy and IDCT/colour stage after stage on one stream (CUDA events), and every kernel's own device time."""
    import torch
    ent_ev, idct_ev = [], []
    for _ in range(steps):
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record(stream)
        batch.entropy()
        b.record(stream)
        batch.idct()
        c.record(stream)
        ent_ev.append((a, b))
        idct_ev.append((b, c))
    torch.cuda.synchronize()
    idct_ms = sum(a.elapsed_time(b) for a, b in idct_ev) / steps
    ent_ms = sum(a.elapsed_time(b) for a, b in ent_ev) / steps
    prof = None
    for _ in range(3):
        pr = batch.profile()
        prof = pr if prof is None else {k: prof[k] + pr[k] for k in pr}
    return ent_ms, idct_ms, {k: v / 3 for k, v in prof.items()}


KERNEL_NAME = {"420": "idct_colour_kernel<2,2,false>", "422": "idct_colour_kernel<2,1,false>", "444": "idct_colour_kernel<1,1,false>",
               "440": "idct_colour_kernel<1,2,false>", "gray": "idct_colour_kernel<1,1,true>"}


def roofline_of(stats, ent_ms, idct_ms, prof, subsampling, n, traffic_key):
    peak, peak_src = measured_peak()
    idct_bytes = stats["coef_bytes"] + stats["rgb_bytes"]
    achieved = idct_bytes / (idct_ms * 1e-3) / 1e9
    per_image, prof_name = recorded_traffic(traffic_key)
    pre = prof["prepass_count"] + prof["prepass_scan"] + prof["prepass_write"]
    wr_bytes = stats["scan_bytes"] + stats["coef_bytes"]
    return {"bound": "hbm", "kernel": KERNEL_NAME[subsampling], "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "frac_of_nominal_8TBps": achieved / 8000.0,
            "traffic": per_image * n if per_image else None,
            "traffic_source": (f"ncu --set full, {prof_name}; kernel source unchanged since" if per_image else
                               "none for this kernel source (profiles/idct_traffic.json holds another build's figure)"),
            "peak_source": peak_src, "ms_per_launch": idct_ms, "algorithmic_bytes_per_launch": idct_bytes,
            "kernels": {
                "prepass_count+scan+write": {"ms": pre, "algorithmic_GBps": 2 * stats["scan_bytes"] / (pre * 1e-3) / 1e9,
                                             "split_ms": [prof["prepass_count"], prof["prepass_scan"], prof["prepass_write"]],
                                             "bound": "instruction issue and latency of the classify / scan / byte-scatter chain"},
                "sync": {"ms": prof["sync"], "bitstream_GBps": stats["scan_bytes"] / max(prof["sync"], 1e-6) / 1e6,
                         "bound": "instruction issue of a serial bit-dependent decode (multi-symbol table lookups)"},
                "verify_scan": {"ms": prof["verify_scan"], "bound": "latency of the longest repair walk"},
                "decode_write": {"ms": prof["decode_write"], "algorithmic_GBps": wr_bytes / (prof["decode_write"] * 1e-3) / 1e9,
                                 "frac_of_hbm_peak": wr_bytes / (prof["decode_write"] * 1e-3) / 1e9 / peak,
                                 "bound": "instruction issue (one symbol per step plus the cooperative block flush), not HBM"},
                "idct_colour": {"ms": prof["idct_colour"]}},
            "entropy_stage": {"ms": ent_ms, "bitstream_GBps": stats["scan_bytes"] / (ent_ms * 1e-3) / 1e9,
                              "algorithmic_GBps": wr_bytes / (ent_ms * 1e-3) / 1e9}}


def parity_check(wl, gen, k_coef, k_oracle, seed):
    """The decoded batch `wl` (results resident on the device) against independent truth, outside any timed region:
    coefficients of `k_coef` images == the encoder's own quantised coefficients (bit-exact), samples of `k_oracle`
    images within 1 LSB of the oracle, and every copy of a distinct file byte-identical to its first decode."""
    import oracle_ffi as O
    import torch
    from concurrent.futures import ThreadPoolExecutor
    np = wl.np
    rng = np.random.default_rng(seed)
    n, b = wl.n, wl.batch
    idx = sorted(set(int(i) for i in rng.integers(0, n, k_coef)) | {0, n - 1})
    coef_exact = True
    for i in idx:
        data, want = gen(i % wl.distinct, True)
        assert data == wl.files[i % wl.distinct]
        got = b.coefficients(i)
        coef_exact = coef_exact and all(np.array_equal(a[:len(w)], w[:len(a)]) for a, w in zip(got, want))
    oidx = idx[:: max(1, len(idx) // k_oracle)][:k_oracle]
    with ThreadPoolExecutor(min(len(oidx), os.cpu_count() or 1)) as ex:
        refs = list(ex.map(lambda i: O.decode(wl.files[i % wl.distinct], layout=O.LAYOUT_SPEC,
                                              ext=O.EXT_DRI if wl.descs[i].restart_interval else O.EXT_NONE), oidx))
    max_abs, mean_abs = 0, 0.0
    for i, o in zip(oidx, refs):
        got = b.device_tensor(i).cpu().numpy()
        d = np.abs(got.astype(np.int16) - o.rgb.astype(np.int16))
        max_abs, mean_abs = max(max_abs, int(d.max())), max(mean_abs, float(d.mean()))
    copies_identical = True
    for i in range(wl.distinct, n):
        copies_identical = copies_identical and bool(torch.equal(b.device_tensor(i), b.device_tensor(i % wl.distinct)))
    ok = coef_exact and max_abs <= 1 and copies_identical
    if not ok:
        raise SystemExit(f"PARITY FAILURE: coef_exact={coef_exact} max_abs={max_abs} copies_identical={copies_identical}")
    return {"coef_exact": coef_exact, "coef_checked": len(idx), "max_abs": max_abs, "mean_abs": mean_abs,
            "oracle_checked": len(oidx), "copies_identical": copies_identical, "copies_checked": n - wl.distinct,
            "against": "encoder's quantised coefficients (bit-exact gate); oracle samples (gate: max |delta| <= 1)"}


DUMP_LIMIT_BYTES = 64 * 10 ** 6
DUMP_SAMPLE_BYTES = 32 * 10 ** 6
DUMP_SEED = 20261020


def dump_outputs(out_dir, batch, n):
    """What the timed decode (jpgpu_batch_decode) returned in its last step, for `n` images of one shape, written so
    that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
    At most 64 MB in all:
      status.npy, bytes_read.npy  float64 (n,)      per-image status and scan bytes consumed (jpgpu_batch_results)
      rgb_sample.npy              float32 (n, K)    K values of every image's decoded (H, W, 3) output, flattened, at
                                                    positions drawn from a fixed seed (all of them when K = H*W*3)
      rgb_images.npy              float32 (m, H, W, 3)  the first m images whole, as many as the rest of the 64 MB allows
    Returns {file name: shape}."""
    import numpy as np
    import torch
    statuses, bytes_read = batch.results()            # synchronises
    size = int(np.prod(batch.shape(0)))
    k = min(size, DUMP_SAMPLE_BYTES // (4 * n))
    rng = np.random.default_rng(DUMP_SEED)
    pos = np.stack([np.arange(k) if k == size else np.sort(rng.integers(0, size, k)) for _ in range(n)])
    pos_dev = torch.from_numpy(pos).cuda()
    sample = torch.empty((n, k), dtype=torch.uint8, device="cuda")
    for i in range(n):
        sample[i] = batch.device_tensor(i).reshape(-1).index_select(0, pos_dev[i])
    arrays = {"status": np.asarray(statuses, np.float64), "bytes_read": np.asarray(bytes_read, np.float64),
              "rgb_sample": sample.cpu().numpy().astype(np.float32)}
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values()) - 1024 * (len(arrays) + 1)   # 1 KB per .npy header
    m = min(n, room // (4 * size))
    if m:
        arrays["rgb_images"] = np.stack([batch.device_tensor(i).cpu().numpy() for i in range(m)]).astype(np.float32)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name + ".npy": list(a.shape) for name, a in arrays.items()}


def copy_ceiling(in_bytes, out_bytes, reps, barrier, max_over_ranks):
    """Plain pinned cudaMemcpyAsync of the same bytes the end-to-end leg moves (H2D and D2H on two streams at once),
    all ranks together: what the platform's PCIe / host memory system gives at this N, whatever the library does."""
    import torch
    hin = torch.empty(in_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(in_bytes, dtype=torch.uint8, device="cuda")
    dout = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")
    s0, s1 = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s0):
            hout.copy_(dout, non_blocking=True)
    once()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s0)
    s1.wait_event(e0)
    for _ in range(reps):
        once()
    s0.wait_stream(s1)
    e1.record(s0)
    barrier()
    return max_over_ranks(e0.elapsed_time(e1)) / reps


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from jpeg_rust_b200 import Batch, MultiDevice, Pipeline, _ffi, context, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")   # a barrier that does not park a spinning kernel on the waiting GPUs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = context(local_rank)
    # an ordinary (non-default) stream: the library replays repeated decodes as a CUDA graph, and the legacy default
    # stream cannot be captured (on it every decode is enqueued kernel by kernel, which at N = 8 - eight processes
    # launching 25 kernels per step over four streams on 32 vCPUs - cost the slowest rank 2-3 %, profiles/r02t, r02u)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # ---- inputs: `distinct` synthetic images, cycled to `images`, each copy with its own host region and its own device
    # buffers.  Every rank decodes the SAME corpus: weak scaling means the same work per GPU, and the job's time is the
    # slowest rank's - with a corpus of its own per rank (rounds 1 and early 2) the "scaling loss" at N = 8 was the rank
    # whose images happened to code into the most bits (6.88 against 6.72 ms, while one process driving the same eight
    # GPUs over identical images measured 6.71-6.72 ms on every one of them: profiles/r02v).
    first = 0

    def gen(i, want_coefs=False):
        return synth.synth_jpeg(first + i, args.width, args.height, args.subsampling, args.quality, args.restart_interval,
                                args.noise, want_coefs=want_coefs)
    files = synth.synth_corpus(args.distinct, args.width, args.height, args.subsampling, args.quality,
                               restart_interval=args.restart_interval, noise_sigma=args.noise, first_index=first)
    ext = _ffi.EXT_DRI if args.restart_interval else _ffi.EXT_NONE
    n = args.images
    wl = Workload(files, n, ext, local_rank)
    batch, stats = wl.batch, wl.stats
    pixels = stats["pixels"]

    # ---- value: bitstreams resident in HBM -> RGB resident in HBM
    batch.upload_from(wl.buf)
    for _ in range(args.warmup):
        batch.decode()
    launches0 = batch.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)          # let nvidia-smi start sampling before the timed region
    ms_per_step = time_decode(batch, stream, args.steps, barrier, max_over_ranks)
    # statuses of the last timed step: checked here, not after the warm-up, because with --warmup 0 nothing has been
    # decoded before the timed region and every image would still read as truncated
    statuses, _ = batch.results()
    bad = [s for s in statuses if s != 0]
    if bad:
        sampler.stop()
        raise SystemExit(f"decode failed for {len(bad)} images, first status {bad[0]}")
    per_rank_ms = None
    if world > 1:   # bookkeeping: every rank's own time, so that the line shows how far the slowest is from the rest
        mine = torch.tensor([time_decode.last_local_ms], dtype=torch.float64, device="cuda")
        allms = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allms, mine)
        per_rank_ms = [float(t.item()) for t in allms]
    launches = batch.launch_count() - launches0
    value = world * pixels / (ms_per_step * 1e-3) / 1e6
    dumped = None
    if args.dump_outputs and rank == 0:   # every rank decodes the same corpus
        dumped = dump_outputs(args.dump_outputs, batch, n)
    ent_ms, idct_ms, prof = stage_times(batch, stream, args.steps)
    if not sampler.lines:   # very short runs: keep the GPU busy with the same work until the sampler has reported
        t_end = time.perf_counter() + 1.0
        while not sampler.lines and time.perf_counter() < t_end:
            batch.decode()
            torch.cuda.synchronize()
    clocks = sampler.stop()   # sampled over the timed region and the per-stage loops: the GPU was under load throughout
    tkey = f"{args.width}x{args.height}_{args.subsampling}"
    roofline = roofline_of(stats, ent_ms, idct_ms, prof, args.subsampling, n, tkey)

    # ---- parity of the timed batch itself (outside the timed region)
    parity = None
    if not args.no_parity:
        batch.decode()
        parity = parity_check(wl, gen, 16, 4, 1234 + rank)

    # ---- 1-vs-N determinism on hardware: every rank also decodes rank 0's first 32 images; digests must agree
    determinism = None
    if world > 1:
        common = [synth.synth_jpeg(i, args.width, args.height, args.subsampling, args.quality, args.restart_interval, args.noise)
                  for i in range(32)]
        cb = Batch(common, ext=ext, device=local_rank)
        cb.upload().decode()
        outs = cb.download()
        st, _ = cb.results()
        assert all(s == 0 for s in st)
        h = hashlib.sha256()
        for o in outs:
            h.update(o.tobytes())
        cb.close()
        gathered = [None] * world
        dist.all_gather_object(gathered, h.hexdigest())     # bookkeeping only: 64 characters per rank
        determinism = {"ranks": world, "images": 32, "identical": len(set(gathered)) == 1,
                       "what": "sha256 over the RGB bytes of rank 0's first 32 images, decoded by every rank on its own GPU"}
        if not determinism["identical"]:
            raise SystemExit(f"DETERMINISM FAILURE: ranks disagree: {gathered}")

    # ---- e2e: host buffers in, host buffers out through the library's pipeline; copies inside the timed region
    e2e = None
    if not args.no_e2e:
        pipe = Pipeline(packed=(wl.buf, wl.owner), descs=wl.descs, device=local_rank, chunk=max(1, min(args.e2e_chunk, n)))
        pipe.run().sync()
        ksteps = max(1, min(args.steps, 3))
        ms_list = []
        for _ in range(ksteps):
            barrier()
            pipe.run()
            ms_list.append(pipe.elapsed_ms())    # CUDA events around the job on the pipeline's streams; synchronises
        barrier()
        e2e_ms = max_over_ranks(sum(ms_list) / len(ms_list))
        st, _ = pipe.results()
        assert all(s == 0 for s in st)
        # the host copy of sampled images equals what the resident-input run left on the device
        for i in (0, n // 2, n - 1):
            assert np.array_equal(pipe.image(i), batch.device_tensor(i).cpu().numpy()), "e2e output differs from the device result"
        in_bytes, out_bytes = int(wl.offs[-1]), pipe.out_bytes
        ceil_ms = copy_ceiling(in_bytes, out_bytes, ksteps, barrier, max_over_ranks)
        e2e_value = world * pixels / (e2e_ms * 1e-3) / 1e6
        ceil_value = world * pixels / (ceil_ms * 1e-3) / 1e6
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
               "ms_per_step": e2e_ms, "gpu_launches_per_step": pipe.launch_count() // (ksteps + 1),
               "copy_ceiling_ms": ceil_ms, "copy_ceiling_value": ceil_value,
               "copy_ceiling_gbs": world * (in_bytes + out_bytes) / (ceil_ms * 1e-3) / 1e9,
               "frac_of_ceiling": e2e_value / ceil_value,
               "note": f"jpgpu_pipeline_run: {(n + args.e2e_chunk - 1) // args.e2e_chunk} chunks of {min(args.e2e_chunk, n)} images "
                       "alternating between two stream sets, one H2D copy + one D2H copy per chunk, pinned host memory, plans made "
                       "once.  copy_ceiling = plain cudaMemcpyAsync of the same bytes both ways at once, all ranks together, same run",
               "numa": "single-node VM: sysfs reports numa_node -1 for the GPUs, one NUMA node, no binding attempted"}
        pipe.close()

    # ---- CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or 2 * cores
        v, dt, cnt = cpu_reference_throughput(files, args.width, args.height, cores, sample)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cnt} of the batch's images, one per thread, {dt:.1f} s wall; oracle = C restatement of the "
                         "reference decoder (not the Rust binary: no rustc in the image)"}

    # ---- BASELINE configs[0] and latency: single images through the single-image entry point (JPEGImage.parse =
    # parse + H2D + decode + D2H, synchronous), next to the reference's algorithm on one host core
    config0 = None
    lena_path = os.path.join(ROOT, "tests", "golden", "fixtures", "lena.jpeg")
    if rank == 0 and os.path.exists(lena_path):
        from jpeg_rust_b200 import JPEGImage, LAYOUT_REF, LAYOUT_SPEC

        def latency(data, layout, reps=20):
            for _ in range(3):
                JPEGImage.parse(data, layout=layout, device=local_rank)
            t0 = time.perf_counter()
            for _ in range(reps):
                JPEGImage.parse(data, layout=layout, device=local_rank)
            return (time.perf_counter() - t0) / reps * 1e3
        lena = open(lena_path, "rb").read()
        gpu_ms = latency(lena, LAYOUT_REF)
        config0 = {"workload": "lena.jpeg 512x512 4:2:2, one image per call, host bytes in, host RGB out, REF layout",
                   "gpu_ms_per_image": gpu_ms, "gpu_mpixel_per_s": 512 * 512 / gpu_ms / 1e3,
                   "one_1080p_420_ms_per_image": latency(files[0], LAYOUT_SPEC)}
        if world == 1 and not args.no_cpu_baseline:
            import oracle_ffi as O
            config0["cpu_ms_per_image_1_core"] = O.time_decode(lena, O.LAYOUT_REF, O.EXT_NONE, O.COS_CALL, 1) * 1e3

    # ---- extra configurations (short, outside `value`)
    extra = None
    if not args.no_extra:
        extra = {}
        esteps = max(2, min(args.steps, 5))

        def short_run(name, efiles, en, eext, sub, egen, w, h, k_oracle=2):
            ew = Workload(efiles, en, eext, local_rank)
            ew.batch.upload_from(ew.buf)
            for _ in range(2):
                ew.batch.decode()
            st, _ = ew.batch.results()
            assert all(s == 0 for s in st), (name, [s for s in st if s][:3])
            ms = time_decode(ew.batch, stream, esteps, barrier, max_over_ranks)
            e_ent, e_idct, e_prof = stage_times(ew.batch, stream, esteps)
            r = {"value": world * ew.stats["pixels"] / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms, "images_per_gpu": en,
                 "bits_per_pixel": 8.0 * sum(ew.sizes) / ew.stats["pixels"], "scaling": "weak",
                 "roofline": roofline_of(ew.stats, e_ent, e_idct, e_prof, sub, en, f"{w}x{h}_{sub}")}
            if not args.no_parity:
                ew.batch.decode()
                r["parity"] = parity_check(ew, egen, 6, k_oracle, 99 + rank)
            ew.close()
            extra[name] = r

        # BASELINE configs[3]: 4K 4:4:4, dense restart intervals (every 16 MCUs): images decode from their interval starts
        def gen4k(i, want_coefs=False):
            return synth.synth_jpeg(100000 + first + i, 3840, 2160, "444", 85, 16, 6.0, want_coefs=want_coefs)
        f4k = synth.synth_corpus(16, 3840, 2160, "444", 85, restart_interval=16, first_index=100000 + first)
        short_run("config3_4k444_dri16", f4k, 64, _ffi.EXT_DRI, "444", gen4k, 3840, 2160, k_oracle=1)   # the oracle takes ~10 s per 4K image
        del f4k

        # a corpus at the density of the reference's own fixtures (lena.jpeg 2.78, 2x2-chroma.jpeg 2.61 bit/pixel): the
        # entropy stage scales with bits, not pixels
        def gendense(i, want_coefs=False):
            return synth.synth_jpeg(200000 + first + i, 1920, 1080, "420", 85, 0, 17.5, want_coefs=want_coefs)
        fd = synth.synth_corpus(min(args.distinct, 128), 1920, 1080, "420", 85, noise_sigma=17.5, first_index=200000 + first)
        short_run("dense_1080p_420_2p7bpp", fd, n, _ffi.EXT_NONE, "420", gendense, 1920, 1080)
        del fd

        # BASELINE configs[4]: a job of --job-images images sharded over the N GPUs, every GPU decodes its share wave after
        # wave through the one batch object, all scans and all RGB outputs resident in HBM (strong scaling)
        share = args.job_images // world
        wave_out = batch.output_bytes()
        K = max(1, min(share // n, int(110e9 // max(wave_out, 1))))   # all outputs stay resident: at most ~110 GB of them
        out_arena = torch.empty(K * wave_out + 256, dtype=torch.uint8, device="cuda")
        out_base = (out_arena.data_ptr() + 255) // 256 * 256
        scan_stride = (int(wl.offs[-1]) + 255) // 256 * 256
        scans = torch.empty(K * scan_stride, dtype=torch.uint8, device="cuda")
        host_in = torch.from_numpy(wl.buf)
        for w in range(K):
            scans[w * scan_stride:w * scan_stride + int(wl.offs[-1])].copy_(host_in, non_blocking=True)
        scan_offs = [int(wl.descs[i].scan) - wl.buf.ctypes.data for i in range(n)]
        torch.cuda.synchronize()

        def run_job():
            for w in range(K):
                batch.set_device_scans(scans.data_ptr() + w * scan_stride, scan_offs)
                batch.set_device_output(out_base + w * wave_out, wave_out)
                batch.decode()
        run_job()
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        run_job()
        w1.record(stream)
        barrier()
        job_ms = max_over_ranks(w0.elapsed_time(w1))
        lo = out_base - out_arena.data_ptr()
        assert torch.equal(out_arena[lo:lo + wave_out], out_arena[lo + (K - 1) * wave_out:lo + K * wave_out]), "waves of identical input differ"
        batch.set_device_output(None, 0)
        batch.upload_from(wl.buf)
        batch.decode()
        torch.cuda.synchronize()
        extra["config4_job_sharded"] = {
            "images": K * n * world, "images_per_gpu": K * n, "waves_per_gpu": K, "value": world * K * pixels / (job_ms * 1e-3) / 1e6,
            "unit": UNIT, "ms": job_ms, "scaling": "strong",
            "resident_GB_per_gpu": {"scans": K * scan_stride / 1e9, "rgb": K * wave_out / 1e9},
            "note": "per wave: device-to-device hand-over of the wave's scan bytes (one kernel), decode into the wave's slice of one "
                    "resident output arena; bitstream / coefficient arenas of one batch object reused; no collective"}
        del out_arena, scans

        # the same weak-scaled job from ONE process through the multi-device handle (jpgpu_multi_*): no torch.distributed,
        # no NCCL anywhere near it - rank 0 drives all N GPUs while the other ranks wait at the barrier
        if world > 1:
            barrier()
            dist.barrier(group=host_group)
            if rank == 0:
                # (whatever happens in here, rank 0 reaches the barrier below: the other ranks are waiting at it)
                try:
                    if torch.cuda.device_count() < world:
                        raise RuntimeError(f"rank 0 sees {torch.cuda.device_count()} of {world} devices")
                    md = MultiDevice(list(range(world)))
                    allf = [files[i % args.distinct] for i in range(n * world)]
                    from jpeg_rust_b200 import pack_files, parse_packed
                    mbuf, moffs, mown = pack_files(allf, pinned=False)
                    mdescs, pst = parse_packed(mbuf, moffs, [len(f) for f in allf], ext)
                    assert not any(pst)
                    md.plan(descs=mdescs, keepalive=(mbuf, mown)).upload().decode().sync()
                    st, _ = md.results()
                    assert all(s == 0 for s in st)
                    md.time_decode(2)
                    per_dev = md.time_decode(esteps)
                    mms = max(per_dev) / esteps
                    extra["multi_device_single_process"] = {
                        "devices": world, "images": n * world, "value": n * world * args.width * args.height / (mms * 1e-3) / 1e6,
                        "unit": UNIT, "ms_per_step": mms, "per_device_ms_per_step": [x / esteps for x in per_dev],
                        "ranges": md.ranges(), "scaling": "weak",
                        "note": "jpgpu_multi_*: one process, one context + stream set + worker thread per device, contiguous image "
                                "ranges balanced by scan bytes, CUDA events per device, job time = slowest device"}
                    md.close()
                except Exception as e:   # the headline line must not be lost to an extra
                    extra["multi_device_single_process"] = {"error": f"{type(e).__name__}: {e}"}
            dist.barrier(group=host_group)   # the other ranks wait on the host: their GPUs are rank 0's for this arm
            barrier()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (IDCT/colour), i16/u8 (entropy)", "data": "synthetic",
            "config": {"workload": f"{n} synthetic {args.width}x{args.height} {args.subsampling} q{args.quality} baseline "
                                   f"JPEGs per GPU ({args.distinct} distinct, own buffers per copy; the same images on every GPU), SPEC layout"
                                   + (f", restart interval {args.restart_interval} MCUs" if args.restart_interval else ""),
                       "images_per_gpu": n, "bits_per_pixel": 8.0 * sum(wl.sizes) / pixels,
                       "l2": "inputs larger than L2 (no flush needed): "
                       f"{stats['scan_bytes'] / 1e6:.0f} MB bitstream, {stats['coef_bytes'] / 1e9:.2f} GB coefficients",
                       "parallelism": f"images sharded over {world} GPU(s), no collective"},
            "parity": parity, "determinism": determinism, "per_rank_ms_per_step": per_rank_ms,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "config0_single_image": config0, "extra": extra, "dumped_outputs": dumped,
            "stage_ms": {"entropy": ent_ms, "idct_colour": idct_ms, "note": "stages run one after the other on one stream; "
                         "`value` is timed over jpgpu_batch_decode, which overlaps the image groups of a batch"},
        }
        print(json.dumps(line), flush=True)
    batch.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
