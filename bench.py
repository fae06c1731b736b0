#!/usr/bin/env python
"""bench.py -- scanned GB/s of the Pire hot path on B200 (BASELINE.json metric).

A "step" is one pass of the scan path over one batch of synthetic strings that is already resident in HBM:
Runner(sc).Begin().Run(str).End() for every string of the batch (pire/run.h:365-392), producing the packed match
bitmap and the per-string accepted-regexp mask.  With N > 1 the batch is sharded by string (weak scaling: every GPU
holds its own 10 GB shard, BASELINE configs[4] at N = 8) through pire_gpu_run_sharded of the C ABI: each rank scans
into its slot of the full bitmap and one in-place NCCL all-gather of the slots completes it on every rank.  The
exchange of step k runs on the communicator's stream and overlaps the scan of step k+1 (two bitmap buffers); all
exchanges finish inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload glue10|headline|utf8mixed]
  python bench.py --impl reference ...     # the reference's own CPU scan (oracle/_ref)

One JSON line on stdout (rank 0).  Keys follow the driver's contract:
  value / roofline   the scan with inputs resident in HBM (algorithmic bytes = payload bytes, 1 B read per input byte,
                     SURVEY.md 8(d)); roofline.kernel_ms is event-timed around the scan launches alone
  e2e                the same metric through pire_gpu_run_batch_host with HOST buffers, copies inside the timed region:
                     pinned (the headline) and pageable (what Runner::Run's callers hold), at N > 1 including the
                     bitmap exchange
  parity             GPU bits and accept masks against the reference on the very bytes the GPU scanned: the first 2^22
                     strings, every planted string and a stratified sample of 32-string units of every rank's shard;
                     any mismatch fails the run
  configs            BASELINE configs[1] and configs[3] on their OWN corpora (this GPU only), each with its parity check
  cpu_baseline       the reference library timed on this box's host cores on a bounded sample of the same bytes
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

STRING_LEN = 1024
STRINGS_PER_GPU = 9_765_632          # x 1 KiB = 10.000007 GB per GPU (multiple of 32 strings)
MIXED_STRINGS_PER_GPU = 1_281_024    # mixed 16 B..64 KiB strings, mean 7.8 KB: ~10 GB per GPU
FALLBACK_HBM_GBS = 6650.0            # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="pire_b200", choices=["pire_b200", "reference"])
    ap.add_argument("--workload", default="glue10", choices=["glue10", "headline", "utf8mixed"])
    ap.add_argument("--strings", type=int, default=0, help="strings per GPU (default: 10 GB worth)")
    ap.add_argument("--variant", default="auto", choices=["auto", "plain", "pred", "priv", "look", "look64", "look1"])
    ap.add_argument("--no-tune", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-records of the other BASELINE configs")
    ap.add_argument("--no-next", action="store_true", help="skip the SURVEY 8(f) rows (prefix scan, counting)")
    ap.add_argument("--collective", default="allgather", choices=["allgather", "allreduce"],
                    help="allgather: pire_gpu_run_sharded (C ABI, NCCL all-gather of bitmap slots, overlapped); "
                         "allreduce: torch.distributed all-reduce of the zeroed full bitmap (north_star's wording, serialized)")
    ap.add_argument("--cpu-sample", type=int, default=1 << 22, help="strings in the CPU-baseline sample (per step of the reference arm)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (match bitmap, accept masks) to DIR/<name>.npy")
    return ap.parse_args()


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return FALLBACK_HBM_GBS, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """SM clock + throttle reasons during the timed region.

    NVML polled every 4 ms from a thread, started before the warm-up (the same counters nvidia-smi prints, exact
    timestamps).  Without NVML the recipe's `nvidia-smi --query-gpu=... -lms 20` line runs as a subprocess (its
    lines reach us through a pipe, so their arrival times are only approximate and a short timed region can end
    before the first one arrives).  Measured (tools/sessions/gpu_r2_s49.sh): neither source, nor both, moves the
    step time (2.367-2.369 ms with NVML + nvidia-smi, NVML at 4 or 10 ms, and without any sampling)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc = [], None
        self.nvml_rows, self.nvml, self.nvml_max, self._halt = [], None, None, False
        self.poll_s = max(1, int(os.environ.get("PIRE_B200_CLOCKS_POLL_MS", "4"))) / 1e3
        try:
            import pynvml
            pynvml.nvmlInit()
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.nvml_thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.nvml_thread.start()
        except Exception:
            self.nvml = None
        # nvidia-smi is the fallback: with NVML at hand its subprocess (a full query every 20 ms) would only add to what
        # the sampling costs the GPU under test; PIRE_B200_CLOCKS_SMI=1 runs it beside NVML all the same
        if self.nvml is not None and not os.environ.get("PIRE_B200_CLOCKS_SMI"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nvml
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._halt:
            try:
                t = time.perf_counter()
                sm = float(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM))
                mask = int(reasons_fn(self._handle))
                self.nvml_rows.append((t, sm, [name for bit, name in bits if mask & bit]))
            except Exception:
                break
            time.sleep(self.poll_s)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    @staticmethod
    def _window(rows, t0, t1):
        inside = [r for r in rows if t0 <= r[0] <= t1]
        if inside:
            return inside
        near = [r for r in rows if t0 - 0.05 <= r[0] <= t1 + 0.05]     # region shorter than the sampling period
        return near or rows[-3:]

    def stop(self, t0, t1):
        if self.nvml:
            self._halt = True
            self.nvml_thread.join(timeout=1.0)
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        rows = self._window(self.nvml_rows, t0, t1) if self.nvml_rows else []
        if rows:
            reasons = sorted({name for _, _, names in rows for name in names})
            return {"sm_mhz": statistics.median(sm for _, sm, _ in rows), "sm_max_mhz": self.nvml_max, "reasons": reasons,
                    "samples": len(rows), "source": "nvml, polled every %g ms" % (self.poll_s * 1e3)}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        rows = self._window(self.rows, t0, t1)
        for _, r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(self.NAMES, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows), "source": "nvidia-smi -lms 20"}


# ----------------------------------------------------------------------------- host CPUs

def host_cpus():
    """What this process may actually use: logical CPUs, its affinity mask, and the cgroup's CPU quota (a 1-GPU lease
    of a 128-thread box can be capped at a dozen CPUs' worth of time while hardware_concurrency() still says 128)."""
    logical = os.cpu_count() or 1
    affinity = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else logical
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, period = f.read().split()
            if q != "max":
                quota = float(q) / float(period)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, period = float(f.read()), float(g.read())
                if q > 0:
                    quota = q / period
        except Exception:
            pass
    return {"logical": logical, "affinity": affinity, "cgroup_cpu_quota": quota}


def numa_bind(gpu_index):
    """Run this rank (and the pinned buffers it allocates from now on: first touch) on the CPUs of its GPU's NUMA
    node.  Eight un-pinned ranks pulling pinned pages across sockets halved the 8-GPU host-buffer throughput in
    round 1.  Returns a description for the JSON line, or None when the topology is not visible."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                  # 00000000:17:00.0 -> 0000:17:00.0
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"gpu": gpu_index, "pci": bus, "numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


# ----------------------------------------------------------------------------- the reference on the host

class PortScanner:
    """Stand-in with RefScanner.run's signature over the oracle port (oracle/pire_oracle.c), used
    only when oracle/_ref (the compiled reference) is not on this box.  Python threads over slices:
    the C call drops the GIL."""

    def __init__(self, image):
        from refpire import Oracle
        self.orc = Oracle(image)

    def run(self, corpus, offsets=None, fixed_len=0, n=None, variant=1, threads=1, want=("final", "mask")):
        import numpy as np
        from concurrent.futures import ThreadPoolExecutor
        threads = max(1, min(threads, n // 1024 or 1))
        final = np.zeros(n, np.uint8)
        mask = np.zeros(n, np.uint32)

        def part(k):
            lo, hi = n * k // threads, n * (k + 1) // threads
            if offsets is not None:
                f, m, _ = self.orc.run(corpus, offsets[lo:hi + 1], n=hi - lo, shortcuts=variant != 2)
            else:
                f, m, _ = self.orc.run(corpus[lo * fixed_len:hi * fixed_len], fixed_len=fixed_len, n=hi - lo, shortcuts=variant != 2)
            final[lo:hi] = f
            mask[lo:hi] = m
        with ThreadPoolExecutor(threads) as pool:
            list(pool.map(part, range(threads)))
        return final, mask, None


class PortRef:
    kind = "port"

    def scanner(self, workload):
        from pire_b200 import workloads as W
        return PortScanner(W.load_image(W.WORKLOADS[workload][0]))


_REF = None


def get_reference():
    """The compiled reference (oracle/_ref) when it is on this box, else the oracle port."""
    global _REF
    if _REF is None:
        from refpire import Ref, have_ref
        if have_ref():
            _REF = Ref()
            _REF.kind = "reference"
        else:
            _REF = PortRef()
    return _REF


_REF_SCANNERS = {}


def reference_scanner(workload):
    from pire_b200 import workloads as W
    if workload not in _REF_SCANNERS:
        ref = get_reference()
        if ref.kind == "port":
            _REF_SCANNERS[workload] = ref.scanner(workload)
        elif workload == "utf8mixed":
            _REF_SCANNERS[workload] = ref.compile(*W.HEADLINE_IU)
        else:
            _REF_SCANNERS[workload] = ref.glue_all(W.GLUE10 if workload == "glue10" else [W.HEADLINE])
    return _REF_SCANNERS[workload]


def host_threads(share=1):
    """Threads for the reference's static partition: what the affinity mask and the cgroup quota really give this
    process, divided between the ranks of a multi-GPU run."""
    cpus = host_cpus()
    usable = cpus["affinity"]
    if cpus["cgroup_cpu_quota"]:
        usable = min(usable, max(1, int(math.ceil(cpus["cgroup_cpu_quota"]))))
    return max(1, usable // max(1, share))


def host_sample(workload, n_sample, first_string=0):
    """A host-generated sample of a workload's corpus (the CPU arm has no GPU bytes to copy)."""
    from pire_b200 import workloads as W
    if workload == "utf8mixed":
        n_sample = min(n_sample, 1 << 17)          # mean string is 7.8 KB: ~1 GB
        sample, offsets = W.MixedSpec(n_sample, first_string=first_string).host_batch(0, n_sample)
        return sample, offsets, n_sample, int(offsets[-1]) / 1e9
    spec = W.SynthSpec(n_sample, STRING_LEN, plants=W.WORKLOADS[workload][1], first_string=first_string)
    return spec.host_sample(0, n_sample), None, n_sample, n_sample * STRING_LEN / 1e9


def time_reference(workload, sample, offsets, n_sample, gb, threads, reps):
    """The reference's own scan, Runner(sc).Begin().Run().End() per string with NonrelocScanner (its fastest variant,
    multi.h:1119-1123), statically partitioned over `threads` host threads; plus one-thread figures on a slice."""
    sc = reference_scanner(workload)
    kind = get_reference().kind
    kw = dict(offsets=offsets) if offsets is not None else dict(fixed_len=STRING_LEN)
    best, final, mask = 1e30, None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        final, mask, _ = sc.run(sample, n=n_sample, variant=1, threads=threads, want=("final", "mask"), **kw)
        best = min(best, time.perf_counter() - t0)
    k = min(n_sample, 1 << 16 if offsets is None else 1 << 13)
    kb = (k * STRING_LEN if offsets is None else int(offsets[k])) / 1e9
    t0 = time.perf_counter()
    sc.run(sample, n=k, variant=1, threads=1, want=("final",), **kw)
    t_mask = time.perf_counter() - t0
    t0 = time.perf_counter()
    sc.run(sample, n=k, variant=2, threads=1, want=("final",), **kw)
    t_nomask = time.perf_counter() - t0
    one = kb / t_mask
    out = {
        "value": gb / best, "unit": "GB/s", "cores": threads, "kind": kind,
        "sample": "%d strings of the same synthetic corpus (%.2f GB), best of %d, %s, static partition by string count" % (
            n_sample, gb, reps, "NonrelocScanner" if kind == "reference" else "oracle port (oracle/_ref absent)"),
        "matches_in_sample": int(final.sum()),
        "one_thread_GBps": one,
        "one_thread_nomask_GBps": kb / t_nomask,
        # how many threads' worth of CPU the box really delivered: the multi-thread figure over the one-thread figure
        "effective_parallelism": (gb / best) / one if one > 0 else None,
        "host_cpus": host_cpus(),
    }
    return out, final, mask


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path, all the host threads it can use, on a
    bounded sample of this arm's workload per step.  No kernel of this repository is on that path (the corpus bytes
    come from the host generator)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from pire_b200 import workloads as W
    t_all = time.perf_counter()
    per_step = min(args.cpu_sample, args.strings or args.cpu_sample)
    sample, offsets, per_step, gb = host_sample(args.workload, per_step)
    threads = host_threads()
    warm_n = per_step if offsets is not None else min(per_step, 1 << 20)
    warm_gb = gb if offsets is not None else warm_n * STRING_LEN / 1e9
    cb, _, _ = time_reference(args.workload, sample, offsets, warm_n, warm_gb, threads, 1)     # warm-up + one-thread figures
    sc = reference_scanner(args.workload)
    kw = dict(offsets=offsets) if offsets is not None else dict(fixed_len=STRING_LEN)
    times, matches = [], 0
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        final, _, _ = sc.run(sample, n=per_step, variant=1, threads=threads, want=("final", "mask"), **kw)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
        matches = int(final.sum())
    total = sum(times)
    value = gb * args.steps / total
    kind = get_reference().kind
    cb.update(value=value, cores=threads, kind=kind, matches_in_sample=matches,
              effective_parallelism=value / cb["one_thread_GBps"] if cb.get("one_thread_GBps") else None,
              sample="%d strings of the same synthetic corpus (%.2f GB) per step, %s" % (
                  per_step, gb, "NonrelocScanner" if kind == "reference" else "oracle port"))
    gpu_strings = args.strings or (MIXED_STRINGS_PER_GPU if args.workload == "utf8mixed" else STRINGS_PER_GPU)
    line = {
        "impl": "reference", "metric": "scanned GB/s", "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "%s: %s; each step = a bounded sample of %d strings (%.2f GB) on the host "
                               "(throughput-normalised: the GPU arm scans %d strings per GPU per step)" % (
                                   args.workload, W.WORKLOADS[args.workload][2], per_step, gb, gpu_strings),
                   "host_threads": threads},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "strings_per_s": per_step * args.steps / total,
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- one workload on one GPU

class Resident:
    """A workload's corpus resident on this GPU, its scanner, and the buffers a scan writes."""

    def __init__(self, workload, n_local, first_string, dev, args, variant="auto"):
        import torch
        import pire_b200 as P
        from pire_b200 import _native as N
        from pire_b200 import workloads as W
        self.workload, self.n, self.first, self.dev = workload, n_local, first_string, dev
        self.image_name, plants, self.desc, self.cfg_index = W.WORKLOADS[workload]
        self.mixed = workload == "utf8mixed"
        self.bin_ms = None
        if self.mixed:
            spec = W.MixedSpec(n_local, first_string=first_string)
            corpus, offsets = spec.device_batch(dev)
            self.batch = P.Batch(corpus, offsets, n=n_local)
            self.payload = self.batch.payload_bytes()
            t0 = time.perf_counter()
            self.batch.bin_by_length()
            torch.cuda.synchronize()
            self.bin_ms = 1e3 * (time.perf_counter() - t0)
        else:
            spec = W.SynthSpec(n_local, STRING_LEN, plants=plants, first_string=first_string)
            corpus = torch.empty(spec.total_bytes(), dtype=torch.uint8, device=dev)
            spec.fill_device(corpus)
            self.batch = P.Batch(corpus, fixed_len=STRING_LEN, n=n_local)
            self.payload = n_local * STRING_LEN
        self.corpus = corpus
        self.sc = P.Scanner(W.load_image(self.image_name), dev.index or 0)
        self.tune_ms = None
        if not args.no_tune:
            t0 = time.perf_counter()
            self.sc.Tune(self.batch, min(n_local, 16384))
            torch.cuda.synchronize()
            self.tune_ms = 1e3 * (time.perf_counter() - t0)
        self.flags = N.RUN_BEGIN | N.RUN_END
        self.masks = torch.empty(n_local, dtype=torch.int32, device=dev)
        self.bits = torch.zeros((n_local + 31) // 32, dtype=torch.int32, device=dev)
        names = dict(N.VARIANT_NAMES)
        self.variant_ms = {}
        if variant == "auto":
            self.variant_ms = self.sc.AutoSelect(self.batch)
            self.chosen = names[self.sc.info().variant]
            if self.mixed and self.variant_ms:
                # info() names the choice for uniform batches; a ragged batch runs the fastest of the variants timed on it
                self.chosen = min(self.variant_ms, key=self.variant_ms.get)
        else:
            self.chosen = variant
            self.sc.set_variant({v: k for k, v in names.items()}[variant])

    def scan(self, bits=None):
        self.sc.run_batch(self.batch, self.flags, self.bits if bits is None else bits, self.masks, None)

    def time_scan(self, reps, bits=None):
        import torch
        self.scan(bits)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            self.scan(bits)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def kernel_name(self):
        if self.mixed:
            mode = {"plain": "plain", "look": "look", "look64": "look", "look1": "look"}.get(self.chosen, "pred")
            if os.environ.get("PIRE_B200_SPLIT", "1") == "0":
                return "ScanGenericKernel<%s>" % mode
            return "ScanSplitKernel<%s> (strings >= 8 KiB, one per warp) + ScanGenericKernel<%s> (the rest)" % (
                "plain" if mode == "plain" else "pred", mode)
        look = "ScanUniformLookKernel<32 slots>" if os.environ.get("PIRE_B200_LOOK_ILP", "2") == "1" \
            else "ScanUniformLook2Kernel<%s regs> (two strings per lane, 32-slot look-ahead filter)" % os.environ.get("PIRE_B200_LOOK_ILP_REGS", "72")
        return {"priv": "ScanUniformPrivKernel", "look": look, "look1": "ScanUniformLookKernel<32 slots> (one string per lane)",
                "look64": "ScanUniformLookKernel<64 slots>"}.get(self.chosen, "ScanUniformKernel<%s>" % self.chosen)


def parity_check(res, world, bits=None, dense=1 << 22, cpu_timing=None):
    """GPU results against the reference ON THE BYTES THE GPU SCANNED (copied back from HBM).

    Fixed-length corpora: the first `dense` strings of this rank's shard, every planted string (1/8 of the corpus,
    where the automaton leaves its resting states) and every 64th 32-string unit of the rest.  Mixed-length
    corpus: three windows of 32 Ki strings (start, middle, end).  Returns (record, cpu_record):
    cpu_record = the timed multi-thread reference scan of the dense prefix when `cpu_timing` asks for one."""
    import numpy as np
    import torch
    n = res.n
    bits = res.bits if bits is None else bits
    threads = host_threads(world)
    sc_ref = reference_scanner(res.workload)
    state = {"checked": 0, "mismatches": 0, "first_bad": None}
    cpu_record = None

    def compare(idx_t, final, mask, what):
        words = bits[(idx_t // 32)]
        got_f = ((words >> (idx_t % 32).to(torch.int32)) & 1).to(torch.uint8).cpu().numpy()
        got_m = res.masks[idx_t].cpu().numpy().view(np.uint32)
        bad = np.nonzero((got_f != final) | (got_m != mask))[0]
        state["checked"] += len(final)
        state["mismatches"] += int(len(bad))
        if len(bad) and state["first_bad"] is None:
            k = int(bad[0])
            state["first_bad"] = {"string": int(idx_t[k].item()) + res.first, "sample": what, "gpu": [int(got_f[k]), int(got_m[k])],
                                  "reference": [int(final[k]), int(mask[k])]}

    if res.mixed:
        win = min(1 << 15, n)
        starts = sorted({0, max(0, (n // 2) // 32 * 32), max(0, (n - win) // 32 * 32)})
        offs_all = res.batch.offsets
        for s0 in starts:
            s1 = min(n, s0 + win)
            o = offs_all[s0:s1 + 1].cpu().numpy().astype(np.uint64)
            host = res.corpus[int(o[0]):int(o[-1])].cpu().numpy()
            final, mask, _ = sc_ref.run(host, o - o[0], n=s1 - s0, variant=1, threads=threads, want=("final", "mask"))
            compare(torch.arange(s0, s1, device=res.dev), final, mask, "window at string %d" % s0)
        what = "%d windows of %d strings (start, middle, end of the shard)" % (len(starts), win)
    else:
        dense = min(dense, n)
        rows = res.corpus[: n * STRING_LEN].view(n, STRING_LEN)
        host = rows[:dense].cpu().numpy().reshape(-1)
        if cpu_timing:
            cpu_record, final, mask = time_reference(res.workload, host, None, dense, dense * STRING_LEN / 1e9, threads, cpu_timing)
        else:
            final, mask, _ = sc_ref.run(host, fixed_len=STRING_LEN, n=dense, variant=1, threads=threads, want=("final", "mask"))
        compare(torch.arange(0, dense, device=res.dev), final, mask, "dense prefix")
        del host
        rest = torch.arange(dense, n, device=res.dev)
        if rest.numel():
            planted = (rest + res.first) % 8 == 0                     # workloads.SynthSpec: plant_every = 8
            keep = planted | ((rest // 32) % 64 == 0)
            idx = rest[keep]
            for lo in range(0, idx.numel(), 1 << 20):
                part = idx[lo:lo + (1 << 20)]
                host = rows[part].cpu().numpy().reshape(-1)
                f2, m2, _ = sc_ref.run(host, fixed_len=STRING_LEN, n=part.numel(), variant=1, threads=threads, want=("final", "mask"))
                compare(part, f2, m2, "planted + stratified")
        what = "first %d strings of the shard + every planted string + every 64th 32-string unit of the rest" % dense
    return {"checked_strings": state["checked"], "mismatches": state["mismatches"], "first_mismatch": state["first_bad"], "what": what,
            "against": "reference (oracle/_ref, NonrelocScanner)" if get_reference().kind == "reference" else "oracle port",
            "bytes": "copied back from the HBM buffer the GPU scanned"}, cpu_record


DUMP_MASKS = 1 << 21                 # accept masks written by --dump-outputs: all of them up to this many, else a seeded sample


def dump_outputs(out_dir, bits, masks):
    """What the scan hands its caller, as float64 (exact for 32-bit words): the whole match bitmap (bit i of word i // 32
    is string i) and the accept mask of every string, or of a fixed seeded sample of DUMP_MASKS strings, with their
    indices.  About 35 MB at the default 9.77 M strings.  At N > 1: the gathered bitmap and rank 0's masks."""
    import numpy as np
    import torch
    n = masks.numel()
    idx = np.arange(n) if n <= DUMP_MASKS else np.sort(np.random.default_rng(0).choice(n, DUMP_MASKS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "match_bits.npy"), bits.cpu().numpy().view(np.uint32).astype(np.float64))
    np.save(os.path.join(out_dir, "accept_mask.npy"),
            masks[torch.from_numpy(idx).to(masks.device)].cpu().numpy().view(np.uint32).astype(np.float64))
    np.save(os.path.join(out_dir, "accept_mask_string.npy"), idx.astype(np.float64))


def sub_config(workload, dev, args):
    """Another BASELINE config on its own corpus, this GPU only: throughput, roofline fraction, parity."""
    import torch
    n = (MIXED_STRINGS_PER_GPU if workload == "utf8mixed" else STRINGS_PER_GPU) // 32 * 32
    res = Resident(workload, n, 0, dev, args)
    ms = res.time_scan(5)
    peak, _ = measured_peak()
    gbps = res.payload / 1e9 / (ms / 1e3)
    out = {"workload": "BASELINE configs[%d]: %s, %d strings (%.2f GB) on its own corpus, this GPU only" % (
               res.cfg_index, res.desc, n, res.payload / 1e9),
           "value": gbps, "unit": "GB/s", "frac": gbps / peak, "kernel_ms": ms, "kernel": res.kernel_name(),
           "kernel_variant": res.chosen, "variant_ms": res.variant_ms or None, "bin_ms": res.bin_ms}
    if not args.no_parity:
        out["parity"], _ = parity_check(res, 1, dense=1 << 20)
    del res
    torch.cuda.empty_cache()
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import pire_b200 as P
    from pire_b200 import _native as N
    from pire_b200 import workloads as W
    from pire_b200.dist import Comm, popcount_bits

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the scan path has no CPU fallback (use --impl reference for the CPU arm)")
    numa = numa_bind(local) if world > 1 or os.environ.get("PIRE_B200_NUMA_BIND") else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            # VERSION and WARN both print NCCL's version banner on stdout; the contract is ONE JSON line there.  An INFO
            # (or higher) setting is somebody collecting the communicator log and is left alone.
            os.environ.pop("NCCL_DEBUG")
        dist.init_process_group("nccl", device_id=dev)
        comm = Comm(local)                           # the C ABI's communicator; torch.distributed only ships its id

    mixed = args.workload == "utf8mixed"
    n_local = (args.strings or (MIXED_STRINGS_PER_GPU if mixed else STRINGS_PER_GPU)) // 32 * 32
    n_global = n_local * world
    lo = rank * n_local
    res = Resident(args.workload, n_local, lo, dev, args, args.variant)
    payload_local = res.payload
    payload_global = payload_local
    if world > 1:
        t = torch.tensor([payload_local], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        payload_global = int(t.item())
        assert comm.bounds(n_global) == (lo, lo + n_local)

    words_local = n_local // 32
    flags = res.flags
    # two full-length bitmaps: the exchange of step k (communicator's stream) overlaps the scan of step k+1
    bits_all = [torch.zeros(words_local * world, dtype=torch.int32, device=dev) for _ in range(2 if world > 1 else 1)]

    def slot(k):
        return bits_all[k % len(bits_all)][rank * words_local:(rank + 1) * words_local]

    step_no = [0]

    def step():
        k = step_no[0]
        step_no[0] += 1
        if world == 1:
            res.scan(slot(k))
        elif args.collective == "allgather":
            comm.run_sharded(res.sc, res.batch, n_global, flags, bits_all[k % 2], res.masks, None, async_exchange=True)
        else:
            full = bits_all[k % 2]
            if rank > 0:
                full[: rank * words_local].zero_()
            if rank < world - 1:
                full[(rank + 1) * words_local:].zero_()
            res.scan(slot(k))
            dist.all_reduce(full, op=dist.ReduceOp.SUM)

    def finish_steps():
        if comm is not None and args.collective == "allgather":
            comm.wait(dev)                           # the last exchange joins the stream inside the timed region

    def barrier():
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("PIRE_B200_NO_CLOCKS") else None
    for _ in range(max(args.warmup, 3)):
        step()
    finish_steps()
    launches0 = N.lib.pire_gpu_launch_count()
    barrier()
    torch.cuda.synchronize()
    t_begin = time.perf_counter()
    e0 = torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e0.record()
    for i in range(args.steps):
        step()
        if i == args.steps - 1:
            finish_steps()
        marks[i].record()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    barrier()
    elapsed_ms = e0.elapsed_time(marks[-1])
    per_step = sorted((marks[i - 1] if i else e0).elapsed_time(marks[i]) for i in range(args.steps))
    launches = N.lib.pire_gpu_launch_count() - launches0
    clocks = sampler.stop(t_begin, t_end) if sampler else None
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = payload_global / 1e9 / (ms_per_step / 1e3)

    last = (step_no[0] - 1) % len(bits_all)
    bits_full = bits_all[last]
    bits_local = slot(last)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bits_full, res.masks)
    # the scan kernel alone (CUDA events around the launches only), for the roofline
    kernel_ms = res.time_scan(min(args.steps, 10), bits_local)
    torch.cuda.synchronize()
    matches_global = popcount_bits(bits_full)
    matches_local_masks = int((res.masks != 0).sum().item())
    local_pop = torch.tensor([popcount_bits(bits_local)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(local_pop, op=dist.ReduceOp.SUM)
    assert int(local_pop.item()) == matches_global, (int(local_pop.item()), matches_global)    # the gathered bitmap is the union of the shards
    assert matches_local_masks == popcount_bits(bits_local)
    assert matches_local_masks >= (n_local // 8) * (0.9 if mixed else 1.0)      # strings < 32 B carry no plant

    # parity at config size, every rank on its own shard; rank 0 also times the reference on the dense prefix
    parity = cpu_baseline = None
    failed = False
    if not args.no_parity:
        want_cpu = 3 if (rank == 0 and world == 1 and not args.no_cpu and not mixed) else None
        parity, cpu_baseline = parity_check(res, world, bits=bits_local, dense=min(args.cpu_sample, 1 << 22), cpu_timing=want_cpu)
        parity["ranks"] = world
        if world > 1:
            # every rank checked its own shard; rank 0 also checks the GATHERED bitmap: every slot against that rank's bits
            t = torch.tensor([parity["checked_strings"], parity["mismatches"]], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            gathered = [torch.empty_like(bits_local) for _ in range(world)] if rank == 0 else None
            dist.gather(bits_local.contiguous(), gathered, dst=0)
            if rank == 0:
                slots_equal = all(torch.equal(gathered[r], bits_full[r * words_local:(r + 1) * words_local]) for r in range(world))
                parity["gathered_bitmap_equals_rank_slots"] = bool(slots_equal)
                parity["checked_strings"], parity["mismatches"] = int(t[0].item()), int(t[1].item()) + (0 if slots_equal else 1)
        failed = parity["mismatches"] != 0

    # end to end: host buffers through the C ABI, H2D and D2H inside the timed region (and the exchange at N > 1)
    e2e = None
    if not args.no_e2e:
        try:
            host = torch.empty(payload_local, dtype=torch.uint8, pin_memory=True)
            host.copy_(res.corpus[:payload_local])
            host_offs = None
            if mixed:
                host_offs = torch.empty(n_local + 1, dtype=torch.int64, pin_memory=True)
                host_offs.copy_(res.batch.offsets)
            torch.cuda.synchronize()
            hb = torch.empty(words_local, dtype=torch.int32, pin_memory=True)
            hm = torch.empty(n_local, dtype=torch.int32, pin_memory=True)
            e2e_bits = torch.zeros(words_local * world, dtype=torch.int32, device=dev)

            def e2e_step(buf):
                N.check(N.lib.pire_gpu_run_batch_host(res.sc._h, buf.ctypes.data, payload_local,
                                                      host_offs.data_ptr() if mixed else None,
                                                      0 if mixed else STRING_LEN, n_local,
                                                      flags, hb.data_ptr(), hm.data_ptr(), None), "run_batch_host")
                if comm is not None:                 # the sharded call's exchange: this rank's bits up, every slot gathered
                    e2e_bits[rank * words_local:(rank + 1) * words_local].copy_(hb, non_blocking=True)
                    comm.gather_bits(n_global, e2e_bits)
                    torch.cuda.current_stream().synchronize()

            def timed(buf, steps):
                e2e_step(buf)
                barrier()
                t0 = time.perf_counter()
                for _ in range(steps):
                    e2e_step(buf)
                dt = time.perf_counter() - t0
                if world > 1:
                    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    dt = float(tt.item())
                return payload_global / 1e9 / (dt / steps)

            e2e_steps = max(1, min(args.steps, 3))
            pinned_gbps = timed(host.numpy(), e2e_steps)
            assert torch.equal(hb, bits_local.cpu()) and torch.equal(hm, res.masks.cpu())
            if comm is not None:
                assert torch.equal(e2e_bits, bits_full)
            e2e = {"value": pinned_gbps, "unit": "GB/s",
                   "h2d_bytes_per_step": payload_local + (8 * (n_local + 1) if mixed else 0),
                   "d2h_bytes_per_step": words_local * 4 + n_local * 4,
                   "steps": e2e_steps,
                   "api": "pire_gpu_run_batch_host: pinned host corpus in, bitmap + accept masks out, streamed in 64 MiB chunks "
                          "(H2D of chunk k+1 overlaps the scan of chunk k)" + ("; then the NCCL gather of the bitmap slots" if comm else ""),
                   "numa": numa}
            # the caller the reference has: a pageable const char* (run.h:271-275)
            try:
                pageable = np.empty(payload_local, np.uint8)
                pageable[:] = host.numpy()
                hb.zero_()
                e2e["pageable"] = {"value": timed(pageable, max(1, min(e2e_steps, 2))), "unit": "GB/s",
                                   "note": "pageable host corpus, staged through the library's pinned buffers by its copy threads"}
                assert torch.equal(hb, bits_local.cpu())
                del pageable
            except Exception as ex:      # noqa: BLE001
                e2e["pageable"] = {"value": None, "error": repr(ex)}
            del host
        except Exception as ex:          # e.g. not enough pinnable host memory
            e2e = {"value": None, "unit": "GB/s", "error": repr(ex)}

    # the rows next to the path (SURVEY 8f) on the same resident bytes, a few launches each
    next_rows = None
    if not mixed and not args.no_next:
        try:
            lens = torch.empty(n_local, dtype=torch.int32, device=dev)
            hf = P.Scanner(W.load_image("hf_glue10"), local)
            counts = torch.empty((n_local, hf.RegexpsCount()), dtype=torch.int32, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream

            def prefix_run():
                N.check(N.lib.pire_gpu_prefix_batch(res.sc._h, res.corpus.data_ptr(), None, STRING_LEN, n_local, flags, 0, lens.data_ptr(), stream),
                        "pire_gpu_prefix_batch")

            def count_run():
                N.check(N.lib.pire_gpu_count_batch(hf._h, res.corpus.data_ptr(), None, STRING_LEN, n_local, flags, counts.data_ptr(), None,
                                                   stream), "pire_gpu_count_batch")
            next_rows = {}
            for key, fn in (("longest_prefix", prefix_run), ("half_final_count_hf_glue10", count_run)):
                fn()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a0.record()
                for _ in range(3):
                    fn()
                a1.record()
                torch.cuda.synchronize()
                next_rows[key] = {"value": payload_local / 1e9 / (a0.elapsed_time(a1) / 3 / 1e3), "unit": "GB/s"}
            next_rows["note"] = "this GPU only, same resident corpus; parity of these entry points is in tests/test_gpu_parity.py"
            del lens, counts, hf
        except Exception as ex:      # noqa: BLE001
            next_rows = {"error": repr(ex)}

    info = res.sc.info()
    chosen, variant_ms, bin_ms, tune_ms = res.chosen, res.variant_ms, res.bin_ms, res.tune_ms
    kernel_name, desc, cfg_index = res.kernel_name(), res.desc, res.cfg_index
    del res
    torch.cuda.empty_cache()

    # the other BASELINE configs on their own corpora (one GPU)
    configs = None
    if rank == 0 and world == 1 and not args.no_configs and not args.strings:
        configs = {}
        for other in ("headline", "glue10", "utf8mixed"):
            if other == args.workload:
                continue
            key = "configs[%d]" % W.WORKLOADS[other][3]
            try:
                configs[key] = sub_config(other, dev, args)
                failed = failed or configs[key].get("parity", {}).get("mismatches", 0) != 0
            except Exception as ex:      # noqa: BLE001
                configs[key] = {"error": repr(ex)}

    if rank != 0:
        if comm is not None:
            comm.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    achieved = payload_local / 1e9 / (kernel_ms / 1e3)
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(args.workload)
    except Exception:
        pass
    line = {
        "metric": "scanned GB/s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "step_ms": {"min": per_step[0], "median": per_step[len(per_step) // 2], "max": per_step[-1]} if per_step else None,
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[%d]: %s; %d synthetic strings per GPU (%.2f GB/GPU), "
                        "1/8 of the strings carry a planted match" % (
                            4 if (world > 1 and args.workload == "glue10") else cfg_index,
                            desc if mixed else desc + " over 1 KiB printable-ASCII strings", n_local, payload_local / 1e9),
            "strings_per_gpu": n_local, "string_len": "16..65535 (CSR, binned by length on device)" if mixed else STRING_LEN,
            "bin_ms": bin_ms, "outputs": "match bitmap + u32 accept mask per string",
            "kernel_variant": chosen, "variant_ms": variant_ms or None, "hot_rows": info.hot_rows, "tuned": bool(info.tuned),
            "tune_ms": tune_ms, "l2": "input (%.1f GB) is far larger than L2; no flush needed" % (payload_local / 1e9),
            "collective": (("pire_gpu_run_sharded: in-place NCCL all-gather of the bitmap slots on the communicator's stream, "
                            "overlapping the next step's scan") if args.collective == "allgather"
                           else "torch.distributed all-reduce(SUM) of the zeroed full bitmap, serialized") if world > 1 else "none (1 GPU)",
        },
        "strings_per_s": n_global / (ms_per_step / 1e3),
        "matches": matches_global, "matches_local_by_mask": matches_local_masks,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": kernel_name, "kernel_ms": kernel_ms,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": payload_local},
        "clocks": clocks,
        "parity": parity,
        "e2e": e2e,
        "configs": configs,
        "next_rows": next_rows,
    }
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    elif not args.no_cpu and world == 1:
        try:
            sample, offsets, ns, gb = host_sample(args.workload, min(args.cpu_sample, n_local))
            line["cpu_baseline"], _, _ = time_reference(args.workload, sample, offsets, ns, gb, host_threads(), 3)
        except Exception as ex:      # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
    if failed:
        line["parity_failed"] = True
    print(json.dumps(line))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main())
