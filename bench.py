#!/usr/bin/env python
"""bench.py -- benchmark of the protocol.Decoder hot path on B200 (BASELINE.json configs 2-5).

Metric (BASELINE.json): IQ Msamples/s decoded (1 sample = I byte + Q byte) on synthetic uint8 IQ
with injected ERT packets.

  python bench.py --gpus N --steps K --warmup W            our arm (libertgpu.so, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm: the reference's algorithm on
                                                           the box's host cores (oracle port: Go
                                                           is not in this image, see DESIGN.md)

Workloads (`--config`, default `scm1g`; all ChipLength 72 = `-symbollength=72`):
  scm1g    BASELINE configs[1]  scm, 1 GiB of IQ per GPU                   <- the headline line
  multi8g  BASELINE configs[2]  scm,scm+,idm (three preambles, one pass), 8 GiB, 1 GPU
  r9004g   BASELINE configs[3]  r900 (incl. the parser's filter+quantize), 4 GiB, 1 GPU
  scm8g    BASELINE configs[4]  scm, 8 GiB per GPU (64 GiB over 8 GPUs)
The line of the headline workload carries a `configs` array with the other workloads measured in the
same run (N = 1: multi8g, r9004g, scm8g; N > 1: scm8g per GPU, i.e. configs[4] at N = 8), each with its
own value, stage times and roofline; `--no-extras` skips them, `--config X` makes X the headline.

For N > 1 the driver launches one rank per GPU with torch.distributed.run; the stream is cut into
N contiguous block-aligned shards (weak scaling) with a leading halo, and there is no collective on
the data path (SURVEY.md section 8e); torch.distributed is used for the barrier and the max-over-ranks
of the device time only.

One JSON line is printed by rank 0.  `value` = whole-job Msamples/s with the IQ resident in HBM
(CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks);
`e2e` = the same through the C-ABI call `ertgpu_decode` with pinned HOST buffers (H2D inside the
timed region); `roofline` = the demod kernel against the measured HBM copy bandwidth;
`cpu_baseline` = the CPU restatement timed on this box (bounded sample); `sustained` = the same
step repeated for >= 2 s.

`--dump-outputs DIR` (GPU arm) writes, for each workload, what the last of the K timed steps
returned: the candidate records of ertgpu_fetch and the counters of ertgpu_last_counts, as
float64 / float32 arrays DIR/<workload>_<field>.npy (see dump_outputs).  The inputs are seeded,
so two builds run with the same arguments can be compared file for file.
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
sys.path.insert(0, ROOT)

CHIP_LENGTH = 72
PACKET_SPACING = 1 << 20
UNIT = "Msamples/s"
WORKLOADS = {
    # name: msgtypes, bytes per GPU, seed (SURVEY.md 8d: 0x5EED0001...5 per config), BASELINE.json config index
    "scm1g": dict(msgtype="scm", bytes=1 << 30, seed=0x5EED0002, baseline_config=1, multi_gpu=True),
    "multi8g": dict(msgtype="scm,scm+,idm", bytes=8 << 30, seed=0x5EED0003, baseline_config=2, multi_gpu=False),
    "r9004g": dict(msgtype="r900", bytes=4 << 30, seed=0x5EED0004, baseline_config=3, multi_gpu=False),
    "scm8g": dict(msgtype="scm", bytes=8 << 30, seed=0x5EED0005, baseline_config=4, multi_gpu=True),
}
KEY_BYTES = {"scm": 12, "scm+": 16, "idm": 92, "netidm": 92}


def metric_name(w):
    return f"IQ Msamples/s decoded ({w['msgtype']}, ChipLength {CHIP_LENGTH}, synthetic uint8 IQ with injected ERT packets)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="scm1g", choices=sorted(WORKLOADS))
    ap.add_argument("--bytes-per-gpu", type=int, default=0, help="override the workload's size (testing)")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0, help="reference arm: threads (default: every CPU the process may use)")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step of each workload returned as DIR/<workload>_<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(name, w, nbytes_per_gpu, world, bs, pkl):
    """The `config` object: identical in both arms (same workload => same dict)."""
    from rtlamr_b200 import shard
    blocks_per_gpu = nbytes_per_gpu // (2 * bs)
    plans = shard.plan(blocks_per_gpu * world, world, bs, pkl)
    return {
        "workload": f"{name}: {w['msgtype']} ChipLength={CHIP_LENGTH} (SymbolLength {2 * CHIP_LENGTH}, BlockSize {bs}), "
                    f"{nbytes_per_gpu >> 20} MiB synthetic uint8 IQ per GPU x {world} GPU(s), one injected packet per 2^20 samples "
                    f"(BASELINE.json configs[{w['baseline_config']}])",
        "msgtype": w["msgtype"], "chip_length": CHIP_LENGTH, "block_size": bs, "bytes_per_gpu": nbytes_per_gpu,
        "blocks_per_gpu": blocks_per_gpu, "total_bytes": nbytes_per_gpu * world, "seed": w["seed"],
        "halo_blocks": max(p.halo_blocks for p in plans),
        "l2": "input per step exceeds the 126 MB L2: no flush needed",
        "sharding": "contiguous block-aligned shards + halo, no collective on the data path",
    }


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every
    ~0.5 ms from a thread, with the `nvidia-smi -lms` recipe as fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml, self.stop_flag, self.thread = None, False, None

    def _visible_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except Exception:
                return self.gpu
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self._visible_index()}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
                rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((time.time(), sm, mx, rs))
            except Exception:
                pass
            time.sleep(0.0005)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0: float, t1: float):
        """Summary of the samples taken in [t0, t1] (the sampler keeps running)."""
        if self.nvml is not None:
            n = self.nvml
            rows = [r for r in list(self.rows) if t0 <= r[0] <= t1] or list(self.rows)[-3:]
            sm = sorted(r[1] for r in rows)
            bits = 0
            for r in rows:
                bits |= r[3]
            names = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            reasons = sorted(k for k, v in names.items() if bits & v)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": rows[0][2] if rows else None,
                    "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        sm, smax, reasons = [], None, set()
        allrows = list(self.rows)
        rows = [r for (t, r) in allrows if t0 - 0.05 <= t <= t1 + 0.05] or [r for (_, r) in allrows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()


# ----------------------------------------------------------------------------- CPU arm
def host_topology():
    """(CPUs this process may use, physical cores among them, cgroup CPU quota in CPUs or None)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                cores.add(f.read().strip())
        except OSError:
            cores.add(str(c))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts and parts[0] != "max":
                    quota = float(parts[0]) / float(parts[1])
            else:
                q = float(parts[0])
                with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                    per = float(f2.read().split()[0])
                if q > 0:
                    quota = q / per
            break
        except (OSError, ValueError, IndexError):
            continue
    return len(cpus), len(cores), quota


def pick_cpu_threads(msgtype, iq_sample, ncpu, ncores, quota):
    """Thread count for the whole-host CPU figure: the fastest of {physical cores, logical CPUs, the cgroup quota}
    on a short calibration sample (SMT helps this latency-bound loop on some hosts, a CPU quota punishes it on others)."""
    cands = sorted({ncpu, ncores} | ({max(1, int(round(quota)))} if quota else set()))
    best, rates = cands[-1], {}
    for t in cands:
        rates[t] = cpu_rate(msgtype, iq_sample, t)[0]
    best = max(rates, key=rates.get)
    return best, {str(k): round(v, 1) for k, v in rates.items()}


def cpu_rate(msgtype, iq, nthreads: int, repeats: int = 1):
    """Msamples/s of the CPU restatement (oracle/ert_oracle.c driven by oracle/ert_oracle_bench.c: Go-faithful
    Search, parsers included): `nthreads` independent decoders over contiguous block-aligned shards of one
    stream, each block one Decode call like main.go:235.  Threads, per-thread decoders and output arrays are
    set up outside the timed region; everything timed runs in C."""
    import oracle
    dt, nc, nm, nblocks = oracle.bench_threads(msgtype, CHIP_LENGTH, iq, nthreads, repeats)
    o = oracle.Oracle(msgtype, CHIP_LENGTH)
    nsamples = nblocks * o.cfg.block_size * repeats
    o.close()
    return nsamples / dt / 1e6, dt, nc, nm


def run_reference(args):
    if args.dump_outputs:
        raise SystemExit("--dump-outputs: the reference arm returns counts only; dumps come from the GPU arm")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np

    import oracle  # noqa: F401  (the reference arm is the one place besides cpu_baseline where bench.py executes oracle/)
    from rtlamr_b200 import synth

    w = WORKLOADS[args.config]
    world = args.gpus
    nbytes_per_gpu = args.bytes_per_gpu or w["bytes"]
    o = oracle.Oracle(w["msgtype"], CHIP_LENGTH)
    bs, bs2, pkl = o.cfg.block_size, o.cfg.block_size2, o.cfg.packet_length
    o.close()
    nbytes_per_gpu = nbytes_per_gpu // bs2 * bs2
    cfg = workload_config(args.config, w, nbytes_per_gpu, world, bs, pkl)
    ncpu, ncores, quota = host_topology()
    # the whole job's stream, bounded so that a run stays within minutes and within host memory
    total = nbytes_per_gpu * world
    cap = 8 << 30
    sample_bytes = min(total, cap) // bs2 * bs2
    nsamples = sample_bytes // 2
    pk, _ = synth.make_packets(w["msgtype"], CHIP_LENGTH, total // 2, seed=1, spacing=PACKET_SPACING)
    iq = synth.host_fill(0, nsamples, w["seed"], pk, nthreads=ncpu)
    calib = None
    if args.cpu_threads:
        nthreads = args.cpu_threads
    else:
        nthreads, calib = pick_cpu_threads(w["msgtype"], iq[: min(sample_bytes, 256 << 20) // bs2 * bs2], ncpu, ncores, quota)
    for _ in range(max(0, min(args.warmup, 2))):
        cpu_rate(w["msgtype"], iq, nthreads)
    vals, t_tot, nmsg = [], 0.0, 0
    steps = max(1, args.steps)
    for _ in range(steps):
        v, dt, nc, nm = cpu_rate(w["msgtype"], iq, nthreads)
        vals.append(v)
        t_tot += dt
        nmsg = nm
    value = nsamples * steps / t_tot / 1e6
    v1, dt1, _, _ = cpu_rate(w["msgtype"], iq[: min(sample_bytes, 256 << 20) // bs2 * bs2], 1)
    sample = (f"the whole stream of the workload ({sample_bytes >> 20} MiB{'' if sample_bytes == total else f' of {total >> 20} MiB'}) per step, "
              f"cut into {nthreads} contiguous block-aligned shards, one decoder thread per shard (pinned), every block one Decode call")
    line = {
        "impl": "reference", "metric": metric_name(w), "value": round(value, 1), "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t_tot / steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": nthreads, "kind": "port",
                         "physical_cores": ncores, "logical_cpus": ncpu, "cgroup_cpu_quota": quota,
                         "thread_count_calibration": calib,
                         "one_core_value": round(v1, 1), "speedup_over_one_core": round(value / v1, 1),
                         "messages_per_step": int(nmsg),
                         "sample": sample + "; C restatement of the Go Decoder incl. Search and parsers (oracle/ert_oracle.c) "
                                            "because no Go toolchain is present"},
        "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- GPU arm
def recovered_keys(got, msgtypes):
    """Identity of every candidate that passed a screen: (msgtype, packet bytes) / (r900, 21 symbols)."""
    import numpy as np
    keys = set()
    for i, mt in enumerate(msgtypes):
        sel = got[(got["check_mask"] >> i) & 1 == 1]
        if len(sel) == 0:
            continue
        if mt in ("r900", "r900bcd"):
            d = sel["r900_digits"].astype(np.int32)
            sym = d[:, 0::2] * 6 + d[:, 1::2]
            for row in np.unique(sym, axis=0):
                keys.add((mt, bytes(row.astype(np.uint8))))
        else:
            nb = KEY_BYTES[mt]
            for row in np.unique(sel["bytes"][:, :nb], axis=0):
                keys.add((mt, bytes(row)))
    return keys


class Job:
    """One workload on this rank's GPU: shard plan, resident synthetic IQ, decoder handle."""

    def __init__(self, name, args, world, rank, local):
        import torch

        from rtlamr_b200 import capi, shard, synth
        self.name, self.w = name, WORKLOADS[name]
        self.world, self.rank, self.local = world, rank, local
        w = self.w
        self.msgtypes = [m.strip() for m in w["msgtype"].split(",")]
        probe = capi.new_decoder(w["msgtype"], CHIP_LENGTH, device=local, max_blocks_per_call=1)
        self.cfg = probe.cfg
        bs, bs2, pkl = self.cfg.block_size, self.cfg.block_size2, self.cfg.packet_length
        probe.close()
        nbytes_per_gpu = (args.bytes_per_gpu or w["bytes"]) // bs2 * bs2
        self.blocks_per_gpu = nbytes_per_gpu // bs2
        self.config = workload_config(name, w, nbytes_per_gpu, world, bs, pkl)
        self.plan = shard.plan(self.blocks_per_gpu * world, world, bs, pkl)[rank]
        self.nblocks = self.plan.last_block - self.plan.first_fed_block          # halo + owned blocks
        self.nbytes = self.nblocks * bs2
        self.nsamples = self.nblocks * bs
        self.total_samples = self.blocks_per_gpu * world * bs
        first_sample = self.plan.first_fed_block * bs
        self.h = capi.new_decoder(w["msgtype"], CHIP_LENGTH, device=local, max_blocks_per_call=self.nblocks,
                                  max_candidates=1 << 20)
        self.pk, self.truth = synth.make_packets(w["msgtype"], CHIP_LENGTH, self.total_samples, seed=1, spacing=PACKET_SPACING)
        self.d_iq = torch.empty(self.nbytes, dtype=torch.uint8, device="cuda")
        capi.synth_fill(local, self.d_iq.data_ptr(), first_sample, self.nsamples, w["seed"], self.pk)
        self.flags = capi.DECODE_ONLY_VALID

    def close(self):
        self.h.close()
        self.d_iq = None

    def step_device(self, st, fetch=False):
        """One pass of the hot path over the resident batch: fresh stream, every kernel of the pipeline,
        then the per-step result read-back (candidate / valid counters, D2H)."""
        h = self.h
        h.reset()
        h.decode_device_async(self.d_iq.data_ptr(), self.nbytes, self.flags, st)
        counts = h.last_counts()
        return h.fetch(1 << 20) if fetch else counts

    def gate(self, st):
        """Correctness gate (untimed): every injected packet this rank owns decodes and passes its screen."""
        got = self.step_device(st, fetch=True)
        got = got[got["block"] >= (self.plan.first_block - self.plan.first_fed_block)]
        keys = recovered_keys(got, self.msgtypes)
        bs, buf, sl = self.cfg.block_size, self.cfg.buffer_length, self.cfg.symbol_length
        mine = [t for t in self.truth if self.plan.owns_start(t.start_sample + sl, bs, buf)
                and t.start_sample + buf < self.total_samples]
        missing = [t for t in mine if (t.msgtype, t.data) not in keys]
        if missing:
            raise SystemExit(f"rank {self.rank} [{self.name}]: {len(missing)} of {len(mine)} injected packets not recovered")
        return len(keys)


def measure(job, args, barrier, sampler, stream, with_e2e, sustained_s):
    """Timed regions of one workload.  Returns this rank's raw numbers."""
    import torch
    st = stream.cuda_stream
    h = job.h
    n_pkts = job.gate(st)
    for _ in range(max(args.warmup, 3)):
        job.step_device(st)
    def timed(nsteps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        t0 = time.time()
        e0.record(stream)
        for _ in range(nsteps):
            job.step_device(st)
            launches += h.last_launches()
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1), launches, t0, time.time()

    # timed region 1: the K steps behind `value` (no events inside a step: Search and Slice are programmatic
    # dependents of the kernel in front of them and move in while it drains)
    ms_total, launches, t_wall0, t_wall1 = timed(args.steps)
    out = {"ms_total": ms_total, "launches": launches, "n_pkts": n_pkts,
           "clocks": sampler.window(t_wall0, t_wall1) if sampler else None}
    if args.dump_outputs:
        # the last timed step's results are still in the handle: read them back outside the timed window
        out["records"], out["counts"] = h.fetch(1 << 20), h.last_counts()
    # timed region 2: the same K steps with CUDA events recorded by the library around each stage (the roofline's
    # kernel time); the events sit between the kernels, so this pass runs them strictly one after another
    h.set_stage_timing(True)
    ms_total2, _, _, _ = timed(args.steps)
    stage_mean, stage_n = h.stage_ms_mean()
    assert stage_n == args.steps
    out["stage_ms"] = stage_mean
    out["ms_total_staged"] = ms_total2
    h.set_stage_timing(False)

    if sustained_s > 0:
        # the same step back to back for >= sustained_s seconds (clocks settle under the power cap)
        per = max(1, int(0.25 / max(out["ms_total"] / args.steps * 1e-3, 1e-6)))
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.time()
        s0.record(stream)
        nsteps = 0
        while time.time() - tw0 < sustained_s:
            for _ in range(per):
                job.step_device(st)
            nsteps += per
        s1.record(stream)
        barrier()
        tw1 = time.time()
        out["sustained"] = {"ms_total": s0.elapsed_time(s1), "steps": nsteps,
                            "clocks": sampler.window(tw0, tw1) if sampler else None}

    if with_e2e:
        import numpy as np
        # ---- end to end through the C-ABI call with pinned host memory (H2D inside the timed region); the buffer is
        # allocated by this thread after it was bound to the GPU's NUMA node (ertgpu_bind_host_thread)
        host = torch.empty(job.nbytes, dtype=torch.uint8, pin_memory=True)
        host.copy_(job.d_iq)
        torch.cuda.synchronize()

        def step_host(ptr):
            h.reset()
            return h.decode((ptr, job.nbytes), job.flags, 1 << 20)

        for _ in range(2):
            step_host(host.data_ptr())
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(args.steps):
            r = step_host(host.data_ptr())
            d2h = r.nbytes + 24
        torch.cuda.synchronize()
        out["e2e_s"] = time.perf_counter() - t0
        out["d2h_bytes"] = d2h
        barrier()
        # ---- the same call with PAGEABLE input (what a Go slice is): the library stages it through its own pinned buffers
        pg = np.array(host.numpy(), copy=True)
        del host
        step_host(pg.ctypes.data)
        barrier()
        t0 = time.perf_counter()
        nrep = max(1, min(args.steps, 3))
        for _ in range(nrep):
            step_host(pg.ctypes.data)
        torch.cuda.synchronize()
        out["e2e_pageable_s"] = (time.perf_counter() - t0) / nrep
        barrier()
    return out


def reduce_over_ranks(world, vals_max, vals_sum):
    import torch
    import torch.distributed as dist
    if world == 1:
        return vals_max, vals_sum
    t = torch.tensor(vals_max, dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s = torch.tensor(vals_sum, dtype=torch.float64, device="cuda")
    dist.all_reduce(s, op=dist.ReduceOp.SUM)
    return [float(x) for x in t], [float(x) for x in s]


def summarise(job, args, raw, world, peak, peak_src):
    """Whole-job numbers of one workload from the rank-reduced raw times."""
    steps = args.steps
    ms_per_step = raw["ms_total"] / steps
    value = job.total_samples / (ms_per_step * 1e-3) / 1e6
    dm = raw["stage_ms"]["demod"]
    achieved = 2.0 * job.nsamples / (dm * 1e-3) / 1e9   # 2 algorithmic bytes per sample (SURVEY.md 8d), this rank's launch
    step_bw = 2.0 * job.nsamples / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "demod_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_sample", 0) * job.nsamples or None
            traffic_src = f"from profile: {tj.get('source', 'profiles/demod_traffic.json')} (dram bytes per sample x samples per launch), not captured in this run"
        except Exception:
            traffic = None
    kern = job.h.demod_kernel_name()
    res = {
        "name": job.name, "metric": metric_name(job.w), "value": round(value, 1), "unit": UNIT,
        "ms_per_step": round(ms_per_step, 4), "config": job.config,
        "pkts_per_step": int(raw["n_pkts"]), "pkts_per_s": round(raw["n_pkts"] / (ms_per_step * 1e-3), 1),
        "gpu_launches": int(raw["launches"]),
        "stage_ms": {k: round(v, 4) for k, v in raw["stage_ms"].items()},
        "stage_ms_note": "second timed pass of the same K steps with CUDA events around each stage (kernels strictly serialised); "
                         f"that pass took {raw['ms_total_staged'] / steps:.4f} ms per step",
        "roofline": {"bound": "hbm", "kernel": kern, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "algorithmic_bytes": "2 B per IQ sample x samples per launch",
                     "whole_step_frac": round(step_bw / peak, 4)},
        "clocks": raw["clocks"],
    }
    if "sustained" in raw:
        s = raw["sustained"]
        ms = s["ms_total"] / s["steps"]
        res["sustained"] = {"value": round(job.total_samples / (ms * 1e-3) / 1e6, 1), "unit": UNIT, "ms_per_step": round(ms, 4),
                            "steps": s["steps"], "seconds": round(s["ms_total"] * 1e-3, 2), "clocks": s["clocks"]}
    if "e2e_s" in raw:
        e2e_value = job.total_samples / (raw["e2e_s"] / steps) / 1e6
        res["e2e"] = {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": job.nbytes * world,
                      "d2h_bytes_per_step": int(raw["d2h_bytes"]) * world,
                      "api": "ertgpu_decode (C ABI), pinned host input (NUMA-local to the GPU), chunked H2D overlapped with kernels",
                      "pageable_input_value": round(job.total_samples / raw["e2e_pageable_s"] / 1e6, 1),
                      "pageable_note": "same call on ordinary (pageable) host memory, e.g. a Go slice: staged through the library's pinned buffers"}
    return res


DUMP_BYTES = 60 << 20   # --dump-outputs: the rows of all workloads together; with the .npy headers under 64 MB


def dump_outputs(directory, tag, job, records, counts, budget):
    """DIR/<tag>_<field>.npy: the candidate records a caller gets from ertgpu_fetch, in (block, preamble_id, idx)
    order, one array per field -- block, idx, preamble_id, check_mask, flags (float64), bytes[:, :packet_bytes]
    and, for r900 workloads, r900_digits (float32) -- plus `counts` = ertgpu_last_counts (candidates, valid).
    If the records need more than `budget` bytes, a fixed seeded sample of rows is kept; `row` holds the
    record numbers written either way."""
    import numpy as np
    cols = {f: records[f].astype(np.float64) for f in ("block", "idx", "preamble_id", "check_mask", "flags")}
    cols["bytes"] = records["bytes"][:, :job.cfg.packet_bytes].astype(np.float32)
    if any(m.startswith("r900") for m in job.msgtypes):
        cols["r900_digits"] = records["r900_digits"].astype(np.float32)
    row_bytes = 8 + sum(c.itemsize * (c.size // max(1, len(c))) for c in cols.values())
    rows = np.arange(len(records))
    if len(rows) * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), budget // row_bytes, replace=False))
    cols = {k: v[rows] for k, v in cols.items()}
    cols["row"] = rows.astype(np.float64)
    cols["counts"] = np.array(counts, dtype=np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, v in cols.items():
        np.save(os.path.join(directory, f"{tag}_{k}.npy"), v)


def run_b200(args):
    import torch
    import torch.distributed as dist

    from rtlamr_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    numa = None
    try:
        affinity0 = os.sched_getaffinity(0)
    except AttributeError:
        affinity0 = None
    if not args.no_numa_bind:
        numa = capi.bind_host_thread(local)   # this process and its pinned buffers live next to the GPU
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sampler = None
    if rank == 0:
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.05)
    peaks = {}
    pp = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pp):
        peaks = json.load(open(pp))
    peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")

    names = [args.config]
    if not args.no_extras and args.config == "scm1g":
        names += ["scm8g"] if world > 1 else ["multi8g", "r9004g", "scm8g"]
    results, cpu = [], None
    for i, name in enumerate(names):
        if world > 1 and not WORKLOADS[name]["multi_gpu"] and i > 0:
            continue
        job = Job(name, args, world, rank, local)
        head = i == 0
        raw = measure(job, args, barrier, sampler, stream, with_e2e=head, sustained_s=args.sustained_seconds if head else 0.0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, name if world == 1 else f"{name}_rank{rank}", job, raw["records"], raw["counts"],
                         DUMP_BYTES // (len(names) * world))
        mx = [raw["ms_total"], raw.get("e2e_s", 0.0), raw.get("e2e_pageable_s", 0.0), raw["sustained"]["ms_total"] if "sustained" in raw else 0.0]
        sm = [float(raw["n_pkts"])]
        mx, sm = reduce_over_ranks(world, mx, sm)
        raw["ms_total"], raw["n_pkts"] = mx[0], sm[0]
        if "e2e_s" in raw:
            raw["e2e_s"], raw["e2e_pageable_s"] = mx[1], mx[2]
        if "sustained" in raw:
            raw["sustained"]["ms_total"] = mx[3]
        if rank == 0:
            results.append(summarise(job, args, raw, world, peak, peak_src))
        if head and rank == 0 and world == 1 and not args.skip_cpu_baseline:
            # cpu_baseline: one core on a bounded sample (the reference's DSP is one goroutine), then every host CPU
            # on the whole stream; the bytes are the workload's own (copied back from the GPU)
            nb = min(job.nbytes, 256 << 20) // job.cfg.block_size2 * job.cfg.block_size2
            iq = job.d_iq.cpu().numpy()
            if affinity0 is not None:
                os.sched_setaffinity(0, affinity0)     # the CPU figure uses every CPU of the host, not only the GPU's node
            ncpu, ncores, quota = host_topology()
            v1, dt1, _, nm1 = cpu_rate(job.w["msgtype"], iq[:nb], 1, repeats=12)
            nthr, calib = pick_cpu_threads(job.w["msgtype"], iq[:nb], ncpu, ncores, quota)
            vall, dtall, _, _ = cpu_rate(job.w["msgtype"], iq, nthr, repeats=4)
            cpu = {"value": round(v1, 1), "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"first {nb >> 20} MiB of the workload's stream decoded 12x by one decoder thread ({dt1:.1f} s), every block one "
                             f"Decode call; C restatement of the Go Decoder incl. Search and parsers, Go toolchain absent",
                   "all_cpus": {"value": round(vall, 1), "threads": nthr, "physical_cores": ncores, "logical_cpus": ncpu,
                                "cgroup_cpu_quota": quota, "thread_count_calibration": calib,
                                "sample": f"the whole {job.nbytes >> 20} MiB stream 4x over {nthr} pinned decoder threads ({dtall:.1f} s)"}}
        job.close()
        torch.cuda.empty_cache()

    if rank == 0:
        sampler.stop()
        head = results[0]
        line = {
            "metric": head["metric"], "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": head["config"],
            "pkts_per_s": head["pkts_per_s"], "pkts_per_step": head["pkts_per_step"],
            "e2e": head.get("e2e"), "gpu_launches": head["gpu_launches"], "stage_ms": head["stage_ms"],
            "roofline": head["roofline"], "clocks": head["clocks"], "sustained": head.get("sustained"),
            "numa": numa,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if len(results) > 1:
            line["configs"] = [{k: v for k, v in r.items() if k not in ("unit",)} for r in results[1:]]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
