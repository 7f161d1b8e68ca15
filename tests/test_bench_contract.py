"""bench.py's JSON contract, checked on CPU through the reference arm (the GPU arm needs a B200)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"}


def test_reference_arm_prints_one_contract_line(built):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--bytes-per-gpu", str(8 << 20)], capture_output=True, text=True, timeout=300, check=True)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert KEYS <= set(j)
    assert j["impl"] == "reference" and j["higher_is_better"] is True and j["vs_baseline"] is None
    assert j["unit"] == "Msamples/s" and j["value"] > 1.0
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in j["config"] and "model" not in j["config"]
    # the reference arm decodes the workload's own stream (same `config` object as the GPU arm prints), cut over
    # every CPU the process may use, and says how many threads / physical cores that was
    assert j["config"]["bytes_per_gpu"] == 8 << 20 and j["config"]["msgtype"] == "scm" and j["config"]["chip_length"] == 72
    assert j["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and j["cpu_baseline"]["physical_cores"] >= 1
    assert j["cpu_baseline"]["one_core_value"] > 1.0


def test_both_arms_print_the_same_config_object(built):
    import bench
    a = bench.workload_config("scm1g", bench.WORKLOADS["scm1g"], 1 << 30, 8, 4096, 13824)
    assert a["halo_blocks"] == 5 and a["blocks_per_gpu"] == 131072 and a["total_bytes"] == 8 << 30
    assert "configs[1]" in a["workload"]
    m = bench.workload_config("multi8g", bench.WORKLOADS["multi8g"], 8 << 30, 1, 8192, 105984)
    assert m["halo_blocks"] == 0 and m["blocks_per_gpu"] == 524288 and "configs[2]" in m["workload"]


def test_cpu_arm_scales_with_threads(built):
    """The C thread driver behind the CPU arm: T decoders over T shards of one stream run in parallel (no GIL,
    nothing allocated in the timed region) and see the same packets as one decoder."""
    import oracle
    from rtlamr_b200 import synth
    n = 1 << 23
    pk, truth = synth.make_packets("scm", 72, n, seed=1, spacing=1 << 19)
    iq = synth.host_fill(0, n, 3, pk, nthreads=4)
    assert (iq == synth.host_fill(0, n, 3, pk)).all()
    t1, c1, m1, nb = oracle.bench_threads("scm", 72, iq, 1)
    ncpu = min(4, oracle.host_cpus())
    tn, cn, mn, _ = oracle.bench_threads("scm", 72, iq, ncpu)
    assert nb == n // 4096 and m1 >= len(truth) - 2 and abs(mn - m1) <= 2 * ncpu   # a shard seam can cut a packet
    if ncpu >= 4:
        # best of three runs each: one run is a window of tens of ms, in which a shared host can take a time slice
        t1 = min([t1] + [oracle.bench_threads("scm", 72, iq, 1)[0] for _ in range(2)])
        tn = min([tn] + [oracle.bench_threads("scm", 72, iq, ncpu)[0] for _ in range(2)])
        assert tn < t1 / 2.0, (t1, tn)


def test_non_zero_ranks_of_the_reference_arm_do_no_work(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=60, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "--steps" in out.stderr and out.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_reproducible(built, tmp_path):
    """Two runs with the same arguments dump the same files, and the records are exactly what one ertgpu_decode of
    the workload's seeded stream returns."""
    import numpy as np

    import bench
    from rtlamr_b200 import capi, synth
    nbytes, steps = 64 << 20, 3
    lines = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                              "--bytes-per-gpu", str(nbytes), "--no-extras", "--skip-cpu-baseline", "--sustained-seconds", "0",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, check=True)
        lines.append(json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0]))
    assert lines[0]["steps"] == steps
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "scm1g_bytes.npy" in names
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    dump = {f[len("scm1g_"):-len(".npy")]: np.load(tmp_path / "a" / f) for f in names}
    for f in names:
        assert np.load(tmp_path / "b" / f).tobytes() == dump[f[len("scm1g_"):-len(".npy")]].tobytes(), f
    assert all(v.dtype in (np.float32, np.float64) for v in dump.values())

    # the same stream generated on the host, decoded from device memory in one call like a timed step
    import torch
    w = bench.WORKLOADS["scm1g"]
    probe = capi.new_decoder(w["msgtype"], bench.CHIP_LENGTH)
    nblocks = nbytes // probe.cfg.block_size2
    probe.close()
    h = capi.new_decoder(w["msgtype"], bench.CHIP_LENGTH, max_blocks_per_call=nblocks, max_candidates=1 << 20)
    nsamples = nblocks * h.cfg.block_size
    pk, _ = synth.make_packets(w["msgtype"], bench.CHIP_LENGTH, nsamples, seed=1, spacing=bench.PACKET_SPACING)
    d_iq = torch.from_numpy(synth.host_fill(0, nsamples, w["seed"], pk)).cuda()
    torch.cuda.synchronize()
    h.decode_device_async(d_iq.data_ptr(), d_iq.numel(), capi.DECODE_ONLY_VALID)
    want, counts = h.fetch(1 << 16), h.last_counts()
    h.close()
    assert len(want) > 0 and np.array_equal(dump["row"], np.arange(len(want)))      # small enough: no sampling
    assert np.array_equal(dump["counts"], np.array(counts, dtype=np.float64))
    for f in ("block", "idx", "preamble_id", "check_mask", "flags"):
        assert np.array_equal(dump[f], want[f].astype(np.float64)), f
    assert np.array_equal(dump["bytes"], want["bytes"][:, :h.cfg.packet_bytes].astype(np.float32))
