#!/usr/bin/env python
"""bench.py — IQ MSamples/s through the BLE receive hot path (demod + detect + decode).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config all|c2|c3|c5|hot]
                    [--dump-outputs DIR]

One "step" = one pass of the receive path over one batch of synthetic IQ.  The headline line is always
BASELINE.json configs[1] ("c2"); the other configurations ride along in the same JSON line under "configs":

  c2   (headline) single ch37 stream, 1 GiB of 4 Msps int8 IQ (2^29 IQ samples) per GPU, one ADV_IND burst per
       4096-sample slot (131072 bursts; 1 % corrupted, 1 % placed across a chunk boundary).  N>1: weak scaling,
       every rank owns one such capture; hit records of all ranks land on rank 0.
  c3   BASELINE configs[2], N=1 only: all 40 BLE channels, 256 MiB each, per-channel access address / CRC init.
  c5   BASELINE configs[4]: 4096 streams x 16 MiB (stream k on channel k mod 40), generated on rank 0, SCATTERED
       to the ranks (time reported on its own), sharded with shard_range; strong scaling, packets/s at 1/2/4/8.
  hot  N=1 only: 1 GiB of full-scale random IQ (50/50 discriminator bits) — the prefilter / resolver stress row.

Every configuration ends with an UNTIMED parity block: 64 seeded (stream, 16-chunk) slices are re-run through the
oracle (oracle/, the CPU restatement pinned to the reference) and compared byte for byte with the records as they
were gathered on rank 0 ("parity": "ok").

`value`   whole-job IQ MSamples/s with the IQ already resident in HBM (CUDA events, max over ranks).
`e2e`     the same metric through the public C-ABI call btle_b200_rx_batch() with HOST buffers: page-locked host ->
          device copy of the step's IQ and device -> host copy of the records inside the timed region; ranks are bound
          to their GPU's NUMA node first (btle_b200_bind_host_numa).
`roofline` HBM roofline of the persistent kernel: algorithmic bytes (2 B per IQ sample + 64 B per packet,
          SURVEY.md §8d) / CUDA-event time per launch vs MEASURED_PEAKS.json.
`cpu_baseline` the reference's own receiver() (oracle/_ref, compiled from /root/reference) timed on this box's host
          cores on a bounded sample of the same stream.
`--impl reference` times that CPU implementation alone (rank 0 only) on the c2 config.
`--dump-outputs DIR` writes, after the timed steps, the c2 records of the last timed step as a caller of the receive path
          receives them (rank 0's gathered buffer, reference order) to DIR/<field>.npy, one float64 / float32 array per record
          field: the inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the tree may be read-only; the benchmark writes nothing into it

STREAM_INT8 = 1 << 30
SLOT_SAMPLES = 4096
SEED = 0x37E15163
CPU_SAMPLE_INT8 = 64 << 20
REF_STEP_SECONDS = 2.0            # --impl reference: one step = enough passes over the 64 MiB sample to last about this long
METRIC = "IQ MSamples/s demod+detect+decode (BLE rx chain, ch37 ADV stream)"
DTYPE = "int32 (int8 IQ in, bit-exact integer path)"
C2_WORKLOAD = ("1 GPU: single ch37 stream, 1 GiB synthetic 4 Msps int8 IQ with injected ADV_IND bursts (BASELINE.json configs[1]; "
               "1 % of the bursts corrupted, 1 % placed across a chunk boundary)")
PARITY_SLICES = 64
PARITY_CHUNKS = 16
DUMP_MAX_RECORDS = 200_000           # --dump-outputs: 248 B per record (float64 fields and index, float32 bytes), at most 50 MB


def host_cores():
    """Host threads this process may use: CPU affinity, capped by a cgroup CPU quota if there is one
    (more processes than the quota allows would only make the CPU arm slower)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:                                                   # cgroup v2
        q, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = int(q) / int(period)
    except Exception:
        try:                                               # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / period
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def committed_traffic():
    """dram bytes per launch from the committed ncu capture (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "span_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.power = []
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_min_mhz": (s[0] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s), "power_w_max": (round(max(self.power), 1) if self.power else None)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------
# the CPU arm: the reference's own receiver() on the host cores
def ref_driver():
    p = os.path.join(ROOT, "oracle", "_ref", "btle_ref_driver")
    return p if os.path.exists(p) else None


def cpu_time_sample(sample_path, target_wall_s, fixed_reps=None):
    """Times the reference receiver() (or, if oracle/_ref is absent, our C port) over the sample.  One worker process
    per host core (receiver() is not re-entrant); the workers are forked and warmed up before the clock starts."""
    cores = host_cores()
    drv = ref_driver()
    if drv:
        def run(reps):
            p = subprocess.run([drv, "time", sample_path, "37", "8e89bed6", "555555", "ffffffff", "0", str(cores), str(reps)],
                               check=True, capture_output=True)
            return json.loads(p.stdout.decode().strip().splitlines()[-1])
        reps = fixed_reps or 1
        r = run(reps)
        while not fixed_reps and target_wall_s > 0 and r["seconds"] < 0.6 * target_wall_s and reps < 65536:
            reps = max(reps + 1, min(65536, int(reps * target_wall_s / max(r["seconds"], 1e-4)) + 1))
            r = run(reps)
        return {"msamples_per_s": r["msamples_per_s"], "packets_per_s": r["packets_per_s"], "kind": "reference",
                "cores": r.get("procs", cores), "seconds": r["seconds"], "reps": r["reps"],
                "per_core": r.get("msamples_per_s_per_core")}
    # port: single-threaded C restatement
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import orc
    iq = np.fromfile(sample_path, dtype=np.int8)
    t0 = time.perf_counter()
    rec = orc.rx_stream(iq)
    dt = time.perf_counter() - t0
    ms = (iq.size // 16384) * 8192 / dt / 1e6
    return {"msamples_per_s": ms, "packets_per_s": len(rec) / dt, "kind": "port", "cores": 1, "seconds": dt, "reps": 1, "per_core": ms}


def make_sample_file(n_int8):
    """The first n_int8 bytes of rank 0's c2 stream, regenerated with the torch generator alone (the CUDA library
    is NOT loaded for it: the reference arm's process must not touch our kernels)."""
    import torch
    from btle_b200 import synth
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    iq, _ = synth.make_adv_stream(n_int8, seed=SEED, channel=37, slot_samples=SLOT_SAMPLES, corrupt_every=100, straddle_every=100,
                                  device=dev, use_cuda_modulator=False)
    f = tempfile.NamedTemporaryFile(prefix="btle_sample_", suffix=".bin", delete=False, dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    f.write(iq.cpu().numpy().tobytes())
    f.close()
    return f.name


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    path = make_sample_file(CPU_SAMPLE_INT8)
    try:
        # passes per step: calibrated once so that a step lasts ~REF_STEP_SECONDS on this machine's core count
        cal = cpu_time_sample(path, REF_STEP_SECONDS)
        reps, kind, cores = cal["reps"], cal["kind"], cal["cores"]
        per_step, pk = [], []
        for i in range(args.warmup + args.steps):
            r = cpu_time_sample(path, 0.0, fixed_reps=reps) if kind == "reference" else cal
            if i >= args.warmup:
                per_step.append(r["seconds"])
                pk.append(r["packets_per_s"])
        samples = (CPU_SAMPLE_INT8 // 16384) * 8192 * reps
        total = sum(per_step)
        value = samples * len(per_step) / total / 1e6
        sample_txt = (f"{reps} passes over the first 64 MiB of the 1 GiB ch37 stream per step (~{total / len(per_step):.1f} s), {cores} worker "
                      "process(es) = all host cores (reference receiver() is not re-entrant); workers forked and warmed up before the clock starts")
        line = {
            "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "MSamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / len(per_step), 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "packets_per_s": round(sum(pk) / len(pk), 1),
            "config": {"workload": C2_WORKLOAD + f"; the CPU arm runs {reps} passes over a bounded 64 MiB sample of it per step (same burst density)",
                       "stream_int8": STREAM_INT8, "sample_int8": CPU_SAMPLE_INT8, "passes_per_step": reps},
            "cpu_baseline": {"value": round(value, 3), "unit": "MSamples/s", "cores": cores, "kind": kind, "sample": sample_txt,
                             "msamples_per_s_per_core": round(value / max(cores, 1), 3)},
            "e2e": {"value": round(value, 3), "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
    finally:
        os.unlink(path)


# ------------------------------------------------------------------------------------------------
class Env:
    """torch / distributed context of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        from btle_b200 import _native
        self.numa_node = _native.bind_host_numa(self.local_rank)       # before any page-locked allocation
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.main = torch.cuda.current_stream(self.dev)
        self.second = torch.cuda.Stream(device=self.dev)

    def sync_all(self):
        self.main.wait_stream(self.second)
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return int(x)
        t = self.torch.tensor([x], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t)
        return int(t.item())


def parity_block(env, rx, gather, buf, d_iq, cfgs_local, stream_lo, n_streams_global, all_cfgs, n_int8, units, seed):
    """Untimed: PARITY_SLICES seeded (stream, chunk-range) slices through the oracle vs the records gathered on rank 0."""
    import numpy as np
    from btle_b200.dist import owner_of
    torch, dist = env.torch, env.dist
    nchunks = n_int8 // 16384
    L = min(PARITY_CHUNKS, nchunks)
    rng = np.random.default_rng(seed)
    slices = []
    for i in range(PARITY_SLICES):
        g = int(rng.integers(0, n_streams_global))
        k0 = int(rng.integers(0, nchunks - L + 1))
        if i == 0:
            k0 = 0
        if i == 1:
            k0 = nchunks - L                       # the end of a capture: look-ahead runs into the zero padding
        slices.append((g, k0))
    mine = []
    for i, (g, k0) in enumerate(slices):
        if owner_of(g, n_streams_global, env.world) == env.rank:
            a, b = 16384 * k0, min(n_int8, 16384 * (k0 + L) + 3088)
            mine.append((i, d_iq[g - stream_lo, a:b].cpu().numpy().tobytes()))
    if env.world > 1:
        gathered = [None] * env.world if env.rank == 0 else None
        dist.gather_object(mine, gathered, dst=0)
    else:
        gathered = [mine]
    if env.rank != 0:
        return None
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orc                                     # the checker (oracle/): untimed, never on the measured path
    from btle_b200.dist import shard_range
    offsets = [shard_range(n_streams_global, env.world, r)[0] for r in range(env.world)]
    recs = gather.ordered(buf, offsets, n_units=units)
    key = recs["stream"].astype(np.int64) * nchunks + recs["chunk"]
    assert (np.diff(key) >= 0).all(), "gathered records are not in (stream, chunk) order"
    blobs = {i: blob for part in gathered for i, blob in part}
    compared, bad = 0, []
    for i, (g, k0) in enumerate(slices):
        c = all_cfgs[g]
        sl = np.frombuffer(blobs[i], dtype=np.int8)
        exp = orc.rx_stream(sl, channel=int(c["channel"]), access_addr=int(c["access_addr"]), access_mask=int(c["access_mask"]),
                            crc_init=int(c["crc_init"]), raw=int(c["raw"]), stream=g)
        exp = exp[exp["chunk"] < L].copy()
        exp["chunk"] += k0
        if not int(c["rssi"]):
            exp["mag_sum"] = 0
        lo, hi = np.searchsorted(key, [g * nchunks + k0, g * nchunks + k0 + L])
        got = recs[lo:hi]
        compared += len(exp)
        if len(got) != len(exp) or got.tobytes() != exp.tobytes():
            bad.append({"stream": g, "chunk0": k0, "gpu": int(len(got)), "oracle": int(len(exp))})
    out = {"parity": "ok" if not bad else "FAIL", "slices": len(slices), "chunks_per_slice": L, "records_compared": compared,
           "checked_on": "records as gathered on rank 0" if env.world > 1 else "records of the device buffer"}
    if bad:
        out["mismatches"] = bad[:8]
        sys.stderr.write(f"PARITY FAILURE: {bad[:8]}\n")
    return out, recs


def run_workload(env, rx, name, d_iq, cfgs_local, stream_lo, n_streams_global, all_cfgs, n_int8, steps, warmup, bursts_local,
                 serial_launches=0, parity_seed=1, keep_last=False):
    """Times `steps` passes over this rank's captures (double-buffered over two CUDA streams), records of all ranks
    on rank 0 (RecordGather), then the parity block.  Returns a dict (rank 0) / partial dict (other ranks); with
    `keep_last`, rank 0's dict holds the records of the last timed step under "last_records"."""
    import numpy as np
    from btle_b200.dist import RecordGather
    torch = env.torch
    dev = env.dev
    ns_local = d_iq.shape[0]
    units = rx.units(ns_local, n_int8) if ns_local else 0
    cap = int(bursts_local * 1.25) + 1024
    if env.world > 1:                              # identical region sizes on every rank
        t = torch.tensor([cap, units], dtype=torch.int64, device=dev)
        env.dist.all_reduce(t, op=env.dist.ReduceOp.MAX)
        cap, units_max = int(t[0].item()), int(t[1].item())
    else:
        units_max = units
    gather = RecordGather(cap, max(units_max, 1), n_buffers=2, device=dev)
    pipe = [env.main, env.second]
    n_samples_local = ns_local * (n_int8 // 16384) * 8192

    def step(i):
        b = i & 1
        with torch.cuda.stream(pipe[b]):
            d_out, d_dir = gather.target(b)
            rx.rx_device_dir(d_iq, cfgs_local, d_out, None, d_dir, pipe[b].cuda_stream)     # packet count = sum of the directory
            gather.complete(b)

    for i in range(warmup):
        step(i)
    env.sync_all()
    launches_per_step = rx.last_launches
    sampler = ClockSampler(physical_gpu_index(env.local_rank))
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.sync_all()
    torch.cuda.profiler.start()                    # lets `ncu --profile-from-start off` see only the timed region
    ev0.record(env.main)
    env.second.wait_event(ev0)
    for i in range(steps):
        step(i)
    env.main.wait_stream(env.second)
    ev1.record(env.main)
    env.sync_all()
    torch.cuda.profiler.stop()
    sampler.stop_flag = True
    sampler.join()
    ms_step = env.max_over_ranks(ev0.elapsed_time(ev1)) / steps
    last = (steps - 1) & 1
    last_records = None
    if keep_last and env.rank == 0:                # before the serial launches below reuse the buffers
        from btle_b200.dist import shard_range
        last_records = gather.ordered(last, [shard_range(n_streams_global, env.world, r)[0] for r in range(env.world)],
                                      n_units=units_max)
    n_found_local = int(gather.target(last)[1][:max(units, 1), 1].sum().item()) if units else 0
    n_found = env.sum_over_ranks(n_found_local)
    n_samples = env.sum_over_ranks(n_samples_local)

    serial = None
    if serial_launches:
        # every launch bracketed by its own pair of events on ONE stream (no overlap between successive launches,
        # no host sync in between): the mean is what the roofline uses
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(serial_launches)]
        torch.cuda.synchronize(dev)
        for i, (a, b) in enumerate(evs):
            d_out, d_dir = gather.target(i & 1)
            a.record(env.main)
            rx.rx_device_dir(d_iq, cfgs_local, d_out, None, d_dir, env.main.cuda_stream)
            b.record(env.main)
        torch.cuda.synchronize(dev)
        per = sorted(a.elapsed_time(b) for a, b in evs)
        serial = {"launches": serial_launches, "mean": round(sum(per) / len(per), 4), "median": round(per[len(per) // 2], 4),
                  "min": round(per[0], 4), "max": round(per[-1], 4),
                  "wall_per_launch": round(evs[0][0].elapsed_time(evs[-1][1]) / serial_launches, 4)}
        last = (serial_launches - 1) & 1
        env.sync_all()

    par = parity_block(env, rx, gather, last, d_iq, cfgs_local, stream_lo, n_streams_global, all_cfgs, n_int8, units_max, parity_seed)
    res = {"name": name, "ms_per_step": ms_step, "n_found": n_found, "n_found_local": n_found_local, "n_samples": n_samples,
           "n_samples_local": n_samples_local, "units": units, "cap": cap, "gather_mode": gather.mode, "serial": serial,
           "launches_per_step": launches_per_step, "clocks": sampler.result(), "last_records": last_records}
    if env.rank == 0:
        parity, recs = par
        res["parity"] = parity
        res["crc_ok"] = int((recs["crc_bad"] == 0).sum())
        res["records_on_rank0"] = int(len(recs))
        if env.world > 1:
            res["records_on_rank0_per_rank"] = gather.counts(last, units_max)
    del gather
    return res


def dump_records(out_dir, recs):
    """The records as float arrays, one file per field (record i is row i of every file); more than DUMP_MAX_RECORDS
    records are thinned to a fixed, seeded, sorted sample: index.npy holds each row's position in the full output,
    total.npy the number of records."""
    import numpy as np
    total = len(recs)
    idx = np.arange(total)
    if total > DUMP_MAX_RECORDS:
        idx = np.sort(np.random.default_rng(0).choice(len(recs), DUMP_MAX_RECORDS, replace=False))
    recs = recs[idx]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"index": idx.astype(np.float64), "total": np.array([total], dtype=np.float64)}
    for f in recs.dtype.names:
        arrays[f] = recs[f].astype(np.float32 if f == "bytes" else np.float64)
    for f, a in arrays.items():
        np.save(os.path.join(out_dir, f + ".npy"), a)


def roofline_of(res, peak, peak_src, launch_ms=None):
    algo = 2.0 * res["n_samples_local"] + 64.0 * res["n_found_local"]
    ms = launch_ms if launch_ms else res["ms_per_step"]
    ach = algo / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
            "algorithmic_bytes_per_launch": algo, "launch_ms": round(ms, 4), "peak_source": peak_src,
            "kernel": "btle_rx_persistent_kernel"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="all", choices=["all", "c2", "c3", "c5", "hot", "sps8"],
                    help="which configurations to run besides the c2 headline (default: every one that applies at this N)")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="kernel experiments only: the JSON line is then not a valid bench line")
    ap.add_argument("--c5-streams", type=int, default=4096, help="(experiments) number of c5 streams; BASELINE.json says 4096")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the c2 records of the last timed step to DIR/<field>.npy (float64 / float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    env = Env()
    torch, dist = env.torch, env.dist
    from btle_b200 import BtleRx, make_cfgs, synth
    from btle_b200.dist import scatter_streams, shard_range
    dev, world, rank = env.dev, env.world, env.rank
    rx = BtleRx(env.local_rank)
    peak, peak_src = measured_peak()
    want = (lambda c: args.config in ("all", c))
    extra = {}

    # ================= c2: the headline =====================================================================
    iq, truth = synth.make_adv_stream(STREAM_INT8, seed=SEED + 7919 * rank, channel=37, slot_samples=SLOT_SAMPLES,
                                      corrupt_every=100, straddle_every=100, device=dev)
    d_iq = iq.view(1, -1)
    n_bursts = len(truth["start_sample"])
    cfg1 = make_cfgs(1, channel=37)
    all_cfgs = make_cfgs(world, channel=37)
    c2 = run_workload(env, rx, "c2", d_iq, cfg1, rank, world, all_cfgs, STREAM_INT8, args.steps, args.warmup, n_bursts,
                      serial_launches=max(args.steps, 50), parity_seed=2, keep_last=bool(args.dump_outputs))
    if rank == 0 and args.dump_outputs:
        dump_records(args.dump_outputs, c2.pop("last_records"))
    n_samples_rank = (STREAM_INT8 // 16384) * 8192
    value = c2["n_samples"] / (c2["ms_per_step"] * 1e-3) / 1e6
    expect_ok = int((~truth["corrupt"]).sum())

    # ---- e2e: host buffers through the public C-ABI call -----------------------------------------------------
    e2e = None
    e2e_steps = 0 if args.skip_e2e else (args.e2e_steps or max(3, min(args.steps, 8)))
    if e2e_steps:
        cap = n_bursts + n_bursts // 4
        h_iq = torch.empty(STREAM_INT8, dtype=torch.int8, pin_memory=True)     # first touched on this rank's NUMA node
        h_iq.copy_(iq)
        torch.cuda.synchronize(dev)
        # what the link can do: plain page-locked -> device copies of the same buffer
        d_tmp = torch.empty(STREAM_INT8, dtype=torch.int8, device=dev)
        d_tmp.copy_(h_iq, non_blocking=True)
        torch.cuda.synchronize(dev)
        env.sync_all()
        t0 = time.perf_counter()
        for _ in range(3):
            d_tmp.copy_(h_iq, non_blocking=True)
        torch.cuda.synchronize(dev)
        h2d_gbs = 3 * STREAM_INT8 / (time.perf_counter() - t0) / 1e9
        del d_tmp
        h_np = h_iq.numpy().reshape(1, -1)
        for _ in range(2):
            r = rx.rx_batch(h_np, cfg1, cap=cap)
        env.sync_all()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r = rx.rx_batch(h_np, cfg1, cap=cap)
        torch.cuda.synchronize(dev)
        dt_local = time.perf_counter() - t0
        dt = env.max_over_ranks(dt_local)
        per_rank = [dt_local]
        if world > 1:
            lst = [None] * world
            dist.all_gather_object(lst, (dt_local, h2d_gbs, env.numa_node))
            per_rank = lst
        e2e_val = world * n_samples_rank * e2e_steps / dt / 1e6
        e2e = {"value": round(e2e_val, 3), "unit": "MSamples/s", "h2d_bytes_per_step": STREAM_INT8 + 24,
               "d2h_bytes_per_step": int(len(r)) * 64 + 8 * rx.units(1, STREAM_INT8) + 4, "steps": e2e_steps, "packets": int(len(r)),
               "api": "btle_b200_rx_batch (C-ABI, page-locked host IQ in, host records out, records in reference order)",
               "numa_node_rank0": env.numa_node, "h2d_peak_gbs_rank0": round(h2d_gbs, 2),
               "pcie_frac_rank0": round((STREAM_INT8 * e2e_steps / dt_local / 1e9) / h2d_gbs, 4)}
        if world > 1:
            e2e["per_rank"] = [{"h2d_gbs": round(STREAM_INT8 * e2e_steps / p[0] / 1e9, 2), "h2d_peak_gbs": round(p[1], 2), "numa_node": p[2]}
                               for p in per_rank]
        # the same call with an ordinary (pageable) buffer: staged through page-locked segments inside the library
        if world == 1:
            h_page = np.empty((1, STREAM_INT8), dtype=np.int8)
            h_page[:] = h_np
            rx.rx_batch(h_page, cfg1, cap=cap)
            t0 = time.perf_counter()
            for _ in range(3):
                rp = rx.rx_batch(h_page, cfg1, cap=cap)
            dtp = time.perf_counter() - t0
            e2e["pageable_host_buffer"] = {"value": round(n_samples_rank * 3 / dtp / 1e6, 3), "unit": "MSamples/s",
                                           "note": "same call, numpy (pageable) IQ: 32 MiB segments through 2 page-locked staging buffers",
                                           "same_records": bool(rp.tobytes() == r.tobytes())}
            del h_page
        del h_np, h_iq

    # ---- CPU baseline (rank 0, N=1 only) -------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        path = make_sample_file(CPU_SAMPLE_INT8)
        try:
            c = cpu_time_sample(path, 4.0)
            cpu = {"value": round(c["msamples_per_s"], 3), "unit": "MSamples/s", "cores": c["cores"], "kind": c["kind"],
                   "packets_per_s": round(c["packets_per_s"], 1), "msamples_per_s_per_core": round(c["per_core"] or 0, 3),
                   "sample": f"first 64 MiB of the same 1 GiB ch37 stream x{c['reps']} passes, {c['cores']} host "
                             f"process(es) forked and warmed up before the clock starts, {c['seconds']:.2f} s wall"}
        finally:
            os.unlink(path)
    del d_iq, iq
    torch.cuda.empty_cache()

    def sub_line(res, workload, scaling, extra_cfg=None):
        v = res["n_samples"] / (res["ms_per_step"] * 1e-3) / 1e6
        o = {"workload": workload, "value": round(v, 1), "unit": "MSamples/s", "ms_per_step": round(res["ms_per_step"], 4),
             "packets_per_s": round(res["n_found"] / (res["ms_per_step"] * 1e-3), 1), "packets_found": res["n_found"],
             "scaling": scaling, "n_gpus": world, "roofline": roofline_of(res, peak, peak_src), "record_gather": res["gather_mode"],
             "clocks": res["clocks"]}
        if rank == 0:
            o["parity"] = res["parity"]
            o["crc_ok"] = res["crc_ok"]
            if "records_on_rank0_per_rank" in res:
                o["records_on_rank0_per_rank"] = res["records_on_rank0_per_rank"]
        if extra_cfg:
            o.update(extra_cfg)
        return o

    sub_steps = max(3, min(args.steps // 10, 20))
    # ================= c3: 40 channels x 256 MiB (N=1) ===========================================================
    if world == 1 and want("c3"):
        cfgs = synth.channel_plan(40)
        n = 256 << 20
        d, tr = synth.synth_streams_device(cfgs, n, seed=1000, device=dev, slot_samples=SLOT_SAMPLES, corrupt_every=100, straddle_every=100)
        res = run_workload(env, rx, "c3", d, cfgs, 0, 40, cfgs, n, sub_steps, 3, len(tr), parity_seed=3)
        extra["c3"] = sub_line(res, "1 GPU: all 40 BLE channels concurrent, 256 MiB IQ each, per-channel access-addr/crcinit (BASELINE.json configs[2])",
                               "n/a (single GPU)", {"bursts": int(len(tr)), "crc_ok_expected_about": int((tr["corrupt"] == 0).sum()), "steps": sub_steps})
        del d, tr, res
        torch.cuda.empty_cache()

    # ================= c5: 4096 streams x 16 MiB, sharded over the ranks ========================================
    if want("c5"):
        NS, n = args.c5_streams, 16 << 20
        cfgs_all = synth.channel_plan(NS)
        lo, hi = shard_range(NS, world, rank)
        n_slots = (n // 2) // SLOT_SAMPLES
        full = None
        gen_s = 0.0
        if rank == 0:
            t0 = time.perf_counter()
            full, _ = synth.synth_streams_device(cfgs_all, n, seed=5000, device=dev, slot_samples=SLOT_SAMPLES, corrupt_every=100,
                                                 straddle_every=100, want_truth=False)
            torch.cuda.synchronize(dev)
            gen_s = time.perf_counter() - t0
        scatter_ms = 0.0
        if world > 1:
            d = torch.empty((hi - lo, n), dtype=torch.int8, device=dev)       # n is a multiple of 16: rows stay 16-byte aligned
            # untimed warm-up of the send/recv channels (NCCL connects peers lazily on first use: ~0.5 s)
            scatter_streams(full[:world] if full is not None else None, world, 4096, src=0, device=dev)
            env.sync_all()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(env.main)
            scatter_streams(full, NS, n, src=0, device=dev, out=d)
            s1.record(env.main)
            env.sync_all()
            scatter_ms = env.max_over_ranks(s0.elapsed_time(s1))
        else:
            d = full
        del full
        torch.cuda.empty_cache()
        res = run_workload(env, rx, "c5", d, cfgs_all[lo:hi], lo, NS, cfgs_all, n, sub_steps, 3, (hi - lo) * n_slots, parity_seed=5)
        moved = (NS - (shard_range(NS, world, 0)[1])) * n
        extra["c5"] = sub_line(res, f"{NS} concurrent 4 Msps IQ streams x 16 MiB (stream k on channel k mod 40), generated on rank 0, "
                                    f"scattered over NVLink and sharded over {world} GPU(s) (BASELINE.json configs[4])", "strong",
                               {"streams": NS, "streams_per_gpu": hi - lo, "bursts": NS * n_slots, "steps": sub_steps,
                                "iq_scatter_ms": round(scatter_ms, 3), "iq_scatter_bytes": int(moved),
                                "iq_scatter_gbs": round(moved / (scatter_ms * 1e-3) / 1e9, 1) if scatter_ms else None,
                                "iq_scatter_note": "one NCCL send/recv per rank out of rank 0's capture tensor; NOT part of ms_per_step",
                                "generation_s_rank0": round(gen_s, 3)})
        del d, res
        torch.cuda.empty_cache()

    # ================= hot: full-scale noise (N=1) =================================================================
    if world == 1 and want("hot"):
        cfgs = make_cfgs(1, channel=37)
        d, _ = synth.synth_streams_device(cfgs, STREAM_INT8, seed=77, device=dev, amplitude=0, noise=1, want_truth=False)
        hot_steps = max(sub_steps, 1500)               # ~0.3 s: long enough for the clock / power sampler to see the steady state
        res = run_workload(env, rx, "hot", d, cfgs, 0, 1, cfgs, STREAM_INT8, hot_steps, 3, 4096, serial_launches=50, parity_seed=7)
        o = sub_line(res, "1 GPU: 1 GiB of full-scale uniform random IQ on ch37 (50/50 discriminator bits): prefilter / resolver stress, no decodable bursts",
                     "n/a (single GPU)", {"steps": hot_steps,
                                          "note": "same instruction count and isolated-launch duration as c2 under ncu; the prefilter lets 3 % of the groups "
                                                  "through, whose exact re-check is spread over all resolver lanes; in a long run random data costs board power "
                                                  "(see clocks) — profiles/r02_hot_vs_c2.md"})
        o["roofline_isolated_launch"] = roofline_of(res, peak, peak_src, res["serial"]["mean"])
        o["single_stream_launch_ms"] = res["serial"]
        extra["hot_noise"] = o
        del d, res
        torch.cuda.empty_cache()

    # ================= sps8: the 8-samples-per-symbol streaming mode (N=1) ============================================
    if world == 1 and want("sps8"):
        import ctypes
        n_samp = 1 << 28                                               # 1 GiB of int16 I,Q = 33.5 s of air at 8 Msps
        gen = torch.Generator(device=dev)
        gen.manual_seed(4)
        cap16 = (torch.randn((n_samp, 2), generator=gen, device=dev, dtype=torch.float16) * 3.0).to(torch.int16)
        # 4096 clean ADV packets (the 39-byte PDU of test_btle_ber.py with counting payloads) through the 8-sps modulator
        npk = 4096
        rngp = np.random.default_rng(8)
        pdus = [bytes([0x42, 0x25]) + int(k).to_bytes(4, "little") + rngp.integers(0, 256, 33, dtype=np.uint8).tobytes() for k in range(npk)]
        air = np.stack([np.frombuffer(synth.air_bytes(p, 37), dtype=np.uint8) for p in pdus])
        bits = torch.from_numpy(np.unpackbits(air, axis=1, bitorder="little").astype(np.int8)).to(dev)
        ti, tq = synth.modulate_batch_8sps(bits)
        gap = n_samp // npk
        pos = torch.arange(npk, device=dev, dtype=torch.int64) * gap + 5000 + torch.from_numpy(rngp.integers(0, 20000, npk)).to(dev)
        idx = pos.unsqueeze(1) + torch.arange(ti.shape[1], device=dev).unsqueeze(0)
        cap16[idx.reshape(-1), 0] += ti.reshape(-1).to(torch.int16)
        cap16[idx.reshape(-1), 1] += tq.reshape(-1).to(torch.int16)
        d_hits = torch.zeros(1 << 20, dtype=torch.int64, device=dev)
        d_cnt = torch.zeros(1, dtype=torch.int32, device=dev)
        L = rx._L
        stp = ctypes.c_void_p(env.main.cuda_stream)

        def hits():
            rx._check(L.btle_b200_sps8_hits_device(rx._h, cap16.data_ptr(), n_samp, 0x8E89BED6, d_hits.data_ptr(), d_hits.numel(), d_cnt.data_ptr(), stp))
        for _ in range(3):
            hits()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(env.main)
        for _ in range(sub_steps):
            hits()
        e1.record(env.main)
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / sub_steps
        n_hits = int(d_cnt.item())
        # the whole mode through the C-ABI with a host buffer (copy + hits + windows + model receiver + records)
        h16 = torch.empty((n_samp, 2), dtype=torch.int16, pin_memory=True)
        h16.copy_(cap16)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        recs = rx.rx_sps8(h16.numpy(), 37)
        dt = time.perf_counter() - t0
        ok = int((recs["rx"]["crc_ok"] != 0).sum())
        sent = {p[2:6] for p in pdus}
        got = {bytes(r["rx"]["pdu"][2:6]) for r in recs if r["rx"]["crc_ok"]}
        ach = 4.0 * n_samp / (ms * 1e-3) / 1e9
        extra["sps8"] = {"workload": "1 GPU: 8-Msps int16 capture (btle_ll -q format), 2^28 samples (1 GiB), 4096 ADV packets on a noise floor; the Python / "
                                     "Verilog model's 8-phase CRC-select receiver, streaming (btle_b200_rx_sps8)",
                         "value": round(n_samp / (ms * 1e-3) / 1e6, 1), "unit": "MSamples/s (8 Msps samples through sps8_hits_kernel, device-resident)",
                         "ms_per_step": round(ms, 4), "steps": sub_steps, "hits": n_hits,
                         "roofline": {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                                      "algorithmic_bytes_per_launch": 4.0 * n_samp, "kernel": "sps8_hits_kernel", "peak_source": peak_src},
                         "e2e": {"value": round(n_samp / dt / 1e6, 1), "unit": "MSamples/s", "api": "btle_b200_rx_sps8 (page-locked host int16 in, records out)",
                                 "h2d_bytes": 4 * n_samp, "packets": int(len(recs)), "crc_ok": ok},
                         "parity": {"parity": "ok" if (got == sent and ok == npk) else "FAIL", "check": "every inserted packet decoded once with CRC ok and its own bytes; "
                                    "exact comparison with the CPU restatement at test size: tests/test_btlelib_compat_gpu.py"}}
        del cap16, h16, d_hits
        torch.cuda.empty_cache()

    # ---- the line ------------------------------------------------------------------------------------------------
    if rank == 0:
        serial = c2["serial"]
        roof = roofline_of(c2, peak, peak_src, serial["mean"])
        roof["traffic"] = committed_traffic()
        roof["pipelined_step_ms"] = round(c2["ms_per_step"], 4)
        roof["pipelined_frac"] = round(roof["algorithmic_bytes_per_launch"] / (c2["ms_per_step"] * 1e-3) / 1e9 / peak, 4)
        roof["peak_note"] = ("`peak` is the driver's COPY bandwidth (reads and writes share the bus); this kernel only reads, and a read-only "
                             "stream on B200 reaches 6.85-7.03 TB/s (tools/probe_hbm_data.py, the c3 row), so `frac` is the isolated launch "
                             "against the copy figure and back-to-back / long rows can pass 1.0; nominal HBM3e peak 8 TB/s")
        roof["frac_of_nominal_8tbs"] = round(roof["achieved"] / 8000.0, 4)
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": "MSamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(c2["ms_per_step"], 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "packets_per_s": round(c2["n_found"] / (c2["ms_per_step"] * 1e-3), 1),
            "config": {"workload": C2_WORKLOAD + ("; one such capture per rank, hit records of all ranks stored into rank 0's buffer by the kernels" if world > 1 else ""),
                       "stream_int8_per_gpu": STREAM_INT8, "bursts_per_gpu": n_bursts, "bursts_across_chunk_boundary_rank0": int(truth["straddle"].sum()),
                       "packets_found": c2["n_found"], "packets_found_rank0": c2["n_found_local"], "crc_ok_all_ranks": c2.get("crc_ok"),
                       "crc_ok_expected_rank0": expect_ok,
                       "packets_note": "found > bursts: a burst whose access address starts in the last 4 samples of a chunk is counted by the "
                                       "reference in both chunks (zeroed search history, btle_rx.c:1518); the oracle and the kernel agree on each",
                       "l2_policy": "input (1 GiB) larger than L2 (126 MB); no flush needed",
                       "step_pipelining": "steps alternate over 2 CUDA streams / 2 output buffers (double-buffered captures)",
                       "single_stream_ms_per_step": serial["mean"], "single_stream_launch_ms": serial,
                       "parallelism": f"dp{world} (independent captures)", "record_gather": c2["gather_mode"],
                       "records_on_rank0_per_rank": c2.get("records_on_rank0_per_rank"), "units_per_launch": c2["units"],
                       "record_order": "emitted in reference order by the kernel (one block per unit + unit directory); no sort / ordering kernels"},
            "parity": c2["parity"], "clocks": c2["clocks"], "e2e": e2e, "gpu_launches": int(c2["launches_per_step"] or 0) * args.steps,
            "roofline": roof, "cpu_baseline": cpu, "configs": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
