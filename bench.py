#!/usr/bin/env python3
"""bench.py -- M3TSZ datapoints/sec (encode + decode) on N B200s of one node.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W`
prints ONE JSON line on rank 0.  One "step" = one pass of the hot path over one
batch: batch ENCODE of S series x P points (lane-per-series sm_100a kernel; every
series into its own segment, like the reference's encoders own their buffers) and batch
DECODE of those segments addressed by (offset, size) -- no compaction pass in between.
Packing into ONE buffer for a fileset is the persist step; its cost (encode with packed
output) is reported next to it as `encode_packed` / `step_packed`.  The batch is 1M series x 1440 points per GPU -- the shape
BASELINE.json's north-star target is quoted on (configs[2-4]; configs[4] = 8M series
over 8 GPUs = this at N=8); with N GPUs every rank holds its own 1M-series shard
(weak scaling, no data-path collective: series are independent).  `--series 100000`
runs configs[1].

  value   = S*P*N / step time, inputs and outputs resident in HBM (CUDA events)
  e2e     = the SAME batch through the C ABI's *_host entry points from pinned HOST
            buffers, chunk by chunk (H2D of the inputs and D2H of the results inside
            the timed region; the encode and the decode leg run from two host threads so
            both PCIe directions stay busy)
  roofline= the decode kernel: algorithmic bytes (compressed bytes + index entries in,
            16 B/dp out) / its average duration inside the timed region
            (roofline_encode = the same accounting for the encode kernel of the step)
  cpu_baseline = the CPU oracle (plain-C restatement of the reference's Go codec; no Go
            toolchain in this image) on the host cores this process may use, bounded sample

`--impl reference` times that CPU oracle as the reference arm on the full batch.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "M3TSZ datapoints/sec encode+decode"
UNIT = "datapoints/s"
SEC = 1_000_000_000
L2_BYTES = 126 * 1024 * 1024


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series", type=int, default=1_000_000, help="series per GPU")
    ap.add_argument("--e2e-series", type=int, default=0,
                    help="series pushed through the host-buffer API per e2e step (0 = the whole batch, "
                         "reduced only if pinned host memory is short)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="e2e steps (0 = min(steps, 20))")
    ap.add_argument("--points", type=int, default=1440)
    ap.add_argument("--int-optimized", type=int, default=1)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline budget (GPU arm)")
    ap.add_argument("--ref-seconds", type=float, default=1200.0,
                    help="reference arm: shrink the per-step sample only if the full batch would exceed this")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="headline step only (no downsample / merge / tiles / fixtures / all-gather side measurements)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) to DIR/<name>.npy; see dump_outputs()")
    return ap.parse_args()


# --------------------------------------------------------------------------- host facts
def usable_cores():
    """Host threads this process can really use: the CPU affinity mask capped by the cgroup
    CPU quota (os.cpu_count() reports the machine, not the lease)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    cores = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return cores, {"os_cpu_count": os.cpu_count(), "sched_affinity": aff,
                   "cgroup_cpu_quota": quota, "used": cores}


def available_host_bytes():
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v != "max":
                lim = int(v)
                use = 0
                try:
                    use = int(open(path.replace("memory.max", "memory.current")
                                   .replace("memory.limit_in_bytes", "memory.usage_in_bytes")).read())
                except Exception:
                    pass
                avail = min(avail, lim - use) if avail is not None else lim - use
            break
        except Exception:
            continue
    return avail if avail is not None else 64 << 30


def bind_to_gpu_numa_node(local_rank):
    """Pins this rank's threads (and so its first-touch pinned allocations) to the NUMA node
    its GPU hangs off; several ranks staging through one socket is what bent the N=8 e2e curve."""
    bdf = None
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        bdf = None
    if bdf is None:
        try:
            bdf = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id",
                                  "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        except Exception:
            return None
    try:
        bdf = bdf.lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None
    return None


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(workload):
    """dram bytes per decode launch from the committed ncu --set full capture of this workload
    (profiles/traffic.json names the capture file); a citation, not a per-run measurement."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(workload)
    except Exception:
        return None


def make_config(S, P, int_opt, bytes_per_dp=7.3):
    """Identical for the GPU arm and the reference arm (parameters only; the measured compressed
    size is reported next to it as `compressed_bytes_per_dp`)."""
    bytes_per_dp = 7.3
    return {"workload": "batch of %d series x %d points per GPU (the north-star target shape "
                        "1M x 1440 = configs[2-4] size; configs[4] = 8M over 8 GPUs), Gaussian "
                        "random walk (x0=100, N(0,1) steps), 60 s cadence, unit=Second; step = "
                        "encode (per-series segments) + decode, datapoints resident point-major "
                        "([point][series])" % (S, P),
            "series_per_gpu": S, "points": P, "int_optimized": bool(int_opt),
            "l2": "inputs %.2f GB and outputs %.2f GB per step >> 126 MB L2, no flush needed"
                  % (S * P * 16 / 1e9, S * P * (16 + bytes_per_dp) / 1e9),
            "parallelism": "series sharded per GPU, no data-path collective"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                  "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU oracle arm
class CpuOracleRunner:
    """Encode + decode of Gaussian-walk chunks with the CPU oracle on `cores` threads (one thread
    per disjoint series range, like the reference's one-goroutine-per-series fan-out).  Work
    buffers belong to the runner and are reused; inputs are generated before the timed region."""

    def __init__(self, n_points, int_opt, cores):
        import numpy as np
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        self.np, self.O = np, O
        self.P, self.int_opt, self.cores = n_points, int_opt, cores
        self.bufs = None

    def make_chunks(self, n_series, chunk, seed):
        from m3_b200 import synth
        chunks = []
        for c0 in range(0, n_series, chunk):
            n = min(chunk, n_series - c0)
            ts, vals, start = synth.gaussian_walk(n, self.P, "cpu", seed=seed + c0)
            chunks.append((ts.numpy(), vals.numpy(), int(start[0])))
        return chunks

    def _ensure(self, S):
        np = self.np
        if self.bufs is None or self.bufs["S"] < S:
            stride = 64 + 20 * self.P
            self.bufs = {"S": S,
                         "enc": (np.zeros((S, stride), dtype=np.uint8), np.zeros(S, dtype=np.uint64),
                                 np.zeros(S, dtype=np.int32)),
                         "dec": (np.zeros((S, self.P), dtype=np.int64), np.zeros((S, self.P), dtype=np.float64),
                                 np.zeros(S, dtype=np.uint32), np.zeros(S, dtype=np.int32)),
                         "blob": np.zeros(S * (8 * self.P + 64), dtype=np.uint8)}
        return self.bufs

    def run_chunk(self, ts_np, vals_np, st):
        np, O = self.np, self.O
        S = ts_np.shape[0]
        b = self._ensure(S)
        enc = tuple(x[:S] for x in b["enc"])
        dec = tuple(x[:S] for x in b["dec"])
        t0 = time.perf_counter()
        out, ln, status = O.encode_batch(ts_np, vals_np, st, 1, self.int_opt, n_threads=self.cores, bufs=enc)
        t1 = time.perf_counter()
        # hand the streams to the decoder as one CSR buffer (not timed: the reference's iterators
        # read the encoders' own buffers)
        off = np.zeros(S + 1, dtype=np.uint64)
        off[1:] = np.cumsum(ln)
        total = int(off[-1])
        blob = b["blob"][:total]
        pos = 0
        for i in range(S):
            n = int(ln[i])
            blob[pos:pos + n] = out[i, :n]
            pos += n
        t2 = time.perf_counter()
        O.decode_batch(blob, off, self.P, self.int_opt, n_threads=self.cores, bufs=dec)
        t3 = time.perf_counter()
        return (t1 - t0), (t3 - t2), total

    def run_step(self, chunks):
        te = td = 0.0
        nbytes = 0
        for ts_np, vals_np, st in chunks:
            a, b, n = self.run_chunk(ts_np, vals_np, st)
            te += a
            td += b
            nbytes += n
        return te, td, nbytes


def cpu_oracle_throughput(n_series, n_points, int_opt, budget_s, steps=1, warmup=0, full=False):
    """Times the CPU oracle on the host cores this process may use.  full=False: a bounded sample
    sized to `budget_s`; full=True: the whole n_series batch per step, shrunk only if
    (steps + warmup) steps would exceed budget_s.  Returns (dp/s, info)."""
    cores, core_info = usable_cores()
    runner = CpuOracleRunner(n_points, int_opt, cores)
    probe_s = max(cores * 8, 128)
    probe = runner.make_chunks(probe_s, probe_s, seed=99)
    runner.run_step(probe)  # warm the library / page in
    te, td, _ = runner.run_step(probe)
    per_series = (te + td) / probe_s
    total_steps = max(1, steps + warmup)
    fit = int(budget_s / total_steps / max(per_series, 1e-9))
    if full:
        S = n_series if fit >= n_series else max(probe_s, fit)
        # host memory: inputs 16 B/dp for the whole batch + one chunk of work buffers
        mem = available_host_bytes()
        max_by_mem = int(0.5 * mem / (n_points * 16))
        if S > max_by_mem:
            S = max(probe_s, max_by_mem)
    else:
        S = int(max(probe_s, min(n_series, fit)))
    S = max(cores, (S // cores) * cores) if S < n_series else S
    chunk = min(S, 100_000)
    chunks = runner.make_chunks(S, chunk, seed=100)
    for _ in range(warmup):
        runner.run_step(chunks)
    tot_e = tot_d = 0.0
    nbytes = 0
    for _ in range(steps):
        te, td, nbytes = runner.run_step(chunks)
        tot_e += te
        tot_d += td
    dp = S * n_points * steps
    info = {
        "cores": cores, "core_info": core_info, "series_per_step": S, "full_batch": S == n_series,
        "compressed_bytes_per_dp": nbytes / float(S * n_points),
        "sample": "%d series x %d points per step%s (Gaussian walk, intOptimized=%s), encode then decode, "
                  "%d threads (sched_getaffinity %s, cgroup quota %s, os.cpu_count %s)"
                  % (S, n_points, " = the whole batch" if S == n_series else " (bounded sample)", bool(int_opt),
                     cores, core_info["sched_affinity"], core_info["cgroup_cpu_quota"], core_info["os_cpu_count"]),
        "encode_dps": dp / tot_e, "decode_dps": dp / tot_d, "ms_per_step": (tot_e + tot_d) * 1e3 / steps,
        "kind": "port",
        "note": "C restatement of the reference algorithm (Go toolchain unavailable); published Go "
                "anchor: BenchmarkM3TSZDecode 69272 ns/op ~ 10.4 M dp/s per core",
    }
    return dp / (tot_e + tot_d), info


def fixture_set_throughput(codec, dev, time_fn, n_streams=200_000):
    """Secondary realistic set (SURVEY.md 8d): the reference's ten int-optimised production
    fixtures (m3tsz/encoder_benchmark_test.go:36-47; millisecond unit, time-unit markers, int
    mode, repeats), tiled to n_streams streams with 64-byte aligned starts and decoded in one
    launch.  The zero padding after each stream's end-of-stream marker is never parsed."""
    import base64
    import torch
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "m3tsz_goldens.json")))
    raw = [base64.b64decode(x) for x in g["fixtures_b64"]["streams"]]
    pts = g["fixtures_b64"]["expected_points"]
    padded = [r + b"\0" * ((-len(r)) % 64) for r in raw]
    reps = max(1, n_streams // len(raw))
    lens = torch.tensor([len(x) for x in padded] * reps, dtype=torch.int64)
    off = torch.zeros(len(lens) + 1, dtype=torch.int64)
    off[1:] = lens.cumsum(0)
    d_blob = torch.frombuffer(bytearray(b"".join(padded) * reps), dtype=torch.uint8).to(dev)
    d_off = off.to(dev)
    dec = codec.decode(d_blob, d_off, max(pts) + 8)
    n = dec.n_points.cpu()
    assert bool((dec.status.cpu() == 0).all()) and n[: len(pts)].tolist() == pts, "fixture decode mismatch"
    total_dp = int(n.sum())
    ms = time_fn(lambda: codec.decode(d_blob, d_off, max(pts) + 8, out=dec), n=3)
    return {"streams": int(len(lens)), "datapoints": total_dp,
            "compressed_bytes_per_dp": sum(len(x) for x in raw) / float(sum(pts)),
            "decode_ms": ms, "decode_dps": total_dp / (ms * 1e-3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, info = cpu_oracle_throughput(args.series, args.points, args.int_optimized, budget_s=args.ref_seconds,
                                        steps=args.steps, warmup=args.warmup, full=True)
    cfg = make_config(args.series, args.points, args.int_optimized)
    if not info["full_batch"]:
        cfg["reference_sample"] = "bounded: %d of %d series per step" % (info["series_per_step"], args.series)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": info["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64/f64 (integer bit manipulation; float64 values)", "data": "synthetic", "config": cfg,
        "compressed_bytes_per_dp": info["compressed_bytes_per_dp"],
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                         "sample": info["sample"], "encode_dps": info["encode_dps"],
                         "decode_dps": info["decode_dps"], "note": info["note"], "core_info": info["core_info"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- GPU arm
def run_e2e(args, codec, ts, vals, start, P, int_opt, rank, world, dev, barrier, dist):
    """The whole batch through m3tsz_encode_batch_host / m3tsz_decode_batch_host from pinned host
    memory, chunk by chunk.  Inputs: one pinned buffer per chunk (distinct data, H2D every step);
    outputs: reusable pinned staging per leg (D2H every step, overwritten by the next chunk).  The
    two legs run from two host threads (two contexts): encode of chunk c+1 overlaps decode of
    chunk c, so the H2D-heavy and the D2H-heavy leg share the full-duplex link."""
    import torch
    from m3_b200.codec import BatchCodec
    S = ts.shape[0]
    chunk = min(S, 100_000)
    want = args.e2e_series or S
    per_series_pinned = P * 16
    budget = 0.4 * available_host_bytes() / max(1, world) - 3 * chunk * P * 16
    Se = int(max(chunk, min(want, S, budget // per_series_pinned)))
    if world > 1:  # every rank runs the same batch (the aggregate below counts Se per rank)
        se_t = torch.tensor([Se], dtype=torch.int64, device=dev)
        dist.all_reduce(se_t, op=dist.ReduceOp.MIN)
        Se = int(se_t.item())
    Se = (Se // chunk) * chunk if Se >= chunk else Se
    n_chunks = (Se + chunk - 1) // chunk
    bounds = [(c * chunk, min(Se, (c + 1) * chunk)) for c in range(n_chunks)]
    h_in = []
    for c0, c1 in bounds:  # distinct pinned inputs per chunk
        h_in.append((ts[c0:c1].cpu().pin_memory(), vals[c0:c1].cpu().pin_memory(), start[c0:c1].cpu().pin_memory()))
    e_cap = chunk * (P * 9 + 128)
    # two sets of encode outputs (the decode leg reads set c%2 while the encode leg fills the other)
    enc_out = [dict(packed=torch.empty(e_cap, dtype=torch.uint8).pin_memory(),
                    off=torch.empty(chunk + 1, dtype=torch.int64).pin_memory(),
                    ln=torch.empty(chunk, dtype=torch.int64).pin_memory(),
                    st=torch.empty(chunk, dtype=torch.int32).pin_memory()) for _ in range(2)]
    h_dts = torch.empty((chunk, P), dtype=torch.int64).pin_memory()
    h_dvals = torch.empty((chunk, P), dtype=torch.float64).pin_memory()
    h_n = torch.empty(chunk, dtype=torch.int32).pin_memory()
    h_dst = torch.empty(chunk, dtype=torch.int32).pin_memory()
    dec_codec = BatchCodec(dev.index, int_optimized=int_opt)  # second context: its own streams + scratch
    state = {"bytes": 0, "err": None}

    def host_step(check=False):
        filled = [threading.Semaphore(0) for _ in range(n_chunks)]
        freed = [threading.Semaphore(0) for _ in range(n_chunks)]
        nbytes = [0] * n_chunks

        def enc_leg():
            try:
                for c, (c0, c1) in enumerate(bounds):
                    if c >= 2:
                        freed[c - 2].acquire()
                    o = enc_out[c % 2]
                    n = c1 - c0
                    codec.encode_host(h_in[c][0], h_in[c][1], h_in[c][2], 1, o["packed"], o["off"][: n + 1],
                                      o["ln"][:n], o["st"][:n], align=64)
                    nbytes[c] = int(o["off"][n])
                    filled[c].release()
            except Exception as e:  # pragma: no cover
                state["err"] = e
                for f in filled:
                    f.release()

        th = threading.Thread(target=enc_leg)
        th.start()
        for c, (c0, c1) in enumerate(bounds):
            filled[c].acquire()
            if state["err"] is not None:
                break
            o = enc_out[c % 2]
            n = c1 - c0
            dec_codec.decode_host(o["packed"][: nbytes[c]], o["off"][: n + 1], P, h_dts[:n], h_dvals[:n], h_n[:n],
                                  h_dst[:n])
            if check:
                assert torch.equal(h_dts[:n], h_in[c][0]) and int((h_dst[:n] != 0).sum()) == 0
            freed[c].release()
        th.join()
        if state["err"] is not None:
            raise state["err"]
        state["bytes"] = sum(nbytes)

    host_step(check=True)
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        host_step()
    barrier()
    l0 = codec.launch_count() + dec_codec.launch_count()
    e_steps = args.e2e_steps or max(1, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        host_step()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    e_launch = codec.launch_count() + dec_codec.launch_count() - l0
    tt = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e_s = float(tt[0]) / e_steps
    nb = state["bytes"]
    h2d = Se * P * 16 + Se * 8 + nb + (Se + n_chunks) * 8
    d2h = nb + (Se + n_chunks) * 8 + Se * 12 + Se * P * 16 + Se * 8
    return {"value": Se * P * world / e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": e_s * 1e3, "steps": e_steps, "launches_per_step": e_launch / e_steps,
            "series_per_step": Se, "chunks_per_step": n_chunks, "whole_batch": Se == S,
            "pcie_gbs_each_way": max(h2d, d2h) / e_s / 1e9,
            "api": "m3tsz_encode_batch_host + m3tsz_decode_batch_host over %d-series chunks (pinned host "
                   "inputs, reusable pinned result staging; encode leg and decode leg on two host threads / "
                   "two contexts)" % chunk}


def run_fetch_e2e(args, codec, ts, vals, start, P, rank, world, dev, barrier, dist):
    """Fetch path with host buffers (RF=3): compressed replica streams up, merged series down."""
    import numpy as np
    import torch
    Sf = min(ts.shape[0], 100_000)
    enc = codec.encode(ts[:Sf], vals[:Sf], start[:Sf], unit=1)
    cpacked, coff = codec.compact(enc, align=64)
    torch.cuda.synchronize()
    off = coff.cpu().numpy()
    ln = enc.out_len.cpu().numpy()
    blob = cpacked[: int(off[-1])].cpu().numpy()
    del enc, cpacked, coff
    # host CSR of 3 replicas per series: the same stream three times (replicas agree on a healthy cluster)
    al = (ln + 63) // 64 * 64
    seq_off = np.zeros(3 * Sf + 1, dtype=np.int64)
    seq_off[1:] = np.cumsum(np.repeat(al, 3))
    total = int(seq_off[-1])
    h_streams = torch.zeros(total + 64, dtype=torch.uint8).pin_memory()
    hs = h_streams.numpy()
    for s in range(Sf):
        seg = blob[off[s]: off[s] + ln[s]]
        for r in range(3):
            o = int(seq_off[3 * s + r])
            hs[o: o + ln[s]] = seg
    h_off = torch.from_numpy(seq_off).pin_memory()
    ar = torch.arange(3 * Sf + 1, dtype=torch.int64)
    h_slice, h_rep, h_ser = ar.clone(), ar.clone(), torch.arange(0, 3 * Sf + 1, 3, dtype=torch.int64)
    h_ts = torch.empty((Sf, P), dtype=torch.int64).pin_memory()
    h_val = torch.empty((Sf, P), dtype=torch.float64).pin_memory()
    h_n = torch.empty(Sf, dtype=torch.int32).pin_memory()
    h_st = torch.empty(Sf, dtype=torch.int32).pin_memory()

    def step():
        codec.fetch_host(h_streams[:total], h_off, h_slice, h_rep, h_ser, P, P, h_ts, h_val, h_n, h_st)

    step()
    assert int((h_st != 0).sum()) == 0 and bool((h_n == P).all())
    assert torch.equal(h_ts, ts[:Sf].cpu())
    barrier()
    n_steps = 5
    t0 = time.perf_counter()
    for _ in range(n_steps):
        step()
    t1 = time.perf_counter()
    tt = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    s = float(tt[0]) / n_steps
    return {"replicas": 3, "series": Sf, "input_dps": 3 * Sf * P * world / s, "output_dps": Sf * P * world / s,
            "ms_per_step": s * 1e3, "h2d_bytes_per_step": total + (3 * Sf + 1) * 8,
            "d2h_bytes_per_step": Sf * P * 16 + Sf * 8,
            "api": "m3tsz_fetch_batch_host (H2D compressed replicas -> decode -> series merge -> D2H merged)"}


DUMP_SEED = 20240601
DUMP_MAX_SCALAR_SERIES = 1 << 20
DUMP_MAX_ROW_SERIES = 256


def dump_outputs(out_dir, enc, dec_pm, start):
    """Writes the results of the timed step (encode into per-series segments, then point-major
    decode of them) as float32 / float64 .npy files under out_dir, so that two builds can be
    compared output for output on the same seeded batch.  Under 64 MB in all:

      series_index         [K]     the series whose full rows are written: a fixed seeded sample
      encode_segments      [K, B]  their compressed segments, one byte per element, zero past out_len
      decode_ts_offset_ns  [P, K]  their decoded timestamps minus the series start (exact in float64)
      decode_values        [P, K]  their decoded values
      encode_out_len, encode_status, decode_n_points, decode_status, decode_unit
                           [M]     per series, for the first M = min(S, 2^20) series
    """
    import numpy as np
    import torch
    P, S = dec_pm.values.shape
    B = enc.out.shape[1]
    K = min(S, DUMP_MAX_ROW_SERIES, max(1, (32 << 20) // (P * 16 + B * 4)))
    M = min(S, DUMP_MAX_SCALAR_SERIES)
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(S, size=K, replace=False))
    idx = torch.from_numpy(rows).to(enc.out.device)
    seg = enc.out[idx]
    seg = seg * (torch.arange(B, device=seg.device)[None, :] < enc.out_len[idx][:, None])
    arrays = {
        "series_index": rows.astype(np.float64),
        "encode_segments": seg.to(torch.float32),
        "decode_ts_offset_ns": (dec_pm.ts[:, idx] - start[idx][None, :]).to(torch.float64),
        "decode_values": dec_pm.values[:, idx],
        "encode_out_len": enc.out_len[:M].to(torch.float64),
        "encode_status": enc.status[:M].to(torch.float32),
        "decode_n_points": dec_pm.n_points[:M].to(torch.float64),
        "decode_status": dec_pm.status[:M].to(torch.float32),
        "decode_unit": dec_pm.unit[:M].to(torch.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    assert total <= 64 << 20, total


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the codec has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from m3_b200 import synth
    from m3_b200.codec import BatchCodec, DecodeResult, PackedResult

    S, P = args.series, args.points
    int_opt = bool(args.int_optimized)
    codec = BatchCodec(local_rank, int_optimized=int_opt)
    ts, vals, start = synth.gaussian_walk(S, P, dev, seed=1000 + rank)
    # per-series segments sized for the data: 9 B per datapoint (Gaussian walk: ~7.3); a series that
    # needs more reports M3TSZ_ERR_CAPACITY and would be re-encoded with m3tsz_encode_bound (20 B/dp)
    stride = ((64 + 9 * P) + 63) // 64 * 64
    from m3_b200.codec import EncodeResult
    enc = EncodeResult(out=torch.empty((S, stride), dtype=torch.uint8, device=dev),
                       out_len=torch.empty(S, dtype=torch.int64, device=dev),
                       status=torch.empty(S, dtype=torch.int32, device=dev))
    seg_off = torch.arange(S, dtype=torch.int64, device=dev) * stride
    seg_flat = enc.out.view(-1)
    # The device-resident batch is kept POINT-major ([point][series], step-major): what the query
    # engine's step iterators consume, and every encode / decode step of a warp then touches 32
    # consecutive elements.  Series-major in and out (the layout of the *_host entry points and of
    # round 1) is timed next to it below.
    ts_pm, vals_pm = ts.t().contiguous(), vals.t().contiguous()
    dec_pm = DecodeResult(ts=torch.empty((P, S), dtype=torch.int64, device=dev),
                          values=torch.empty((P, S), dtype=torch.float64, device=dev),
                          n_points=torch.empty(S, dtype=torch.int32, device=dev),
                          status=torch.empty(S, dtype=torch.int32, device=dev),
                          unit=torch.empty(S, dtype=torch.uint8, device=dev), annotations=None)
    dec = DecodeResult(ts=dec_pm.ts.view(S, P), values=dec_pm.values.view(S, P), n_points=dec_pm.n_points,
                       status=dec_pm.status, unit=dec_pm.unit, annotations=None)  # same memory, series-major view
    dec_events = []

    def encode():
        codec.encode(ts_pm, vals_pm, start, unit=1, out=enc, point_major=True)

    def decode():
        codec.decode(seg_flat, seg_off, P, out=dec_pm, lengths=enc.out_len, point_major=True)

    def step(record=False):
        encode()
        if record:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            decode()
            e1.record()
            dec_events.append((e0, e1))
        else:
            decode()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for _ in range(args.warmup):
        step()
    barrier()
    # sanity: the timed path round-trips (float mode exactly; int mode up to the reference's own
    # near-integer rounding -- the parity tests compare those series with the oracle bit for bit)
    assert int((enc.status != 0).sum()) == 0 and int((dec_pm.status != 0).sum()) == 0
    assert torch.equal(dec_pm.ts, ts_pm)
    mism = int((dec_pm.values.view(torch.int64) != vals_pm.view(torch.int64)).sum())
    assert mism <= S * P * 1e-6, mism
    compressed_bytes = int(enc.out_len.sum().item())

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = codec.launch_count()
    barrier()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step(record=True)
    ev1.record()
    barrier()
    launches = codec.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    ms_total = ev0.elapsed_time(ev1)
    dec_ms = sum(a.elapsed_time(b) for a, b in dec_events) / len(dec_events)
    t = torch.tensor([ms_total, dec_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, dec_ms_max = float(t[0]), float(t[1])
    ms_per_step = ms_total / args.steps
    value = S * P * world / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:  # before the timings below reuse enc and dec_pm
        dump_outputs(args.dump_outputs, enc, dec_pm, start)

    # separate per-kernel timings (same buffers, outside the headline region)
    def time_fn(fn, n=5):
        fn()
        torch.cuda.synchronize()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    enc_ms = time_fn(encode)
    # series-major inputs and outputs (round 1's layout)
    enc_sm_ms = time_fn(lambda: codec.encode(ts, vals, start, unit=1, out=enc))
    assert int(enc.out_len.sum().item()) == compressed_bytes
    dec_sm_ms = time_fn(lambda: codec.decode(seg_flat, seg_off, P, out=dec, lengths=enc.out_len))
    assert torch.equal(dec.ts, ts)
    # the persist variant: encode straight into one packed buffer (fileset data-file layout)
    del enc, seg_flat, seg_off
    torch.cuda.empty_cache()
    cap_bytes = compressed_bytes + 64 * S + 4096
    pk = PackedResult(packed=torch.empty(cap_bytes, dtype=torch.uint8, device=dev),
                      offsets=torch.empty(S, dtype=torch.int64, device=dev),
                      out_len=torch.empty(S, dtype=torch.int64, device=dev),
                      status=torch.empty(S, dtype=torch.int32, device=dev),
                      total=torch.zeros(1, dtype=torch.int64, device=dev))
    encp = lambda: codec.encode_packed(ts, vals, start, unit=1, align=64, out=pk)
    encp()
    assert int((pk.status != 0).sum()) == 0 and int(pk.out_len.sum().item()) == compressed_bytes
    encp_ms = time_fn(encp)
    encp_pm = lambda: codec.encode_packed(ts_pm, vals_pm, start, unit=1, align=64, out=pk, point_major=True)
    encp_pm()
    assert int((pk.status != 0).sum()) == 0 and int(pk.out_len.sum().item()) == compressed_bytes
    encp_pm_ms = time_fn(encp_pm)
    del ts_pm, vals_pm
    torch.cuda.empty_cache()
    decp_ms = time_fn(lambda: codec.decode(pk.packed, pk.offsets, P, out=dec, lengths=pk.out_len))
    extras = not args.no_extras
    side = {}
    if extras:
        s0 = int(start[0].item())
        n_win = (P * 60 + 299) // 300
        side["fixture_set"] = fixture_set_throughput(codec, dev, time_fn)
        # segment checksums (row N2): Adler-32 of every stream of the packed batch
        ck, ck_st = codec.segment_checksums(pk.packed, pk.offsets, lengths=pk.out_len)
        assert int((ck_st != 0).sum()) == 0
        ck_ms = time_fn(lambda: codec.segment_checksums(pk.packed, pk.offsets, lengths=pk.out_len))
        side["segment_checksum"] = {"streams": S, "bytes": compressed_bytes, "ms": ck_ms,
                                    "algorithmic_gbs": compressed_bytes / (ck_ms * 1e-3) / 1e9}
        del ck, ck_st
        # fused decode + 5-min Gauge downsample (config 4) on the full batch needs CSR offsets:
        # re-pack the batch once in series order (not timed)
        full_slots = None
        if S <= 1_000_000:
            torch.cuda.empty_cache()
            full_slots = codec.encode(ts, vals, start, unit=1)
            fpacked, foff = codec.compact(full_slots, align=64)
            del full_slots
            ds = codec.decode_downsample(fpacked, foff, s0, 300 * SEC, n_win)
            assert int((ds.status != 0).sum()) == 0 and bool((ds.count == 5).all())
            ds_ms = time_fn(lambda: codec.decode_downsample(fpacked, foff, s0, 300 * SEC, n_win, out=ds))
            side["decode_downsample"] = {
                "windows": n_win, "ms": ds_ms, "series": S,
                "algorithmic_gbs": (compressed_bytes + n_win * S * 32) / (ds_ms * 1e-3) / 1e9,
                "frac_of_hbm": (compressed_bytes + n_win * S * 32) / (ds_ms * 1e-3) / 1e9 / measured_peak_gbs()[0],
                "read_gbs": compressed_bytes / (ds_ms * 1e-3) / 1e9, "dps": S * P / (ds_ms * 1e-3)}
            del ds
            dsl = codec.decode_downsample(fpacked, foff, s0, 300 * SEC, n_win, want_last=True)
            dsl_ms = time_fn(lambda: codec.decode_downsample(fpacked, foff, s0, 300 * SEC, n_win, out=dsl,
                                                             want_last=True))
            side["decode_downsample_last"] = {"ms": dsl_ms, "algorithmic_gbs":
                                              (compressed_bytes + n_win * S * 48) / (dsl_ms * 1e-3) / 1e9}
            del dsl
            # tile aggregation (row N3): decode -> Gauge per 5 min -> re-encode, packed
            tiles, n_tiles = codec.aggregate_tiles(fpacked, foff, s0, 300 * SEC, n_win)
            assert int((tiles.status != 0).sum()) == 0 and bool((n_tiles == n_win).all())
            tile_ms = time_fn(lambda: codec.aggregate_tiles(fpacked, foff, s0, 300 * SEC, n_win, out=tiles), n=3)
            tile_bytes = int(tiles.total.item())
            side["aggregate_tiles"] = {"ms": tile_ms, "source_dps": S * P / (tile_ms * 1e-3), "step_s": 300,
                                       "agg": "last", "out_bytes": tile_bytes,
                                       "algorithmic_gbs": (compressed_bytes + tile_bytes) / (tile_ms * 1e-3) / 1e9}
            del tiles, n_tiles, fpacked, foff
            torch.cuda.empty_cache()
        # series merge (row N1): RF=3 fetch shape -- every 3 consecutive decoded streams are the
        # replicas of one series (same timestamps => 3 inputs collapse to 1 output per timestamp)
        Sm = (min(S, 300_000) // 3) * 3
        m_slice = torch.arange(Sm + 1, dtype=torch.int64, device=dev)
        m_rep = torch.arange(Sm + 1, dtype=torch.int64, device=dev)
        m_ser = torch.arange(0, Sm + 1, 3, dtype=torch.int64, device=dev)
        mg = lambda: codec.merge_series(dec.ts[:Sm], dec.values[:Sm], dec.n_points[:Sm], dec.status[:Sm], m_slice,
                                        m_rep, m_ser, P)
        m_out = mg()
        assert int((m_out[3] != 0).sum()) == 0 and bool((m_out[2] == P).all())
        del m_out
        merge_ms = time_fn(mg, n=3)
        side["series_merge"] = {"replicas": 3, "series": Sm // 3, "ms": merge_ms,
                                "input_dps": Sm * P / (merge_ms * 1e-3),
                                "algorithmic_gbs": (Sm * P * 16 + (Sm // 3) * P * 16) / (merge_ms * 1e-3) / 1e9}
        # the same merge over point-major arrays (what decode writes in the timed step)
        pm_ts, pm_v = dec.ts[:Sm].t().contiguous(), dec.values[:Sm].t().contiguous()
        mgp = lambda: codec.merge_series(pm_ts, pm_v, dec.n_points[:Sm], dec.status[:Sm], m_slice, m_rep, m_ser, P,
                                         point_major=True)
        m_out = mgp()
        assert int((m_out[3] != 0).sum()) == 0 and bool((m_out[2] == P).all())
        del m_out
        mergep_ms = time_fn(mgp, n=3)
        side["series_merge"].update({"point_major_ms": mergep_ms, "point_major_input_dps": Sm * P / (mergep_ms * 1e-3),
                                     "point_major_algorithmic_gbs": (Sm * P * 16 + (Sm // 3) * P * 16) /
                                     (mergep_ms * 1e-3) / 1e9})
        del pm_ts, pm_v
        # Prometheus epilogue (row N4) over the decoded batch: ns -> ms, plain and counter-normalised
        Sp = min(S, 300_000)
        pr = lambda: codec.prom_convert(dec.ts[:Sp], dec.values[:Sp], dec.n_points[:Sp])
        pr()
        prom_ms = time_fn(pr, n=3)
        hr = torch.ones(Sp, dtype=torch.uint8, device=dev)
        prr = lambda: codec.prom_convert(dec.ts[:Sp], dec.values[:Sp], dec.n_points[:Sp], 300 * SEC, hr)
        prr()
        prom_r_ms = time_fn(prr, n=3)
        side["prom_convert"] = {"series": Sp, "ms": prom_ms, "dps": Sp * P / (prom_ms * 1e-3),
                                "algorithmic_gbs": Sp * P * 32 / (prom_ms * 1e-3) / 1e9,
                                "counter_normalised_ms": prom_r_ms}
        del hr
        torch.cuda.empty_cache()

    # ---- fetch-side all-gather (only when a query spans shards) ----
    allgather = None
    if world > 1 and extras:
        from m3_b200.sharded import fetch_allgather_decoded
        try:
            allgather = fetch_allgather_decoded(codec, pk, P, dist, dev, barrier)
        except Exception as e:  # a side measurement must not take the headline down with it
            allgather = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- e2e: the same batch through the *_host C ABI with pinned host buffers ----
    e2e = fetch = None
    if not args.no_e2e:
        if extras:
            fetch = run_fetch_e2e(args, codec, ts, vals, start, P, rank, world, dev, barrier, dist)
        del dec
        torch.cuda.empty_cache()
        e2e = run_e2e(args, codec, ts, vals, start, P, int_opt, rank, world, dev, barrier, dist)
        if numa:
            e2e["numa_binding"] = numa

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the decode kernel ----
    peak, peak_src = measured_peak_gbs()
    alg_bytes = compressed_bytes + S * 16 + S * P * 16 + S * 9  # in: streams + (offset, size); out: ts, val, n/status/unit
    achieved = alg_bytes / (dec_ms_max * 1e-3) / 1e9
    workload = "%dx%d" % (S, P)
    traffic = recorded_traffic(workload)
    roofline = {"bound": "hbm", "kernel": "m3tsz::decode_kernel<%s,3> (point-major outputs)" % ("true" if int_opt else "false"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": "profiles/traffic.json (ncu --set full capture, committed)",
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": dec_ms_max,
                "bytes_per_dp": alg_bytes / (S * P)}

    # the other (larger) half of the step, same accounting: 16 B/dp + start in; streams + (length, status) out
    enc_alg_bytes = S * P * 16 + S * 8 + compressed_bytes + S * 12
    enc_achieved = enc_alg_bytes / (enc_ms * 1e-3) / 1e9
    roofline_encode = {"bound": "hbm",
                       "kernel": "m3tsz::encode_kernel<%s,false,1> (point-major inputs staged by TMA tensor copies, "
                                 "per-series segments)" % ("true" if int_opt else "false"),
                       "achieved": enc_achieved, "peak": peak, "unit": "GB/s", "frac": enc_achieved / peak,
                       "algorithmic_bytes_per_launch": enc_alg_bytes, "kernel_ms": enc_ms,
                       "note": "issue-bound, not HBM-bound (profiles/r02c_encode_pm_tma_400kx1440.ncu_summary.txt)"}

    cpu = None
    if not args.no_cpu_baseline:
        cv, info = cpu_oracle_throughput(S, P, int_opt, budget_s=args.cpu_seconds)
        cpu = {"value": cv, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
               "sample": info["sample"], "encode_dps": info["encode_dps"], "decode_dps": info["decode_dps"],
               "note": info["note"], "core_info": info["core_info"]}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64/f64 (integer bit manipulation; float64 values)",
        "data": "synthetic", "config": make_config(S, P, int_opt),
        "compressed_bytes_per_dp": compressed_bytes / (S * P),
        "encode_dps": S * P / (enc_ms * 1e-3), "decode_dps": S * P / (dec_ms_max * 1e-3),
        "encode_ms": enc_ms, "decode_ms": dec_ms_max,
        "series_major": {"encode_ms": enc_sm_ms, "decode_ms": dec_sm_ms, "step_ms": enc_sm_ms + dec_sm_ms,
                         "decode_frac_of_hbm": alg_bytes / (dec_sm_ms * 1e-3) / 1e9 / peak,
                         "note": "the same step with series-major ([series][point]) inputs and outputs"},
        "encode_packed": {"ms": encp_ms, "dps": S * P / (encp_ms * 1e-3), "point_major_input_ms": encp_pm_ms,
                          "decode_from_packed_ms": decp_ms,
                          "step_packed_ms": encp_ms + decp_ms,
                          "note": "encode with one packed output buffer (m3tsz_encode_batch_packed) + decode of it"},
        "roofline": roofline, "roofline_encode": roofline_encode, "cpu_baseline": cpu, "e2e": e2e, "e2e_fetch": fetch, "gpu_launches": launches,
        "clocks": clocks, "fetch_allgather": allgather,
    }
    line.update(side)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
