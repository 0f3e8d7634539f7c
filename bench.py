#!/usr/bin/env python
"""bench.py — rows/s through scan + filter + GROUP BY (BASELINE.json's metric) on N B200s.

A step = one pass of the hot path over one batch of synthetic columns (SURVEY.md §8d):
    SELECT `0_1`, COUNT(*), SUM(`0_3`), AVG(`0_4`) FROM t WHERE `0_2` < 2^19 GROUP BY `0_1`
N = 1 : config C2 — 100M rows, 4 columns (int32, int32, float64, float64), 1k groups, 24 B/row.
N > 1 : config C4 — one region of 125M rows per GPU (weak scaling; N = 8 is the 1e9-row case), partial
        tables merged by ONE ncclAllGather of compact group rows + merge kernel inside bkgpu_finish.

    value      : device-resident columns, timed with CUDA events on the launching stream, max over ranks
    e2e        : same query through the C ABI with HOST (pinned, NUMA-local) columns: H2D inside the timed region;
                 e2e.pageable = the same from ordinary (pageable) host memory, e2e.warm = the region registered once
                 (bkgpu_region_register, the column-cache analogue) and queried again, e2e.cold_ms = init .. close latency
    parity     : the GPU result of the timed workload checked on every run — against Acero over the FULL table (per-region
                 Acero results summed over the ranks at N > 1), against the row-engine oracle on the cpu_baseline sample, and
                 against torch on the device columns (COUNT exact, SUM / AVG within 1e-6 relative)
    configs    : the other BASELINE.json configs on this run's GPUs (C1 count-where, C3 join + aggregate, C5 top-k over all N
                 ranks with the NCCL gather-merge): ms per step, GB/s on the config's algorithmic bytes, parity flag
    roofline / cpu_baseline : see DESIGN.md "Measurement"
`--impl reference` times the reference's CPU engine (the Acero plan it builds, all host threads); it never loads libbkgpu.so.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rows/sec scan+filter+GROUP BY"
K_FILTER = 1 << 19
N_GROUPS = 1000
BYTES_PER_ROW = 24


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default 100M at N=1, 125M per region at N>1)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1 / C3 / C5 side results")
    ap.add_argument("--no-parity", action="store_true", help="skip the Acero / oracle checks of the timed workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result columns of the last timed step to DIR/<tuple>_<slot>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir, columns):
    """columns: {"<tuple>_<slot>": array} of one GROUP BY result.  Written as float64 (COUNT fits exactly), rows ordered by the
    group key `0_1`: the engines return groups in no particular order, and a fixed order lets two builds be compared row for row."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    order = np.argsort(columns["0_1"], kind="stable")
    for name, values in columns.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(values)[order].astype(np.float64))


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def workload_name(n_gpus, rows):
    if n_gpus == 1:
        return f"C2: scan+filter+COUNT/SUM/AVG GROUP BY ({N_GROUPS} groups), {rows // 10**6}M rows x 4 cols (int32,int32,f64,f64), 1xB200"
    return (f"C4: same query, {n_gpus} regions x {rows // 10**6}M rows -> {n_gpus}xB200, partial aggregates merged by one "
            f"ncclAllGather + merge kernel")


def common_config(n_gpus, rows):
    """identical in both arms (the driver compares them)"""
    return {"workload": workload_name(n_gpus, rows), "rows_per_gpu": rows, "selectivity": 0.5, "groups": N_GROUPS,
            "algorithmic_bytes_per_row": BYTES_PER_ROW,
            "l2": f"inputs {rows * BYTES_PER_ROW / 1e9:.1f} GB per GPU >> 126 MB L2: no flush needed",
            "step": "bkgpu_reset + bkgpu_push(on_device) + bkgpu_finish + bkgpu_get_next"}


def host_cpu_info():
    """what the CPU numbers ran on: logical CPUs, CPUs this process may use, cgroup CPU quota"""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        info["sched_affinity"] = None
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota = None if txt[0] == "max" else float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0]); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                quota = None if q < 0 else q / per
            break
        except (OSError, ValueError, IndexError):
            continue
    info["cgroup_cpu_quota"] = quota
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except OSError:
        pass
    return info


# ----------------------------------------------------------------------------------------------
# clocks: sampled DURING the timed region (B200_PROFILING.md)
# ----------------------------------------------------------------------------------------------
CLOCK_SAMPLE_S = float(os.environ.get("BKGPU_BENCH_CLOCK_MS", "10")) / 1e3   # NVML queries share the driver with the launches they sit beside: a sample per 10 ms


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  NVML in a background thread (the first sample at once, then one every BKGPU_BENCH_CLOCK_MS = 10 ms); `nvidia-smi -lms` as a subprocess when pynvml is not importable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.p = None
        self.f = None
        self.nvml = None
        self.samples = []
        self.stop_flag = False
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample(self):
        n = self.nvml
        try:
            reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        except Exception:
            reasons = 0
        self.samples.append((float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)), int(reasons)))

    def _loop(self):
        while not self.stop_flag:
            try:
                self._sample()
            except Exception:
                break
            time.sleep(CLOCK_SAMPLE_S)

    def start(self):
        if self.nvml:
            import threading
            self.stop_flag = False
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.nvml:
            try:
                self._sample()   # the region has just ended (the caller synchronised): still the loaded state
            except Exception:
                pass
            self.stop_flag = True
            if self.thread:
                self.thread.join(timeout=2)
            if self.samples:
                bits = 0
                for _, r in self.samples:
                    bits |= r
                out.update(sm_mhz=statistics.median([c for c, _ in self.samples]), sm_max_mhz=self.max_sm,
                           reasons=sorted(name for bit, name in self.REASONS if bits & bit), samples=len(self.samples), source="nvml")
            return out
        if not self.p:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm), source="nvidia-smi")
        return out


# ----------------------------------------------------------------------------------------------
# reference arm: the CPU engine of the reference's vectorized path (Acero), all host threads.
# Pure numpy / pyarrow: this process never loads libbkgpu.so or torch.
# ----------------------------------------------------------------------------------------------
def host_table_numpy(rows, row0=0):
    """datagen.c2_table in chunks (the counter-based generator makes any row range independently)"""
    import numpy as np
    from baikaldb_b200 import datagen
    from baikaldb_b200.column import make_column
    from concurrent.futures import ThreadPoolExecutor
    chunk = 4_000_000
    offs = list(range(0, rows, chunk))
    with ThreadPoolExecutor(max_workers=min(32, max(1, (os.cpu_count() or 2) // 2))) as ex:   # (numpy releases the GIL in the mixing arithmetic)
        parts = list(ex.map(lambda o: datagen.c2_table(row0 + o, min(chunk, rows - o), n_groups=N_GROUPS), offs))
    return [make_column(c.tuple_id, c.slot_id, c.prim_type, np.concatenate([p[i].values for p in parts])) for i, c in enumerate(parts[0])]


def run_reference(args):
    rank, local_rank, world = env_rank()
    if rank != 0:
        return 0
    import pyarrow as pa
    from oracle import acero_oracle as A
    n_gpus = args.gpus
    rows_per_gpu = args.rows or (100_000_000 if n_gpus == 1 else 125_000_000)
    total = rows_per_gpu * n_gpus
    sample = min(total, 100_000_000)     # a bounded sample of the workload per step (the rate is per row)
    cpu = host_cpu_info()
    cores = cpu["sched_affinity"] or cpu["os_cpu_count"] or 1
    pa.set_cpu_count(cores)
    t0 = time.perf_counter()
    cols = host_table_numpy(sample)
    gen_s = time.perf_counter() - t0
    table = A.to_table(cols)
    # Acero's table_source hands out 1Mi-row batches; the thread pool works on them in parallel
    for _ in range(max(args.warmup, 1)):
        out = A.c2_filter_groupby(table, K_FILTER, use_threads=True)
    assert out.num_rows == N_GROUPS
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = A.c2_filter_groupby(table, K_FILTER, use_threads=True)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {name: out.column(name).to_numpy() for name in out.column_names})
    value = sample * args.steps / dt
    # the reference's DEFAULT executes the declaration single-threaded (FLAGS vectorlized_parallel_execution = false,
    # src/runtime/arrow_io_excutor.cpp:266-270): reported beside the all-threads number
    one = table.slice(0, min(sample, 20_000_000))
    A.c2_filter_groupby(one, K_FILTER, use_threads=False)
    t1 = time.perf_counter(); A.c2_filter_groupby(one, K_FILTER, use_threads=False); d1 = time.perf_counter() - t1
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64/f64", "data": "synthetic",
        "config": common_config(n_gpus, rows_per_gpu),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} rows of the workload per step, the Acero plan the reference builds (table_source -> filter -> "
                                   f"aggregate(hash_count_all, hash_sum, hash_mean)), use_threads=True, pyarrow {A.arrow_version()} "
                                   "(the reference pins baikalgroup/arrow release-16.1.0)",
                         "host": cpu, "acero_1thread_rows_per_s": one.num_rows / d1,
                         "acero_1thread_note": "use_threads=False is the reference's default (arrow_io_excutor.cpp:266-270)",
                         "table_generation_s": gen_s},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries also write there (NCCL prints "NCCL version ..." to stdout when
    NCCL_DEBUG is set on the box): keep the real stdout aside and point fd 1 at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def bind_to_gpu_numa(dev):
    """Run this rank's host threads (and first-touch its pinned buffers) on the NUMA node the GPU hangs off: the eight H2D
    streams of an 8-GPU node otherwise pull half their data across the socket link.  Returns a description for the JSON line."""
    bdf = None
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev)
        if all(hasattr(pr, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
            bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    except Exception:
        bdf = None
    try:
        if bdf is None:
            import pynvml
            pynvml.nvmlInit()
            bdf = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(dev)).busId
            bdf = bdf.decode() if isinstance(bdf, bytes) else bdf
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:      # NVML prints an 8-digit domain, sysfs uses 4
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"node": None, "note": "single NUMA node"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus": len(allowed)}
    except Exception as e:   # best effort: the numbers are still valid, only possibly slower
        return {"node": None, "note": f"not bound: {type(e).__name__}"}


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    import numpy as np
    import torch
    import torch.distributed as dist
    from baikaldb_b200 import _lib, datagen, queries
    from baikaldb_b200._lib import BkgpuColumn, BkgpuStats
    from baikaldb_b200.plan import PrimitiveType as T

    rank, local_rank, world = env_rank()
    n_gpus = args.gpus
    if world != n_gpus:
        if world == 1 and n_gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run --nproc-per-node N")
    torch.cuda.set_device(local_rank)
    dev = local_rank
    numa = bind_to_gpu_numa(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    L = _lib.lib()
    rows = args.rows or (100_000_000 if n_gpus == 1 else 125_000_000)
    row0 = rank * rows
    stream = torch.cuda.current_stream()
    DT = {int(T.INT32): torch.int32, int(T.INT64): torch.int64, int(T.DOUBLE): torch.float64}

    def gen_col(n, prim, gdist, seed, column_id, r0=0, lo=0, hi=0, scale=1.0):
        t = torch.empty(n, dtype=DT[int(prim)], device="cuda")
        _lib.check(L.bkgpu_gen_column(dev, t.data_ptr(), int(prim), gdist, seed, column_id, r0, n, lo, hi, scale))
        return t

    def col_array(specs):
        """specs: (tuple, slot, prim, tensor)"""
        arr = (BkgpuColumn * len(specs))()
        for i, (tup, slot, prim, t) in enumerate(specs):
            arr[i].tuple_id, arr[i].slot_id, arr[i].prim_type, arr[i].elem_size = tup, slot, int(prim), 0
            arr[i].values, arr[i].validity, arr[i].length = t.data_ptr(), None, t.numel()
        return arr

    # ---- synthetic region of this rank, generated in HBM ----
    tensors = []
    for slot, pt, gdist, lo, hi, scale in datagen.C2_COLUMNS:
        tensors.append(gen_col(rows, pt, gdist, 2, slot, row0, lo, N_GROUPS if slot == 1 else hi, scale))
    dcols = col_array([(0, c[0], c[1], t) for c, t in zip(datagen.C2_COLUMNS, tensors)])

    # ---- NCCL communicator of the library (unique id travels over torch.distributed) ----
    comm = ctypes.c_void_p()
    if world > 1:
        idbuf = (ctypes.c_uint8 * 128)()
        if rank == 0:
            _lib.check(L.bkgpu_nccl_unique_id(idbuf))
        idt = torch.tensor(list(idbuf), dtype=torch.uint8, device="cuda")
        dist.broadcast(idt, 0)
        idbuf = (ctypes.c_uint8 * 128)(*idt.cpu().tolist())
        _lib.check(L.bkgpu_nccl_comm_create(ctypes.byref(comm), idbuf, world, rank, dev))

    bench_opts = [kv.split("=") for kv in filter(None, os.environ.get("BKGPU_BENCH_OPTS", "").split(","))]   # A/B of kernel variants

    def open_plan(plan, with_comm=True, extra=()):
        pb = plan.serialize()
        hh = ctypes.c_void_p()
        _lib.check(L.bkgpu_init(ctypes.byref(hh), pb, len(pb), dev, comm if (world > 1 and with_comm) else None))
        _lib.check(L.bkgpu_set_option(hh, b"stream", stream.cuda_stream), hh)
        for k, v in list(bench_opts) + list(extra):
            _lib.check(L.bkgpu_set_option(hh, k.encode() if isinstance(k, str) else k, int(v)), hh)
        _lib.check(L.bkgpu_open(hh), hh)
        return hh, pb

    h, plan_bytes = open_plan(queries.c2_filter_groupby(K_FILTER))   # default options: nothing a planner would not know
    out = (BkgpuColumn * 16)()

    def drain(hh, keep=False):
        eos = ctypes.c_int(0)
        nrows_total, nbytes, kept = 0, 0, {}
        while not eos.value:
            ncols, nrows = ctypes.c_int(16), ctypes.c_int64(0)
            _lib.check(L.bkgpu_get_next(hh, out, ctypes.byref(ncols), ctypes.byref(nrows), ctypes.byref(eos)), hh)
            n = nrows.value
            nrows_total += n
            nbytes += sum(out[i].elem_size for i in range(ncols.value)) * n
            if keep and n:
                for i in range(ncols.value):
                    dt = {int(T.INT32): np.int32, int(T.INT64): np.int64, int(T.DOUBLE): np.float64}.get(out[i].prim_type)
                    if dt is None:
                        continue
                    a = np.frombuffer((ctypes.c_uint8 * (n * np.dtype(dt).itemsize)).from_address(out[i].values), dtype=dt).copy()
                    key = (out[i].tuple_id, out[i].slot_id)
                    kept[key] = a if key not in kept else np.concatenate([kept[key], a])
        return nrows_total, nbytes, kept

    def step(cols, on_device, hh=None, ncols=4, nrows=None, keep=False):
        hh = hh or h
        _lib.check(L.bkgpu_reset(hh), hh)
        _lib.check(L.bkgpu_push(hh, cols, ncols, rows if nrows is None else nrows, on_device), hh)
        _lib.check(L.bkgpu_finish(hh), hh)
        return drain(hh, keep)

    def get_stats(hh=None):
        st = BkgpuStats()
        _lib.check(L.bkgpu_get_stats(hh or h, ctypes.byref(st)), hh or h)
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run_step, steps, warmup, hh=None, all_ranks=True, keep_last=False):
        """all_ranks=False: a measurement only this rank takes part in (no barrier, no reduction over the ranks);
        keep_last: the last timed step copies its result columns out (run_step(keep=True))"""
        sync = barrier if all_ranks else torch.cuda.synchronize
        for _ in range(warmup):
            run_step()
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(dev)
        sampler.start()
        launches0 = get_stats(hh).kernel_launches
        e0.record(stream)
        res = None
        kernel_ms, kernel_launches, kernel_bytes, coll_ms = 0.0, 0, 0, 0.0
        for i in range(steps):
            res = run_step(keep=True) if keep_last and i == steps - 1 else run_step()
            st = get_stats(hh)
            kernel_ms += st.main_kernel_ms; kernel_launches += st.main_kernel_launches
            kernel_bytes += st.main_kernel_bytes; coll_ms += st.collective_ms
        e1.record(stream)
        sync()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1)
        if world > 1 and all_ranks:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        st = get_stats(hh)
        return {"ms": ms, "res": res, "clocks": clocks, "launches": st.kernel_launches - launches0, "stats": st,
                "kernel_ms": kernel_ms, "kernel_launches": kernel_launches, "kernel_bytes": kernel_bytes, "coll_ms": coll_ms}

    # ---- value: device-resident columns ----
    r = timed(lambda keep=False: step(dcols, 1, keep=keep), args.steps, max(args.warmup, 3), keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"{tup}_{slot}": v for (tup, slot), v in r["res"][2].items()})
    if os.environ.get("BKGPU_BENCH_TRACE"):   # per-rank view of the timed region (stderr)
        sys.stderr.write(f"[rank {rank}] step {r['ms'] / args.steps:.4f} ms  kernel {r['kernel_ms'] / max(r['kernel_launches'], 1):.4f} ms  "
                         f"collective {r['coll_ms'] / args.steps:.4f} ms  launches/step {r['launches'] / args.steps:.1f}\n")
    total_rows = rows * world
    value = total_rows * args.steps / (r["ms"] / 1e3)
    ngroups_out = r["res"][0]

    # ---- parity of the timed workload (not timed) ----
    parity = {}

    def gpu_result(cols=dcols, n=None):
        _, _, kept = step(cols, 1, nrows=n, keep=True)
        order = np.argsort(kept[(0, 1)])
        return {k: v[order] for k, v in kept.items()}

    def same_groups(got, keys, cnt, sa, avg):
        ok = len(got[(0, 1)]) == len(keys) and np.array_equal(got[(0, 1)], keys)
        ok = ok and np.array_equal(got[(1, 1)], cnt)                                       # COUNT(*): bit-exact
        ok = ok and np.allclose(got[(1, 2)], sa, rtol=1e-6, atol=0)                        # SUM(double): 1e-6 relative
        ok = ok and np.allclose(got[(1, 3)], avg, rtol=1e-6, atol=1e-9)                    # AVG(double)
        return bool(ok)

    try:   # torch on the same device columns (full size, every rank's region, summed over the ranks)
        key, filt, a, b = tensors
        m = filt < K_FILTER
        k64 = key[m].to(torch.int64)
        cnt = torch.bincount(k64, minlength=N_GROUPS)
        sa = torch.zeros(N_GROUPS, dtype=torch.float64, device="cuda").index_add_(0, k64, a[m])
        sb = torch.zeros(N_GROUPS, dtype=torch.float64, device="cuda").index_add_(0, k64, b[m])
        if world > 1:
            for t in (cnt, sa, sb):
                dist.all_reduce(t)
        got_full = gpu_result()
        parity["torch_full"] = same_groups(got_full, np.arange(N_GROUPS), cnt.cpu().numpy(), sa.cpu().numpy(), (sb / cnt).cpu().numpy())
        del m, k64, cnt, sa, sb
    except Exception as e:  # verification must never hide the measurement
        parity["torch_full"] = f"error: {type(e).__name__}: {e}"
        got_full = None

    host_np = None
    if not args.no_parity:
        try:   # Acero (the reference's vectorized engine) over the full table: this rank's region, partial results summed over the ranks
            import pyarrow as pa
            from baikaldb_b200.column import make_column
            from oracle import acero_oracle as A
            host_np = [t.cpu().numpy() for t in tensors]
            pa.set_cpu_count(max(1, (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()) // max(world, 1)))
            table = A.to_table([make_column(0, c[0], c[1], v) for c, v in zip(datagen.C2_COLUMNS, host_np)])
            t0 = time.perf_counter()
            res = A.c2_filter_groupby(table, K_FILTER, use_threads=True)
            acero_s = time.perf_counter() - t0
            ak = res.column("0_1").to_numpy(); o = np.argsort(ak)
            part = np.zeros((3, N_GROUPS), dtype=np.float64)          # count, sum(0_3), sum(0_4) = mean x count, by group key
            acnt = res.column("1_1").to_numpy()[o].astype(np.int64)
            part[0, ak[o]] = acnt
            part[1, ak[o]] = res.column("1_2").to_numpy()[o]
            part[2, ak[o]] = res.column("1_3").to_numpy()[o] * acnt
            cnt_t = torch.from_numpy(part[0].astype(np.int64)).cuda()
            sums_t = torch.from_numpy(part[1:]).cuda()
            if world > 1:
                dist.all_reduce(cnt_t); dist.all_reduce(sums_t)
            acnt = cnt_t.cpu().numpy(); asum = sums_t.cpu().numpy()
            if got_full is not None:
                parity["acero_full"] = same_groups(got_full, np.arange(N_GROUPS), acnt, asum[0], asum[1] / np.maximum(acnt, 1))
            parity["acero_rows_checked"] = int(total_rows)
            parity["acero_seconds_per_region"] = acero_s
            del table, res
        except Exception as e:
            parity["acero_full"] = f"error: {type(e).__name__}: {e}"

    # ---- e2e: host columns through the same calls, H2D inside the timed region ----
    e2e = None
    if not args.no_e2e:
        e_steps = max(1, min(args.steps, 10))
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in tensors]    # first touched on this rank's NUMA node
        for hb, t in zip(host, tensors):
            hb.copy_(t)
        torch.cuda.synchronize()
        hcols = col_array([(0, c[0], c[1], hb) for c, hb in zip(datagen.C2_COLUMNS, host)])
        re = timed(lambda: step(hcols, 0), e_steps, 1)
        e2e = {"value": total_rows * e_steps / (re["ms"] / 1e3), "unit": "rows/s", "steps": e_steps,
               "ms_per_step": re["ms"] / e_steps, "h2d_bytes_per_step": rows * BYTES_PER_ROW * world,
               "d2h_bytes_per_step": int(re["res"][1]) + 16, "host_memory": "pinned (cudaHostAlloc), first touched on the GPU's NUMA node",
               "numa": numa, "h2d_gbs_per_gpu": rows * BYTES_PER_ROW * e_steps / (re["ms"] / 1e3) / 1e9}
        # pageable host memory (what an Arrow RecordBatch hands over): threaded copy into pinned bounce buffers inside the library
        try:
            if host_np is None:
                host_np = [t.cpu().numpy() for t in tensors]
            pcols = (BkgpuColumn * 4)()
            for i, (c, v) in enumerate(zip(datagen.C2_COLUMNS, host_np)):
                pcols[i].tuple_id, pcols[i].slot_id, pcols[i].prim_type, pcols[i].elem_size = 0, c[0], int(c[1]), 0
                pcols[i].values, pcols[i].validity, pcols[i].length = v.ctypes.data, None, rows
            p_steps = max(1, min(args.steps, 5))
            rp = timed(lambda: step(pcols, 0), p_steps, 1)
            e2e["pageable"] = {"value": total_rows * p_steps / (rp["ms"] / 1e3), "ms_per_step": rp["ms"] / p_steps,
                               "h2d_gbs_per_gpu": rows * BYTES_PER_ROW * p_steps / (rp["ms"] / 1e3) / 1e9,
                               "of_pinned": (re["ms"] / e_steps) / (rp["ms"] / p_steps)}
        except Exception as e:
            e2e["pageable"] = f"error: {type(e).__name__}: {e}"
        # warm: the region registered once (host -> HBM, timed as `register_ms`), then queried from the resident copy
        try:
            region_id = 1000 + rank
            torch.cuda.synchronize(); t0 = time.perf_counter()
            _lib.check(L.bkgpu_region_register(dev, region_id, hcols, 4, rows, 0))
            reg_ms = (time.perf_counter() - t0) * 1e3

            def warm_step():
                _lib.check(L.bkgpu_reset(h), h)
                _lib.check(L.bkgpu_push_region(h, region_id), h)
                _lib.check(L.bkgpu_finish(h), h)
                return drain(h)
            rw = timed(warm_step, e_steps, 1)
            e2e["warm"] = {"value": total_rows * e_steps / (rw["ms"] / 1e3), "ms_per_step": rw["ms"] / e_steps, "register_ms": reg_ms,
                           "note": "region resident in HBM (bkgpu_region_register), query = reset + push_region + finish + get_next"}
            _lib.check(L.bkgpu_region_evict(dev, region_id))
        except Exception as e:
            e2e["warm"] = f"error: {type(e).__name__}: {e}"
        # cold latency of ONE request: the reference builds the tree per request (src/store/region.cpp:3072)
        try:
            cold = {}
            for trial in ("first", "second"):   # (the second request in the process shows what a store pays per query once the driver is warm)
                torch.cuda.synchronize(); t0 = time.perf_counter(); marks = []
                pbc = queries.c2_filter_groupby(K_FILTER).serialize()
                hc = ctypes.c_void_p()
                _lib.check(L.bkgpu_init(ctypes.byref(hc), pbc, len(pbc), dev, None)); marks.append(("init", time.perf_counter()))
                _lib.check(L.bkgpu_set_option(hc, b"stream", stream.cuda_stream), hc)
                _lib.check(L.bkgpu_open(hc), hc); marks.append(("open", time.perf_counter()))
                _lib.check(L.bkgpu_push(hc, dcols, 4, rows, 1), hc); marks.append(("push", time.perf_counter()))
                _lib.check(L.bkgpu_finish(hc), hc); marks.append(("finish", time.perf_counter()))
                drain(hc); marks.append(("get_next", time.perf_counter()))
                L.bkgpu_close(hc); marks.append(("close", time.perf_counter()))
                prev = t0; parts = {}
                for name, t in marks:
                    parts[name] = round((t - prev) * 1e3, 3); prev = t
                cold[trial] = {"total": round((marks[-1][1] - t0) * 1e3, 3), **parts}
            e2e["cold_ms"] = {"device_resident_init_to_close": cold["second"]["total"], "calls": cold,
                              "note": "bkgpu_init + open + push + finish + get_next + close of a NEW plan (no communicator), wall clock per call"}
        except Exception as e:
            e2e["cold_ms"] = f"error: {type(e).__name__}: {e}"
        e2e["parity"] = parity
        del host

    # ---- roofline of the dominant kernel (algorithmic bytes / CUDA-event duration of its launches) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    achieved = (r["kernel_bytes"] / max(r["kernel_launches"], 1)) / (r["kernel_ms"] / max(r["kernel_launches"], 1) / 1e3) / 1e9 if r["kernel_ms"] > 0 else 0.0
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "latest_traffic.json")))
        kname = r["stats"].main_kernel_name.decode()
        entry = prof.get(kname) or prof.get(kname.replace("_fx", ""))   # (the FX variant reads the same columns once: no capture of its own yet -> the lean kernel's)
        if entry:  # DRAM bytes per launch, scaled from the committed ncu capture to this launch's row count
            traffic = entry["dram_bytes_per_row"] * rows
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": r["stats"].main_kernel_name.decode(), "peak_source": peak_src,
                "kernel_ms_per_launch": r["kernel_ms"] / max(r["kernel_launches"], 1),
                "kernel_share_of_step": r["kernel_ms"] / r["ms"] if r["ms"] else None,
                "collective_ms_per_step": r["coll_ms"] / args.steps}

    # ---- CPU baseline beside it (rank 0, N = 1): the row-engine restatement, one thread; its result checks the GPU's ----
    cpu_baseline = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        from baikaldb_b200.column import make_column
        from oracle import oracle as row_oracle

        def sample_cols(n):
            return [make_column(0, dcols[i].slot_id, dcols[i].prim_type, tensors[i][:n].cpu().numpy()) for i in range(4)]
        probe = sample_cols(1_000_000)
        t0 = time.perf_counter(); row_oracle.execute(plan_bytes, probe); dt = time.perf_counter() - t0
        n_s = int(min(rows, max(2_000_000, 15.0 / (dt / 1e6))))
        cols = sample_cols(n_s)
        t0 = time.perf_counter(); res = row_oracle.execute(plan_bytes, cols); dt = time.perf_counter() - t0
        cpu_baseline = {"value": n_s / dt, "unit": "rows/s", "cores": 1, "kind": "port",
                        "sample": f"first {n_s} rows of the workload, oracle/bk_oracle.c (row-engine restatement, one thread like one bthread per fragment)",
                        "host": host_cpu_info(), "seconds": dt, "groups": res.nrows}
        try:   # the same rows through the GPU path must give the oracle's groups
            sub = col_array([(0, c[0], c[1], t[:n_s]) for c, t in zip(datagen.C2_COLUMNS, tensors)])
            got_s = gpu_result(cols=sub, n=n_s)
            oc = {c.name: c for c in res.columns}
            oo = np.argsort(oc["0_1"].values)
            parity["oracle_sample"] = same_groups(got_s, oc["0_1"].values[oo], oc["1_1"].values[oo], oc["1_2"].values[oo], oc["1_3"].values[oo])
            parity["oracle_rows_checked"] = n_s
        except Exception as e:
            parity["oracle_sample"] = f"error: {type(e).__name__}: {e}"
        cpu_baseline["parity_vs_gpu"] = parity.get("oracle_sample")

    # ---- the other BASELINE.json configs on these GPUs ----
    configs = None
    if not args.no_configs:
        configs = {}
        c_steps, c_warm = max(3, min(args.steps, 10)), 2

        def side(name, plan, pushes, n_rows, algo_bytes, check, with_comm=False, steps=c_steps):
            """pushes: [(col_array, ncols, nrows)]; check(kept) -> bool"""
            try:
                hh, _ = open_plan(plan, with_comm=with_comm)

                def one(keep=False):
                    _lib.check(L.bkgpu_reset(hh), hh)
                    for arr, nc, nr in pushes:
                        _lib.check(L.bkgpu_push(hh, arr, nc, nr, 1), hh)
                    _lib.check(L.bkgpu_finish(hh), hh)
                    return drain(hh, keep)
                rr = timed(one, steps, c_warm, hh=hh, all_ranks=False)
                ms = rr["ms"] / steps
                _, _, kept = one(keep=True)
                ok = check(kept)
                st = rr["stats"]
                configs[name] = {"ms_per_step": ms, "rows": n_rows, "rows_per_s": n_rows / (ms / 1e3), "algorithmic_bytes": algo_bytes,
                                 "gbs": algo_bytes / (ms / 1e3) / 1e9 / (world if with_comm else 1), "frac_of_measured_hbm": algo_bytes / (ms / 1e3) / 1e9 / peak / (world if with_comm else 1),
                                 "main_kernel": st.main_kernel_name.decode(), "main_kernel_ms": rr["kernel_ms"] / steps,
                                 "gpu_launches_per_step": rr["launches"] / steps, "parity": ok}
                L.bkgpu_close(hh)
            except Exception as e:
                configs[name] = {"error": f"{type(e).__name__}: {e}"}

        if rank == 0:
            # C1: COUNT(*) WHERE int32 < k at a bandwidth-relevant size (the 1M-row case of BASELINE.json is a plumbing test)
            n1 = 100_000_000
            x = gen_col(n1, T.INT32, 0, 1, 1, 0, 0, 1 << 20)
            want1 = int((x < K_FILTER).sum().item())
            side("C1_count_where_100M", queries.c1_count_where(K_FILTER), [(col_array([(0, 1, T.INT32, x)]), 1, n1)], n1, 4 * n1,
                 lambda k: int(k[(1, 1)][0]) == want1)
            del x
            # C3: 100M-row fact JOIN 10M-row dimension ON int32 key, GROUP BY a dimension attribute
            nf, nd = 100_000_000, 10_000_000
            fk = gen_col(nf, T.INT32, 0, 3, 1, 0, 0, nd); v = gen_col(nf, T.DOUBLE, 1, 3, 2)
            pk = gen_col(nd, T.INT32, datagen.DIST_PERMUTATION, 3, 11, 0, 0, nd); attr = gen_col(nd, T.INT32, 0, 3, 12, 0, 0, N_GROUPS)
            attr_of_key = torch.empty(nd, dtype=torch.int64, device="cuda"); attr_of_key[pk.to(torch.int64)] = attr.to(torch.int64)
            grp = attr_of_key[fk.to(torch.int64)]
            cnt3 = torch.bincount(grp, minlength=N_GROUPS).cpu().numpy()
            sv3 = torch.zeros(N_GROUPS, dtype=torch.float64, device="cuda").index_add_(0, grp, v).cpu().numpy()
            del attr_of_key, grp

            def check3(k):
                o = np.argsort(k[(1, 2)])
                return bool(np.array_equal(k[(1, 2)][o], np.arange(N_GROUPS)) and np.array_equal(k[(2, 1)][o], cnt3) and np.allclose(k[(2, 2)][o], sv3, rtol=1e-6, atol=0))
            side("C3_join_groupby_100Mx10M", queries.c3_join_groupby(),
                 [(col_array([(1, 1, T.INT32, pk), (1, 2, T.INT32, attr)]), 2, nd), (col_array([(0, 1, T.INT32, fk), (0, 2, T.DOUBLE, v)]), 2, nf)],
                 nf, 12 * nf + 8 * nd, check3, steps=max(2, c_steps // 2))
            del fk, v, pk, attr
        # C5: ORDER BY int64 LIMIT 1000 — one region of 125M rows per GPU, every rank, merged by the NCCL gather-merge at N > 1
        n5 = 125_000_000
        k5 = gen_col(n5, T.INT64, 3, 5, 1, rank * n5); p5 = gen_col(n5, T.INT32, 0, 5, 2, rank * n5, 0, 1 << 30)
        top = torch.topk(k5, 1000, largest=False, sorted=True)
        tk, tp = top.values, p5[top.indices].to(torch.int64)
        if world > 1:   # the global top-k = top-k of the ranks' top-k
            allk = [torch.empty_like(tk) for _ in range(world)]; allp = [torch.empty_like(tp) for _ in range(world)]
            dist.all_gather(allk, tk); dist.all_gather(allp, tp)
            ck, cp = torch.cat(allk), torch.cat(allp)
            o = torch.argsort(ck, stable=True)[:1000]
            tk, tp = ck[o], cp[o]
        tk, tp = tk.cpu().numpy(), tp.cpu().numpy()

        def check5(k):
            return bool(len(k[(0, 1)]) == 1000 and np.array_equal(k[(0, 1)], tk) and np.array_equal(k[(0, 2)].astype(np.int64), tp))
        saved = configs
        try:
            hh5, _ = open_plan(queries.c5_topk(1000), with_comm=True, extra=[(b"region_base", rank * n5)])
            arr5 = col_array([(0, 1, T.INT64, k5), (0, 2, T.INT32, p5)])

            def one5(keep=False):
                _lib.check(L.bkgpu_reset(hh5), hh5)
                _lib.check(L.bkgpu_push(hh5, arr5, 2, n5, 1), hh5)
                _lib.check(L.bkgpu_finish(hh5), hh5)
                return drain(hh5, keep)
            r5 = timed(one5, c_steps, c_warm, hh=hh5)
            ms5 = r5["ms"] / c_steps
            _, _, kept5 = one5(keep=True)
            ok5 = check5(kept5)
            if world > 1:
                f = torch.tensor([1 if ok5 else 0], device="cuda"); dist.all_reduce(f, op=dist.ReduceOp.MIN); ok5 = bool(f.item())
            saved[f"C5_topk_1000_of_{world}x125M"] = {
                "ms_per_step": ms5, "rows": n5 * world, "rows_per_s": n5 * world / (ms5 / 1e3), "algorithmic_bytes": 8 * n5 * world,
                "gbs": 8 * n5 / (ms5 / 1e3) / 1e9, "frac_of_measured_hbm": 8 * n5 / (ms5 / 1e3) / 1e9 / peak,
                "main_kernel": r5["stats"].main_kernel_name.decode(), "main_kernel_ms": r5["kernel_ms"] / c_steps,
                "gpu_launches_per_step": r5["launches"] / c_steps, "collective_ms_per_step": r5["coll_ms"] / c_steps, "parity": ok5,
                "note": "per-GPU GB/s on 8 B/row; every rank holds the merged top-k (ties by (region, row))"}
            L.bkgpu_close(hh5)
        except Exception as e:
            saved[f"C5_topk_1000_of_{world}x125M"] = {"error": f"{type(e).__name__}: {e}"}
        del k5, p5

    if rank == 0:
        parity_ok = all(v is True for k, v in parity.items() if k in ("torch_full", "acero_full", "oracle_sample"))
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": r["ms"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64/f64", "data": "synthetic",
            "config": common_config(n_gpus, rows),
            "clocks": {k: r["clocks"][k] for k in ("sm_mhz", "sm_max_mhz", "reasons")},
            "e2e": e2e, "gpu_launches": int(r["launches"]), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "hbm_gbs_whole_step": total_rows * BYTES_PER_ROW * args.steps / (r["ms"] / 1e3) / 1e9 / world,
            "result_groups": ngroups_out, "parity": parity, "parity_ok": parity_ok, "verified_vs_torch": parity.get("torch_full"),
            "configs": configs, "options": dict((k, int(v)) for k, v in bench_opts),
        }
        emit(line)
    L.bkgpu_close(h)
    if world > 1:
        L.bkgpu_nccl_comm_destroy(comm)
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
