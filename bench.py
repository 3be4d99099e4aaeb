#!/usr/bin/env python3
"""bench.py -- H.x throughput of the B200-native hot path (driver contract; DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--dtype c128|f64] [--secondary a,b|none]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's algorithm on the host cores (oracle port)

A "step" is one matrix-vector product y <- H x over the whole basis of the workload.  The workload is
``heisenberg_square_6x6`` (BASELINE.json configs[4], the configuration the 1/2/4/8-GPU sweep of the metric is quoted
on; it fits one B200) for EVERY N, so the driver's 1 -> 8 curve measures a problem that can scale; the other BASELINE
configs run as ``secondary`` entries of the same JSON line (a few products each, with their own parity figure).

  value        basis states / s with x, y resident in HBM: CUDA events on the launching stream around each product,
               L2 flushed between timed products, max over ranks.  Under torchrun (N > 1) the basis is hash-partitioned
               over the ranks (hash64_01 % N, reference src/StatesEnumeration.chpl:122-136) and the product is the
               collective dmv_matvec (exchange named in ``run.exchange``); scaling is "strong".
  e2e          the same metric through the public host-buffer call (pinned host x -> C ABI -> host y), H2D and D2H
               inside the timed region.
  parity       EVERY line, at every N: max error of sampled rows of y against the CPU oracle, which recomputes those
               rows column by column (oracle_expected_rows: y[i] = D_i x_i + sum_b conj(H_bi) x_b with H_bi from
               computeOffDiag on source i), using the reference's criterion |a-b| <= max(1e-14, 1e-12 max(|a|,|b|))
               (test/TestMatrixVectorProduct.chpl:15-20).  x follows the reference's recipe (input_for_matvec.py:8,31:
               RandomState(42), rand(N) - 0.5 in global sorted order; the imaginary part continues the stream).
  roofline     algorithmic bytes of SURVEY.md 8(d) / duration of the dominant kernel against MEASURED_PEAKS.json, plus
               what actually limits that kernel (measured DRAM traffic, issue-slot share) from the committed ncu
               capture (profiles/ncu_constants.json).
  cpu_baseline the reference's algorithm restated in C (oracle/oracle.c, OpenMP, group elements as Benes networks) on
               a bounded slab of source rows, on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# pin the OpenMP threads of the CPU arm before libgomp is loaded (two boxes of the pool disagreed 6x without it) -- only
# when this process is alone: under torchrun every rank would bind its main thread to the SAME first place and the
# ranks would time-share one core (8 GPUs: ms-scale launch jitter, measured)
if int(os.environ.get("WORLD_SIZE", "1")) == 1:
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DEFAULT_WORKLOAD = "heisenberg_square_6x6"   # BASELINE.json configs[4]: the scaling-sweep configuration
SECONDARY = ["heisenberg_chain_24", "heisenberg_kagome_16", "heisenberg_chain_32_symm", "heisenberg_chain_36_symm"]
X_RECIPE = "numpy RandomState(42): rand(N) - 0.5 in global sorted order (+ 1j (rand(N) - 0.5) for c128)"
L2_NOTE = "GPU arm: 256 MB written between timed products (L2 flush); CPU arm: not applicable"
METRIC = "H.x basis states/s"
DUMP_ROWS, DUMP_SEED = 1 << 21, 0     # --dump-outputs: 48 MB for c128


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DMV_WORKLOAD", DEFAULT_WORKLOAD))
    ap.add_argument("--dtype", default=os.environ.get("DMV_DTYPE", "c128"), choices=["c128", "f64"])
    ap.add_argument("--secondary", default=os.environ.get("DMV_SECONDARY", ",".join(SECONDARY)),
                    help="comma-separated workloads measured briefly beside the main one, or 'none'")
    ap.add_argument("--sample-rows", type=int, default=2048, help="rows per rank checked against the oracle")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write y of the last timed product (a fixed, seeded sample of its rows) as DIR/*.npy")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------------------
# helpers shared by both arms (nothing of the product is imported here)
# ------------------------------------------------------------------------------------------------------------------
def recipe_x(n: int, cplx: bool) -> np.ndarray:
    """The reference's input recipe (input_for_matvec.py:8,31) in global sorted order."""
    rs = np.random.RandomState(42)
    x = rs.rand(n) - 0.5
    if cplx:
        x = x + 1j * (rs.rand(n) - 0.5)
    return x


def _affinity_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


_HOST_THREADS = _affinity_threads()   # read before libgomp binds the main thread to one place (OMP_PROC_BIND)


def host_threads() -> int:
    return _HOST_THREADS


def host_description() -> dict:
    model, quota = None, None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                quota = f.read().strip()
            break
        except OSError:
            continue
    return {"cpu_model": model, "cgroup_cpu_quota": quota, "affinity_threads": host_threads(),
            "omp_proc_bind": os.environ.get("OMP_PROC_BIND"), "omp_places": os.environ.get("OMP_PLACES")}


def criterion_violations(a: np.ndarray, b: np.ndarray) -> int:
    """Elements failing the reference's approxEqual (test/TestMatrixVectorProduct.chpl:15-20)."""
    return int(np.count_nonzero(np.abs(a - b) > np.maximum(1e-14, 1e-12 * np.maximum(np.abs(a), np.abs(b)))))


class CpuArm:
    """The reference's product on the host cores: oracle/oracle.c with the group as Benes networks, OpenMP over the
    chunks of a slab of source rows (kind "port": the Chapel + Haskell toolchain of the reference is not in the image)."""

    def __init__(self, workload: str, cplx: bool, reps: np.ndarray | None = None):
        from oracle import model as omodel
        from oracle import pyoracle as po
        self.po = po
        po.set_num_threads(host_threads())     # torchrun exports OMP_NUM_THREADS=1: use every host thread anyway
        self.threads = po.num_threads()
        self.basis, self.matrix = omodel.load_model(os.path.join(ROOT, "data", workload + ".yaml"))
        self.model = po.Model(self.matrix, networks=True)
        t = time.perf_counter()
        self.reps = reps if reps is not None else po.enumerate_states_parallel(self.basis, networks=True)[0]
        self.enumerate_s = time.perf_counter() - t
        self.n = int(self.reps.shape[0])
        self.x = recipe_x(self.n, cplx)
        self.y = np.zeros_like(self.x)
        self.slab = None

    def run_slab(self, lo: int, hi: int) -> float:
        t = time.perf_counter()
        self.po.matvec_rows(self.model, self.reps, self.x, self.y, lo, hi, num_tasks=self.threads)
        return time.perf_counter() - t

    def calibrate(self, seconds_per_step: float):
        """Pick a contiguous slab of source rows in the middle of the basis that takes about seconds_per_step."""
        probe = min(self.n, max(64 * self.threads, 4096))
        mid = self.n // 2
        lo = max(0, mid - probe // 2)
        self.run_slab(lo, lo + probe)                       # touch the pages, start the threads
        dt = self.run_slab(lo, lo + probe)
        rows = int(min(self.n, max(probe, probe * seconds_per_step / max(dt, 1e-6))))
        lo = max(0, mid - rows // 2)
        self.slab = (lo, lo + rows)
        return self.slab

    def step(self) -> float:
        return self.run_slab(*self.slab)

    def sample_text(self) -> str:
        lo, hi = self.slab
        frac = (hi - lo) / self.n
        return (f"source rows [{lo}, {hi}) of {self.n} ({100 * frac:.2f} % of the product: diagonal, term generation, "
                f"orbit scans as Benes networks, search, atomic add), {self.threads} OpenMP threads")


def run_reference(args):
    """`--impl reference`: nothing of the product is imported -- model inputs through oracle/model.py, basis through
    the oracle's parallel enumeration (untimed), each step = one bounded slab of the product."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cplx = args.dtype == "c128"
    arm = CpuArm(args.workload, cplx)
    arm.calibrate(1.0)
    rows = arm.slab[1] - arm.slab[0]
    for _ in range(args.warmup):
        arm.step()
    times = [arm.step() for _ in range(args.steps)]
    ms = 1e3 * float(np.mean(times))
    value = rows / (ms * 1e-3)
    nnz = count_terms_cpu(arm)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "states/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": args.workload, "basis_states": arm.n, "off_diag_terms": nnz, "x": X_RECIPE, "l2": L2_NOTE},
        "cpu_baseline": {"value": value, "unit": "states/s", "cores": arm.threads, "kind": "port",
                         "sample": arm.sample_text(), "ms_best_step": 1e3 * float(np.min(times)),
                         "basis_enumeration_s": arm.enumerate_s, **host_description()},
        "e2e": {"value": value, "unit": "states/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def count_terms_cpu(arm: CpuArm) -> int:
    """Emitted off-diagonal terms of the whole product (the `off_diag_terms` of the config), by the oracle's term
    kernel over the whole basis in chunks (integer work only: no orbit scans)."""
    po, total = arm.po, 0
    off = arm.matrix.off_diag
    lib = po.lib()
    step = 1 << 18
    betas = np.zeros(step * max(1, len(off)), dtype=np.uint64)
    coeffs = np.zeros(step * max(1, len(off)), dtype=np.complex128)
    offsets = np.zeros(step + 1, dtype=np.int64)
    for lo in range(0, arm.n, step):
        chunk = np.ascontiguousarray(arm.reps[lo:lo + step])
        total += int(lib.oracle_apply_off_diag_x1(len(off), off.v, off.m, off.r, off.x, off.s, chunk.shape[0], chunk,
                                                  betas, coeffs, offsets, None, 1))
    return total


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML, every DMV_CLOCK_PERIOD_MS = 5 ms)."""

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if visible:
                try:
                    idx = int(visible.split(",")[self.index])
                except ValueError:
                    pass
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                    "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                    "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                self._stop.wait(1e-3 * float(os.environ.get("DMV_CLOCK_PERIOD_MS", "5")))
        except Exception as e:  # NVML missing: fall back to one nvidia-smi query
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                a, b = [float(v) for v in out.stdout.strip().split(",")]
                self.sm.append(a)
                self.sm_max = b
            except Exception:
                self.reasons.add(f"unsampled ({type(e).__name__})")

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        time.sleep(0.01)
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons) or ["unsampled"]}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(sm)}


def ncu_constants(key: str):
    """Per-launch figures of the dominant kernel from the committed ncu capture (profiles/ncu_constants.json)."""
    path = os.path.join(ROOT, "profiles", "ncu_constants.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(key)
    return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class Workload:
    """One model input on this rank: operator, local block of the hash partition, x by the reference's recipe."""

    def __init__(self, name: str, cplx: bool, world: int, rank: int, local_rank: int):
        import torch
        from distributed_matvec_b200 import DistributedOperator, Operator, load_config_from_yaml
        self.name, self.cplx, self.world, self.rank = name, cplx, world, rank
        self.E = 16 if cplx else 8
        basis, matrix = load_config_from_yaml(os.path.join(ROOT, "data", name + ".yaml"))
        self.group_order = len(basis.group) if basis.requires_projection() else 1
        t0 = time.perf_counter()
        if world > 1:
            self.dop = DistributedOperator(matrix, device=local_rank)
            self.op = self.dop.op
        else:
            self.op = Operator(matrix, device=local_rank)
        if os.environ.get("DMV_EXCHANGE"):
            self.op.set_option("exchange", int(os.environ["DMV_EXCHANGE"]))
        if os.environ.get("DMV_MODE"):
            self.op.set_option("mode", int(os.environ["DMV_MODE"]))
        self.op.basis.build()
        torch.cuda.synchronize()
        self.build_s = time.perf_counter() - t0
        self.n_local = self.op.basis.numberStates()
        self.op.use_torch_stream()
        # the whole sorted basis (for the recipe's x and for the oracle check); on one rank it is the local block
        if world > 1:
            g = Operator(matrix, device=local_rank)
            g.basis.build()
            self.reps_global = g.basis.representatives()
            g.close()
            from oracle import pyoracle as po
            self.local_rows = np.flatnonzero(po.locale_idx_of(self.reps_global, world) == rank)
        else:
            self.reps_global = self.op.basis.representatives()
            self.local_rows = np.arange(self.n_local)
        assert self.local_rows.shape[0] == self.n_local
        self.n_total = int(self.reps_global.shape[0])
        self.x_global = recipe_x(self.n_total, cplx)
        x_host = np.ascontiguousarray(self.x_global[self.local_rows])
        self.x_pinned = torch.from_numpy(x_host).pin_memory()
        self.y_pinned = torch.zeros_like(self.x_pinned).pin_memory()
        self.x_dev = self.x_pinned.cuda(non_blocking=True)
        self.y_dev = torch.zeros_like(self.x_dev)
        self.op.plan()
        self.nnz_local = self.op.numberTerms()

    def product(self):
        self.op.matvec(self.x_dev, self.y_dev)

    def exchange_name(self) -> str:
        if self.world == 1:
            return "none (one rank)"
        if self.op.info("replicated"):
            return "replicated x: peer-direct all-gather of x over NVLink + row traversal" if self.op.info("peer_gather") > 0 \
                else "replicated x: NCCL all-gather of x + row traversal"
        if self.op.info("rounds") > 1:
            return f"records: peer-direct NVLink stores from k_generate in {self.op.info('rounds')} overlapped rounds"
        if self.op.info("peer_direct"):
            return "records: peer-direct NVLink stores from k_generate"
        return "records: NCCL send/recv buckets"

    def kernel_name(self) -> str:
        if self.op.info("gather"):
            return "k_gather"
        if self.op.info("rows"):
            return "k_rows"
        if self.world > 1 and self.op.info("replicated"):
            return "k_pull"
        return "k_pull" if self.op.info("pull") else "k_generate"

    def check(self, sample_rows: int, threads: int) -> dict:
        """Sampled rows of the last product against the oracle (column-by-column recomputation)."""
        import torch
        from oracle import model as omodel
        from oracle import pyoracle as po
        torch.cuda.synchronize()
        self.y_dev.zero_()
        self.product()
        torch.cuda.synchronize()
        self.op.synchronize()
        y = self.y_dev.cpu().numpy()
        po.set_num_threads(max(1, threads))
        _, omatrix = omodel.load_model(os.path.join(ROOT, "data", self.name + ".yaml"))
        rng = np.random.default_rng(1234 + self.rank)
        k = min(sample_rows, self.n_local)
        pick = np.sort(rng.choice(self.n_local, size=k, replace=False))
        expect = po.expected_rows(omatrix, self.reps_global, self.x_global, self.local_rows[pick])
        got = y[pick]
        scale = max(float(np.abs(expect).max()), 1e-300)
        return {"rows": int(k), "max_abs_err": float(np.abs(got - expect).max()),
                "max_rel_err": float(np.abs(got - expect).max() / scale),
                "violations": criterion_violations(got, expect)}

    def close(self):
        self.op.close()


def time_products(w: Workload, steps: int, warmup: int, flush, barrier, dist, local_rank: int, sample_clocks: bool,
                  keep_last: bool = False):
    import torch
    from distributed_matvec_b200 import _native as nat
    for _ in range(max(warmup, 3)):
        flush.fill_(1)
        w.product()
    barrier()
    w.op.synchronize()
    launches0 = nat.lib().dmv_launch_count()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:
        sampler.__enter__()
    barrier()
    for k in range(steps):
        flush.fill_(k & 0xFF)
        if w.world > 1:
            dist.barrier()
        starts[k].record()
        w.product()
        ends[k].record()
    barrier()
    if sampler:
        sampler.__exit__()
    launches = nat.lib().dmv_launch_count() - launches0
    if keep_last:
        w.op.synchronize()
        w.y_last = w.y_dev.cpu().numpy()     # before the untimed products below overwrite y
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    t = torch.tensor([float(np.mean(step_ms)), float(np.min(step_ms))] + step_ms, dtype=torch.float64, device="cuda")
    if w.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    w.steps_ms = [round(float(v), 3) for v in t[2:]]          # every timed step, max over ranks
    w.op.synchronize()
    # dominant kernel: the generate stage of the library's own CUDA-event timeline
    kern, refill = [], []
    for k in range(min(steps, 5)):
        flush.fill_(k)
        torch.cuda.synchronize()
        w.product()
        torch.cuda.synchronize()
        tm = w.op.timings()
        kern.append(tm["generate(diag+offdiag+local accumulate)"])
        refill.append(tm.get("table refill (k_rows; part of generate)", 0.0))
    # k_rows: the generate stage is k_table_fill (values of the hash table, once per product) + k_rows; the roofline is
    # quoted on k_rows alone and the refill is reported beside it
    w.table_refill_ms = float(np.mean(refill)) if w.kernel_name() == "k_rows" else 0.0
    kernel_ms = float(np.mean(kern))
    if 0.0 < w.table_refill_ms < kernel_ms:
        kernel_ms -= w.table_refill_ms
    return float(t[0]), float(t[1]), kernel_ms, int(launches), (sampler.summary() if sampler else None)


def dump_outputs(w: Workload, out_dir: str, dist):
    """`--dump-outputs`: y of the last timed product at a fixed, seeded sample of DUMP_ROWS rows of the global sorted
    basis (every row when the basis is smaller), so that two builds can be compared output for output.  y.npy holds
    float64 values, shape (rows,) for f64 and (rows, 2) = (real, imag) for c128; y_rows.npy the row indices (float64)."""
    import torch
    n = w.n_total
    k = min(n, DUMP_ROWS)
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=k, replace=False))
    pos = np.minimum(np.searchsorted(rows, w.local_rows), k - 1)
    mine = rows[pos] == w.local_rows
    sample = np.zeros(k, dtype=w.y_last.dtype)
    sample[pos[mine]] = w.y_last[mine]
    if w.world > 1:      # every sampled row is owned by exactly one rank
        t = torch.from_numpy(sample.view(np.float64)).cuda()
        dist.all_reduce(t)
        sample = t.cpu().numpy().view(sample.dtype)
    if w.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        y = sample.view(np.float64)
        np.save(os.path.join(out_dir, "y.npy"), y.reshape(k, 2) if w.cplx else y)
        np.save(os.path.join(out_dir, "y_rows.npy"), rows.astype(np.float64))


def roofline_of(w: Workload, kernel_ms: float, clocks: dict | None, dtype: str) -> dict:
    peak, peak_kind = measured_peaks()
    bytes_alg = w.n_local * (8 + 2 * w.E) + w.nnz_local * (8 + 2 * w.E)
    achieved = bytes_alg / (kernel_ms * 1e-3) / 1e9
    kernel = w.kernel_name()
    const = ncu_constants(f"{kernel}:{w.name}:{dtype}") if w.world == 1 else None
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "traffic": const.get("dram_bytes") if const else None, "peak_kind": peak_kind, "kernel": kernel,
           "kernel_ms": kernel_ms, "table_refill_ms": getattr(w, "table_refill_ms", 0.0),
           "algorithmic_bytes": int(bytes_alg),
           "model": "SURVEY 8(d): N (8 + 2E) + nnz (8 + 2E) bytes per product"}
    limiter = {}
    if const:
        if const.get("dram_bytes"):
            limiter["dram_frac_of_peak"] = const["dram_bytes"] / (kernel_ms * 1e-3) / 1e9 / peak
            limiter["traffic_over_algorithmic"] = const["dram_bytes"] / bytes_alg
        if const.get("warp_instructions") and clocks and clocks.get("sm_mhz"):
            limiter["issue_slot_frac"] = const["warp_instructions"] / (kernel_ms * 1e-3 * 148 * 4 * clocks["sm_mhz"] * 1e6)
        limiter["source"] = const.get("source")
        for k in ("l1_wavefront_pct", "note"):
            if k in const:
                limiter[k] = const[k]
    if w.group_order > 1:
        limiter["group_order"] = w.group_order
        limiter["orbit_elements_per_s"] = (w.nnz_local + w.n_local) * w.group_order / (kernel_ms * 1e-3)
    out["limiter"] = limiter
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the product of the GPU arm; --impl reference times a slab of rows")
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cplx = args.dtype == "c128"
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    check_threads = max(1, host_threads() // world)

    w = Workload(args.workload, cplx, world, rank, local_rank)
    totals = torch.tensor([w.n_local, w.nnz_local], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(totals)
    n_total, nnz_total = int(totals[0]), int(totals[1])
    assert n_total == w.n_total

    ms_per_step, ms_best, kernel_ms, launches, clocks = time_products(w, args.steps, args.warmup, flush, barrier, dist,
                                                                     local_rank, True, keep_last=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(w, args.dump_outputs, dist)

    # ---- e2e: pinned host x -> public call -> host y; wall clock around the blocking call
    for _ in range(2):
        w.op.matvec(w.x_pinned.numpy(), w.y_pinned.numpy())
    barrier()
    e2e_times = []
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        barrier()
        t1 = time.perf_counter()
        w.op.matvec(w.x_pinned.numpy(), w.y_pinned.numpy())
        e2e_times.append(time.perf_counter() - t1)
    t = torch.tensor([1e3 * float(np.mean(e2e_times)), 1e3 * float(np.min(e2e_times))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms, e2e_best = float(t[0]), float(t[1])
    stage = w.op.timings()

    # ---- parity of this very configuration: sampled rows against the oracle, worst rank
    par = w.check(args.sample_rows, check_threads)
    pt = torch.tensor([par["max_abs_err"], par["max_rel_err"], float(par["violations"])], dtype=torch.float64, device="cuda")
    rows_checked = torch.tensor([par["rows"]], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(pt, op=dist.ReduceOp.MAX)
        dist.all_reduce(rows_checked)
    parity = {"max_abs_err": float(pt[0]), "max_rel_err": float(pt[1]), "violations_worst_rank": int(pt[2]),
              "rows_checked": int(rows_checked[0]), "against": "oracle_expected_rows (column-by-column, naive group)",
              "criterion": "|a-b| <= max(1e-14, 1e-12 max(|a|,|b|)) per element; max_rel_err = max|a-b| / max|b|"}

    line = {
        "metric": METRIC, "value": n_total / (ms_per_step * 1e-3), "unit": "states/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "c128" if cplx else "f64", "data": "synthetic",
        "config": {"workload": args.workload, "basis_states": n_total, "off_diag_terms": nnz_total, "x": X_RECIPE,
                   "l2": L2_NOTE},
        "run": {"terms_per_s": nnz_total / (ms_per_step * 1e-3), "partition": f"hash64_01 % {world}",
                "exchange": w.exchange_name(), "kernel": w.kernel_name(), "ms_best_step": ms_best,
                "steps_ms": w.steps_ms,
                "basis_build_s": w.build_s, "torus_mode": w.op.info("torus_mode"), "canon_mode": w.op.info("canon_mode")},
        "max_rel_err": parity["max_rel_err"], "parity": parity,
        "e2e": {"value": n_total / (e2e_ms * 1e-3), "unit": "states/s", "ms_per_step": e2e_ms, "ms_best_step": e2e_best,
                "h2d_bytes_per_step": int(w.n_local * w.E), "d2h_bytes_per_step": int(w.n_local * w.E),
                "stages_ms": stage},
        "gpu_launches": int(launches),
        "roofline": roofline_of(w, kernel_ms, clocks, args.dtype),
        "clocks": clocks,
    }

    # ---- CPU baseline (rank 0, one GPU only): the oracle port on a bounded slab of the same workload
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(args.workload, cplx, reps=w.reps_global)
        arm.calibrate(args.cpu_seconds / 4.0)
        times = [arm.step() for _ in range(3)]
        rows = arm.slab[1] - arm.slab[0]
        line["cpu_baseline"] = {"value": rows / min(times), "unit": "states/s", "cores": arm.threads, "kind": "port",
                                "sample": arm.sample_text() + f"; best of 3 ({1e3 * min(times):.0f} ms)",
                                **host_description()}
    main_name = args.workload
    w.close()
    del w

    # ---- the other BASELINE configs, briefly: value, kernel time and their own parity figure.  A watchdog keeps them
    # from costing the main line: if they are not through in time (a hung collective), every rank prints / exits.
    secondary = []
    line["secondary"] = secondary

    def give_up(signum, frame):
        secondary.append({"error": "secondary workloads timed out; entries above are complete"})
        if rank == 0:
            print(json.dumps(line), flush=True)
        os._exit(0)

    import signal
    signal.signal(signal.SIGALRM, give_up)
    signal.alarm(int(os.environ.get("DMV_SECONDARY_TIMEOUT", "420")))
    names = [] if args.secondary.strip().lower() in ("", "none") else [s for s in args.secondary.split(",") if s]
    for name in names:
        if name == main_name:
            continue
        try:
            s = Workload(name, cplx, world, rank, local_rank)
            ms, best, kms, _, _ = time_products(s, 5, 3, flush, barrier, dist, local_rank, False)
            sp = s.check(min(args.sample_rows, 1024), check_threads)
            st = torch.tensor([sp["max_rel_err"], float(sp["violations"])], dtype=torch.float64, device="cuda")
            tot = torch.tensor([s.n_local, s.nnz_local], dtype=torch.int64, device="cuda")
            if world > 1:
                dist.all_reduce(st, op=dist.ReduceOp.MAX)
                dist.all_reduce(tot)
            secondary.append({"workload": name, "basis_states": int(tot[0]), "off_diag_terms": int(tot[1]),
                              "value": int(tot[0]) / (ms * 1e-3), "ms_per_step": ms, "ms_best_step": best,
                              "kernel": s.kernel_name(), "kernel_ms": kms, "exchange": s.exchange_name(),
                              "max_rel_err": float(st[0]), "violations_worst_rank": int(st[1]),
                              "basis_build_s": s.build_s})
            s.close()
            del s
        except Exception as e:   # a secondary entry must not cost the main line
            secondary.append({"workload": name, "error": f"{type(e).__name__}: {e}"[:300]})
    signal.alarm(0)

    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
