#!/usr/bin/env python3
"""bench.py -- pod-fit decisions/s of the autoscaler tick on B200 (driver contract, see DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|small]
                    [--dump-outputs DIR]

A "step" is one whole tick of the hot path over one synthetic snapshot (SURVEY.md section 8d):
    occupancy (K1) + get_pods_to_schedule (K0) + get_pending_pods (first-fit pipeline over nodes)
    + fulfill_pending (first-fit pipeline over bins, pool arithmetic) + maintain (idle scan K6, actions).
`value` = decisions / s with the snapshot resident in HBM; `e2e` = the same through the host-buffer plugin calls
(pinned host arrays, H2D + D2H inside the timed region).  A *decision* is one evaluation the reference itself
performs of KubeNode.can_fit (kube.py:173) or of a `(x - pod.resources).possible` pool/bin test
(scaler.py:134,139, capacity.py:30); the count is checked against the oracle's count in the parity tests.

N = 1 (the driver's BENCH line): headline = BASELINE.json configs[1] (c2: 100k pending pods x 10k nodes x 4 dims x
1 pool); `configs.c3` and `configs.c5` carry the larger single-GPU configurations (1M x 100k x 8 x 8; the
idle-node scan over 1M nodes) measured in the same run, each with value / e2e / roofline.
N > 1 (torchrun, one rank per GPU): ONE cluster -- c3 -- on all ranks in cluster mode (include/acsfit.h): strong
scaling; the result is asserted equal, bit for bit, to the single-GPU result of the same snapshot computed in the
same run, whose time is reported next to it (`strong_scaling`).  `configs.c4` (10M x 1M, N = 8) and the former
weak-scaling "fleet" measurement are secondary keys.

--dump-outputs DIR writes what the last timed step of the headline tick returned, as DIR/<name>.npy in float64
(see dump_outputs), so that two builds can be compared output for output on the same seeded snapshot.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (P, N, D, T)
    "small": (20000, 2000, 4, 1),
    "c2": (100000, 10000, 4, 1),          # BASELINE.json configs[1] -- the metric's config
    "c3": (1000000, 100000, 8, 8),        # configs[2]
    "c4": (10000000, 1000000, 8, 8),      # configs[3]: one cluster on 8 GPUs
}
C5_NODES = 1000000                         # configs[4]: idle-node scan, ~10 running pods per node, 8 thresholds
C5_THRESHOLDS = [60, 300, 900, 1800, 3600, 7200, 21600, 86400]
METRIC = "pod-fit decisions/sec"
UNIT = "decisions/s"
SEED = 20260921 + 2
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_SEED = 20260921


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """samples SM clocks / throttle reasons during the timed region: in-process through NVML (nvidia-ml-py), so that
    no process is spawned beside the timed loop; the nvidia-smi command line is the fallback."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.samples = []  # (sm_mhz, sm_max_mhz, [reason flags])
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))  # static: read once
            self._bits = [getattr(pynvml, n, 0) for n in ("nvmlClocksThrottleReasonHwSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown",
                                                          "nvmlClocksThrottleReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwPowerCap")]
        except Exception:
            self._nvml = None
        try:  # one throw-away reading now: the first query of a process initialises driver paths (measured: a 7.7 ms
            self._sample()  # stall of the concurrently running tick when it happened inside the timed region)
        except Exception:
            pass

    def _sample(self):
        if self._nvml is not None:
            n = self._nvml
            sm = n.nvmlDeviceGetClockInfo(self._handle, n.NVML_CLOCK_SM)
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle)
            return (int(sm), self._max_mhz, [bool(mask & b) for b in self._bits])
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) < 6:
            return None
        return (int(float(parts[0])), int(float(parts[1])), [p.lower().startswith("active") for p in parts[2:6]])

    def _run(self):
        # Every NVML query takes driver locks that the tick's own launches and copies need: measured on the B200 box, a
        # 50 ms period put a 10-24 ms outlier into about one c2 step in twenty, a 1 s period none.  So: a first sample
        # shortly after the timed region starts (the GPU is under load since the warm-up), then four per second.
        if self._stop.wait(0.02):
            return
        while not self._stop.is_set():
            try:
                s = self._sample()
                if s:
                    self.samples.append(s)
            except Exception:
                pass
            self._stop.wait(float(os.environ.get("ACSFIT_BENCH_SAMPLE_PERIOD", 0.25)))

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(s[0] for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[2][i] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self._nvml is not None else "nvidia-smi"}


def algorithmic_bytes(decisions, P, N, D):
    """SURVEY.md 8(d): 8*D bytes per decision (the node / bin row the reference touches) plus the
    compulsory P*(8D+4) + N*(16D+4) once per tick."""
    return decisions * 8 * D + P * (8 * D + 4) + N * (16 * D + 4)


def idle_bytes(R, N, D, S):
    """SURVEY.md 8(d), idle scan on a contiguous table: R(8D+1) rows + flag bytes, 8(N+1) row pointers,
    N(4+8+1) node type / age / flags (capacity rows are per TYPE: negligible), S*N states written."""
    return R * (8 * D + 1) + 8 * (N + 1) + N * (4 + 8 + 1) + S * N


def occupancy_bytes(R, N, D):
    return R * 8 * D + 8 * (N + 1) + N * 16 * D


def ncu_traffic(name):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this round
    (profiles/r02_traffic.json, written by tools/summarise_profiles.py from the .ncu-rep), or None."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(name)
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
# CPU arms: the plain-C oracle port, and the reference's own CPython loop (oracle/_ref)
# ---------------------------------------------------------------------------------------------
def oracle_tick(oracle, c):
    used = np.zeros((c["N"], c["D"]), dtype=np.float64)
    oracle.occupancy(c["row_ptr"], c["run_idx"], c["req_run"], used)
    mask, ev0 = oracle.feasible_mask(c["req"], c["unit_all"])
    feas = c["req"][mask.astype(bool)]
    placed, ev1 = oracle.first_fit_nodes(feas, c["cap_type"], c["node_type"], used)
    pend = feas[placed < 0]
    ev2 = 0
    if len(pend):
        r = oracle.fulfill_pending(pend, len(pend), c["unit_ordered"], c["pool_actual"], c["pool_max"],
                                   c["pool_ignored"], c["over_provision"])
        ev2 = r["evals"]
    st = oracle.node_states(c["row_ptr"], c["run_idx"], c["req_run"], c["flags_run"], c["cap_type"], c["node_type"],
                            c["node_flags"], c["node_age"], len(feas) > 0, [1800])[0]
    budget = c["pool_actual"].astype(np.int64) - 1
    oracle.maintain_actions(st, c["node_pool"], budget, np.ones(c["T"], np.uint8), True)
    return ev0 + ev1 + ev2


def time_oracle(c, steps, warmup):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    oracle.build()
    times, decisions = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        decisions = oracle_tick(oracle, c)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return decisions, times


def python_reference(shapes):
    """the unmodified reference (staged in oracle/_ref by oracle/build_ref.py) on scaled-down shapes of the c2
    generator, BASELINE.md section 3; None when the staged copy is not there."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_shim
        if not ref_shim.available():
            return None
        import ref_bench
        return ref_bench.time_reference(shapes=shapes, seed=SEED)
    except Exception as e:  # never let the baseline leg take the GPU line down
        return {"error": "%s: %s" % (type(e).__name__, e)}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores.  The
    reference is pure Python; its unmodified files are staged in oracle/_ref (oracle/build_ref.py) and imported
    under oracle/ref_shim.py.  Each step is a bounded sample of the workload -- 2000 pods x 200 nodes of the
    same generator (decisions/s is size-independent for the reference, BASELINE.md section 2) -- run
    single-threaded: CPython holds the GIL and first fit is order-dependent.  Falls back to the plain-C port
    (oracle/acsfit_oracle.c) when the staged copy is missing; the port's figure is reported either way."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
    name = args.config if args.gpus == 1 else "c3"
    P, N, D, T = CONFIGS[name]
    steps, warmup = args.steps, args.warmup
    # the C port on a bounded sample of the same workload (full c2; c3 scaled to 1/8 of the pods and nodes)
    Ps, Ns = (P, N) if P * N <= 2 * 10 ** 9 else (P // 8, N // 8)
    cs = syn.make_cluster(Ps, Ns, D, T, seed=SEED)
    dec_port, t_port = time_oracle(cs, 1, 0)
    port = {"value": dec_port / t_port[0], "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%s tick at %d pods x %d nodes, plain-C port of the reference loops (oracle/acsfit_oracle.c), "
                      "1 of %d host cores" % (name, Ps, Ns, os.cpu_count())}
    values, ref = [], None
    for i in range(warmup + steps):
        ref = python_reference(((2000, 200),))
        if not ref or "error" in ref:
            break
        if i >= warmup:
            values.append(ref["value"])
    if values:
        value = float(np.mean(values))
        shape = ref["shapes"][0]
        base = {"value": value, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": "the unmodified reference (oracle/_ref, CPython %s, 1 of %d host cores, %s): "
                          "get_pods_to_schedule + get_pending_pods + fulfill_pending on 2000 pods x 200 nodes of the "
                          "%s generator, %d timed step(s); results checked against the C port: %s"
                          % (ref["python"], os.cpu_count(), cpu_model(), name, steps, shape["matches_oracle"]),
                "port": port}
        ms = shape["seconds"] * 1e3
    else:
        value, base, ms = port["value"], dict(port, python=ref), t_port[0] * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if args.gpus == 1 else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(name, P, N, D, T, args.gpus), "bounded_sample": base["sample"]},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_name(name, P, N, D, T, world):
    s = "%s: %d pending pods x %d nodes x %d dims x %d pool(s)" % (name, P, N, D, T)
    return s if world == 1 else s + ", one cluster"


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
class Workload(object):
    """one synthetic snapshot resident on one GPU + pinned host copies, and the two forms of the tick."""

    def __init__(self, eng, c, pinned=True):
        import torch
        self.eng, self.c = eng, c
        i64, i32, f64, u8 = torch.int64, torch.int32, torch.float64, torch.uint8
        self.d = {"req": eng.dev(c["req"], f64), "cap_type": eng.dev(c["cap_type"], f64),
                  "node_type": eng.dev(c["node_type"], i32), "row_ptr": eng.dev(c["row_ptr"], i64),
                  "run_idx": None,  # the synthetic table is contiguous (run_idx = arange): bulk-copy K1 / K6
                  "req_run": eng.dev(c["req_run"], f64),
                  "flags_run": eng.dev(c["flags_run"], u8), "node_flags": eng.dev(c["node_flags"], u8),
                  "node_age": eng.dev(c["node_age"], i64), "node_pool": eng.dev(c["node_pool"], i32)}
        self.used = torch.zeros((c["N"], c["D"]), dtype=f64, device=eng.device)
        self.budget = c["pool_actual"].astype(np.int64) - 1
        self.scalable = np.ones(c["T"], np.uint8)
        self.thr = np.array([1800], np.int64)
        self.h = None
        if pinned:
            def pin(a):
                return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
            assert np.array_equal(c["run_idx"], np.arange(len(c["run_idx"])))
            self.h = {k: pin(c[k]) for k in ("req", "cap_type", "node_type", "row_ptr", "req_run",
                                             "flags_run", "node_flags", "node_age", "node_pool")}
            self.h["run_idx"] = None
            self.h_used = pin(np.zeros((c["N"], c["D"])))
            P = c["P"]
            self.h_out = {"feasible": pin(np.empty(P, np.uint8)), "placed": pin(np.empty(P, np.int32)),
                          "acc_pool": pin(np.empty(P, np.int32))}
            R = c["req_run"].shape[0]
            csr = c["row_ptr"].nbytes + c["req_run"].nbytes
            self.h2d = (csr + self.h_used.nbytes                                                   # occupancy_host
                        + c["req"].nbytes + c["cap_type"].nbytes + c["node_type"].nbytes + self.h_used.nbytes  # scale_up_host
                        + csr + c["flags_run"].nbytes + c["cap_type"].nbytes + c["node_type"].nbytes
                        + c["node_flags"].nbytes + c["node_age"].nbytes + c["node_pool"].nbytes + 8)          # maintain_host
            self.d2h = self.h_used.nbytes + P * (1 + 4 + 4) + self.h_used.nbytes + 2 * c["N"]
            del R

    def pool_args(self):
        c = self.c
        return (c["unit_all"], c["unit_ordered"], c["pool_actual"], c["pool_max"], c["pool_ignored"], c["over_provision"])

    def step_device(self):
        eng, d = self.eng, self.d
        self.used.zero_()
        eng.occupancy(d["row_ptr"], d["run_idx"], d["req_run"], self.used)                       # row E (K1)
        r = eng.scale_up(d["req"], *self.pool_args(), d["cap_type"], d["node_type"], self.used)  # rows F0, F1, F
        st = eng.node_states(d["row_ptr"], d["run_idx"], d["req_run"], d["flags_run"], d["cap_type"], d["node_type"],
                             d["node_flags"], d["node_age"], r["n_to_schedule"] > 0, self.thr)   # row I (K6)
        self.last_maintain = eng.maintain_actions(st[0], d["node_pool"], self.budget, self.scalable, True)  # row J
        return r

    def outputs(self, r):
        """what a caller of step_device receives from the step that returned `r` (host copies)."""
        state, action = self.last_maintain
        out = {k: r[k].cpu().numpy() for k in ("feasible", "placed", "acc_pool")}
        out.update({k: r[k] for k in ("new_size", "units_needed", "bins_opened")})
        out.update({k: np.array([r[k]]) for k in ("n_to_schedule", "n_pending", "num_unaccounted", "decisions")})
        out.update({"used": self.used.cpu().numpy(), "node_state": state.cpu().numpy(), "node_action": action.cpu().numpy()})
        return out

    def step_host(self):
        eng, h = self.eng, self.h
        self.h_used.fill(0.0)
        eng.occupancy_host(h["row_ptr"], h["run_idx"], h["req_run"], self.h_used)
        r = eng.scale_up_host(h["req"], *self.pool_args(), h["cap_type"], h["node_type"], self.h_used, out=self.h_out)
        eng.maintain_host(h["row_ptr"], h["run_idx"], h["req_run"], h["flags_run"], h["cap_type"], h["node_type"],
                          h["node_flags"], h["node_age"], h["node_pool"], r["n_to_schedule"] > 0, 1800, self.budget,
                          self.scalable, True)
        return r

    def pipeline_leg(self, flush, reps):
        """the dominant kernel (first-fit pipeline launches) bracketed by CUDA events inside the library"""
        import torch
        eng, d, c = self.eng, self.d, self.c
        eng.set_timing(True)
        ms, dec, byt = 0.0, 0, 0
        for _ in range(reps):
            flush.fill_(1)
            self.used.zero_()
            eng.occupancy(d["row_ptr"], d["run_idx"], d["req_run"], self.used)
            torch.cuda.synchronize()
            r = eng.scale_up(d["req"], *self.pool_args(), d["cap_type"], d["node_type"], self.used)
            s = eng.pipeline_stats()
            ms += s["ms"]
            dec += s["decisions"]
            byt += algorithmic_bytes(s["decisions"], c["P"], c["N"] + int(r["bins_opened"].sum()), c["D"])
        eng.set_timing(False)
        return ms / reps, dec / reps, byt / reps


def dump_outputs(directory, arrays):
    """write each array as <directory>/<name>.npy in float64 (exact for the int32 / int64 counts and uint8 codes
    the tick returns).  Should the whole exceed DUMP_LIMIT_BYTES, arrays are cut along their first axis to one fixed,
    seeded sample of rows (the same rows for every array of the same length), and the row numbers are written as
    <name>_rows.npy.  Arrays of at most 65536 rows (pool sizes, counts) are always written whole."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    big = [k for k, a in arrays.items() if a.ndim and a.shape[0] > 65536]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        small = total - sum(arrays[k].nbytes for k in big)
        keep = (DUMP_LIMIT_BYTES - small) / (2.0 * (total - small))  # half of what is left: room for the row numbers
        for name in big:
            a = arrays[name]
            rows = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(a.shape[0], int(a.shape[0] * keep), replace=False))
            arrays[name], arrays[name + "_rows"] = a[rows], rows.astype(np.float64)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


LAST_STEP_MS = []


MIN_WARM_SECONDS = 0.25


def timed(step_fn, steps, warmup, flush, barrier, launch_count, min_warm_seconds=0.0):
    import torch
    # W untimed steps, and (single-process runs: min_warm_seconds > 0) at least that long: the per-step list of the
    # round-2 runs shows the first one or two timed steps slower than the rest (8.9-9.0 against 8.7 ms, once 16 ms)
    # when the SM clock is still ramping up from idle after only ~30 ms of load.  (Never time-based under torchrun:
    # cluster-mode ticks are collective, every rank must run the same number of them.)
    t_warm = time.perf_counter()
    n_warm = 0
    while n_warm < warmup or (warmup > 0 and time.perf_counter() - t_warm < min_warm_seconds):
        step_fn()
        n_warm += 1
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    # CPython's cyclic GC is paused over the timed steps (as Cluster.loop_logic pauses it over a tick): a generation-2
    # pass over the interpreter's ~10^6 objects (torch is imported) takes 10-30 ms and lands inside some step, between two
    # launches of the tick - measured as one c3 step in eight at 187 instead of 154 ms.
    import gc
    gc.collect()
    gc_was_on = gc.isenabled()
    gc.disable()
    try:
        barrier()
        l0 = launch_count()
        res = None
        for a, b in ev:
            flush.fill_(1)  # evict L2 between timed iterations
            torch.cuda.synchronize()
            a.record()
            res = step_fn()
            b.record()
        barrier()
    finally:
        if gc_was_on:
            gc.enable()
    global LAST_STEP_MS
    LAST_STEP_MS = [a.elapsed_time(b) for a, b in ev]
    return res, sum(LAST_STEP_MS), launch_count() - l0


INT_LANE_OPS_PER_CLK_SM = 77.0  # measured: tools/ubench6.cu, profiles/r02b_ubench6.txt (IADD + LOP3 mix, all SMs busy)


def physical_roofline(kernel_dec_per_s, nw, sm_mhz, kernel_ms=None, placements=None, sms=148):
    """what actually bounds the pipeline.  (1) The candidate scan is integer-issue work: a pair costs 2 ops per packed
    word + 1 compare (acsfit_kernels.cuh) at the measured int32 issue rate; credited decisions ~ pairs tested.
    (2) Below that ceiling sits the sequential placement chain: first fit is a recurrence, every placement waits for
    the previous one on the frontier warp (DESIGN.md section 6) -- reported as kernel time per placement."""
    if not sm_mhz:
        return None
    out = {"achieved": kernel_dec_per_s, "unit": UNIT}
    if nw:
        ops = 2 * nw + 1
        out["limiter"] = ("the sequential placement chain (see chain_ns_per_placement; a placing step costs ~77 cycles in the "
                          "frontier warp's loop plus per-batch and per-tile work, and nothing else can proceed past it); the scan's own ceiling is int32 "
                          "issue: %d ops per pair at %d packed word(s) per row" % (ops, nw))
        out["ceiling"] = sms * INT_LANE_OPS_PER_CLK_SM * sm_mhz * 1e6 / ops
        out["frac"] = kernel_dec_per_s / out["ceiling"]
        out["source"] = "tools/ubench6.cu: %.0f int32 lane-ops/clk/SM (profiles/r02b_ubench6.txt) x SM clock under load" % INT_LANE_OPS_PER_CLK_SM
    else:
        out["limiter"] = "fp64 compare issue (float64 scan: D DSETP per pair, ~45 lane-ops/clk/SM, tools/ubench5.cu) and the placement chain"
    if kernel_ms and placements:
        out["chain_ns_per_placement"] = kernel_ms * 1e6 / placements
        out["placements_per_step"] = int(placements)
    return out


def sub_record_c3(eng, syn, flush, steps, peak):
    import torch
    P, N, D, T = CONFIGS["c3"]
    c = syn.make_cluster(P, N, D, T, seed=SEED)
    w = Workload(eng, c)
    nb = lambda: torch.cuda.synchronize()  # noqa: E731
    res, dev_ms, _ = timed(w.step_device, steps, 2, flush, nb, lambda: eng.launch_count, MIN_WARM_SECONDS)
    res_h, host_ms, _ = timed(w.step_host, steps, 1, flush, nb, lambda: eng.launch_count, MIN_WARM_SECONDS)
    assert res_h["decisions"] == res["decisions"]
    k_ms, k_dec, k_bytes = w.pipeline_leg(flush, min(steps, 3))
    achieved = k_bytes / (k_ms * 1e-3) / 1e9
    return {"workload": workload_name("c3", P, N, D, T, 1), "steps": steps, "ms_per_step": dev_ms / steps,
            "value": res["decisions"] * steps / (dev_ms * 1e-3), "unit": UNIT,
            "decisions_per_step": int(res["decisions"]), "pending": res["n_pending"],
            "bins_opened": [int(x) for x in res["bins_opened"]],
            "pods_per_s": P / (dev_ms / steps * 1e-3),
            "e2e": {"value": res["decisions"] * steps / (host_ms * 1e-3), "unit": UNIT, "ms_per_step": host_ms / steps,
                    "h2d_bytes_per_step": int(w.h2d), "d2h_bytes_per_step": int(w.d2h)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic("pipeline_c3"), "kernel_ms_per_step": k_ms,
                         "kernel_decisions_per_s": k_dec / (k_ms * 1e-3),
                         "note": "SURVEY 8(d) bytes (64 per decision at D = 8) over the pipeline's kernel time; rows "
                                 "stay on chip, so this exceeds the HBM peak -- see physical"}}, k_dec / (k_ms * 1e-3)


def sub_record_c5(eng, syn, flush, peak):
    """BASELINE configs[4]: node states for 1M nodes x 8 idle thresholds (K6) and the occupancy sums (K1),
    each timed alone with CUDA events (cold L2: flushed before every launch)."""
    import torch
    i64, i32, f64, u8 = torch.int64, torch.int32, torch.float64, torch.uint8
    out = {}
    for D in (4, 8):
        c = syn.make_idle_cluster(C5_NODES, D=D, T=1 if D == 4 else 8, seed=SEED + 3)
        R, N = c["req_run"].shape[0], c["N"]
        d = {k: eng.dev(c[k], t) for k, t in (("row_ptr", i64), ("req_run", f64), ("flags_run", u8),
                                              ("cap_type", f64), ("node_type", i32), ("node_flags", u8), ("node_age", i64))}
        d["run_idx"] = None  # contiguous table
        used = torch.zeros((N, D), dtype=f64, device=eng.device)
        thr = np.array(C5_THRESHOLDS, np.int64)

        def best_of(fn, reps=7):
            ts = []
            for _ in range(reps):
                flush.fill_(1)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            return float(np.median(ts))
        k6 = best_of(lambda: eng.node_states(d["row_ptr"], d["run_idx"], d["req_run"], d["flags_run"], d["cap_type"],
                                             d["node_type"], d["node_flags"], d["node_age"], False, thr))
        k1 = best_of(lambda: eng.occupancy(d["row_ptr"], d["run_idx"], d["req_run"], used))
        b6, b1 = idle_bytes(R, N, D, len(C5_THRESHOLDS)), occupancy_bytes(R, N, D)
        out["D%d" % D] = {
            "running_pods": int(R),
            "node_states": {"ms": k6, "nodes_per_s": N / (k6 * 1e-3), "algorithmic_bytes": int(b6),
                            "roofline": {"bound": "hbm", "achieved": b6 / (k6 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                         "frac": b6 / (k6 * 1e-3) / 1e9 / peak, "traffic": ncu_traffic("k6_D%d" % D)}},
            "occupancy": {"ms": k1, "algorithmic_bytes": int(b1),
                          "roofline": {"bound": "hbm", "achieved": b1 / (k1 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                       "frac": b1 / (k1 * 1e-3) / 1e9 / peak, "traffic": ncu_traffic("k1_D%d" % D)}},
            "timing": "CUDA events around the Python call (includes the launch and, for node_states, the thresholds' "
                      "H2D); the ncu kernel durations are in profiles/r02_summary.md"}
    out["workload"] = "c5: idle-node scan, %d nodes x ~10 running pods, %d idle thresholds" % (C5_NODES, len(C5_THRESHOLDS))
    return out


def python_surface(eng, syn, c, reps=3):
    """the tick through the reference's own entry point: Cluster.loop_logic (alias scale_loop) fed kube-API style
    dicts for every node and pod of the snapshot -- object construction, flattening, the GPU path and the log /
    hand-off code all inside the timed region (SURVEY.md section 8(f)1: host-side ingestion)."""
    import logging
    from kubernetes_acs_engine_autoscaler_b200 import agent_pool, snapshot
    from kubernetes_acs_engine_autoscaler_b200.cluster import Cluster

    class Obj(object):
        __slots__ = ("obj",)

        def __init__(self, o):
            self.obj = o

        @property
        def name(self):
            return self.obj["metadata"]["name"]
    st = syn.kube_objects(c)
    nodes, pods = [Obj(o) for o in st["nodes"]], [Obj(o) for o in st["pods"]]
    cl = Cluster(None, 1800, 1, "a", "b", "c", "d", "e", "f", 600, "rg", None, "", over_provision=c["over_provision"], dry_run=True)
    cl.list_nodes, cl.list_pods = (lambda: nodes), (lambda: pods)
    cl.arm_template, cl.arm_parameters = {}, st["arm_parameters"]
    calls = []
    orig_init = agent_pool.AgentPool.__init__

    def pool_init(self, *a, **k):  # AgentPool.max_size is a plain attribute (100 upstream): the benchmark pools are unbounded
        orig_init(self, *a, **k)
        self.max_size = int(c["pool_max"][0])
    agent_pool.AgentPool.__init__ = pool_init
    prev_engine = snapshot._engine
    snapshot.set_engine(eng)
    logging.disable(logging.CRITICAL)
    try:
        times = []
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            ok = cl.loop_logic()
            times.append(time.perf_counter() - t0)
            calls.append(ok)
    finally:
        logging.disable(logging.NOTSET)
        agent_pool.AgentPool.__init__ = orig_init
        snapshot._engine = prev_engine
    best = min(times[1:])
    return {"seconds_per_tick": best, "pods": len(pods), "nodes": len(nodes), "returned": bool(calls[-1]),
            "pods_per_s": len(pods) / best,
            "what": "Cluster.loop_logic(), dry run, on kube-style dicts of the c2 snapshot (best of %d after one warm-up): "
                    "KubePod / KubeNode construction, flattening, GPU tick, decisions mapped back" % reps}


def run_single(args):
    import torch
    from kubernetes_acs_engine_autoscaler_b200 import build as acs_build
    from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
    from kubernetes_acs_engine_autoscaler_b200.engine import Engine
    torch.cuda.set_device(0)
    acs_build.build()
    eng = Engine(0)
    P, N, D, T = CONFIGS[args.config]
    c = syn.make_cluster(P, N, D, T, seed=SEED)
    w = Workload(eng, c)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)  # > 126 MB L2
    nb = lambda: torch.cuda.synchronize()  # noqa: E731
    peak, peak_src = load_peaks()
    with ClockSampler(0) as clocks:
        res, dev_ms, launches = timed(w.step_device, args.steps, args.warmup, flush, nb, lambda: eng.launch_count, MIN_WARM_SECONDS)
        step_ms, steps_in_order = sorted(LAST_STEP_MS), [round(x, 3) for x in LAST_STEP_MS]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, w.outputs(res))
        res_h, host_ms, _ = timed(w.step_host, args.steps, max(1, args.warmup // 2), flush, nb, lambda: eng.launch_count, MIN_WARM_SECONDS)
    assert res_h["decisions"] == res["decisions"]
    k_ms, k_dec, k_bytes = w.pipeline_leg(flush, max(1, min(args.steps, 5)))
    stats = eng.pipeline_stats()
    clk = clocks.summary()
    achieved = k_bytes / (k_ms * 1e-3) / 1e9
    nw = {4: 1, 8: 1}.get(D, 1)  # the synthetic request tables fit one packed word (tests/test_rank_math_cpu.py)
    if os.environ.get("ACSFIT_RANKS") == "0":
        nw = 0
    value = res["decisions"] * args.steps / (dev_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "ms_per_step_spread": {"min": step_ms[0], "median": step_ms[len(step_ms) // 2], "max": step_ms[-1]},
        "ms_steps": steps_in_order,  # every timed step, in order (value / ms_per_step are their mean)
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.config, P, N, D, T, 1), "seed": SEED,
                   "decisions_per_step": int(res["decisions"]), "pods_to_schedule": res["n_to_schedule"],
                   "pending": res["n_pending"], "bins_opened": [int(x) for x in res["bins_opened"]],
                   "tick": "occupancy (K1) + scale_up (K0, nodes pass, bin passes) + node_states (K6) + maintain",
                   "l2": "flushed between timed iterations (256 MiB fill)", "python_gc": "paused over the timed steps",
                   "warm_up": "W untimed steps, continued until %.2f s have passed (SM clock settled)" % MIN_WARM_SECONDS,
                   "parallelism": "1 rank"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic("pipeline_%s" % args.config), "peak_source": peak_src,
                     "kernel": "firstfit_pipeline_kernel (nodes + bins launches)", "kernel_ms_per_step": k_ms,
                     "kernel_decisions_per_s": k_dec / (k_ms * 1e-3),
                     "note": "achieved = SURVEY 8(d) algorithmic bytes (8*D per decision) / kernel time; node and bin "
                             "rows are held on chip, so real DRAM traffic (`traffic`, ncu) is far below it: the "
                             "kernel is not HBM-bound, `physical` names what does bound it",
                     "physical": physical_roofline(k_dec / (k_ms * 1e-3), nw, clk.get("sm_mhz"), k_ms, res["n_to_schedule"])},
        "e2e": {"value": res["decisions"] * args.steps / (host_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(w.h2d),
                "d2h_bytes_per_step": int(w.d2h), "ms_per_step": host_ms / args.steps,
                "path": "acsfit_occupancy_host + acsfit_scale_up_host + acsfit_maintain_host on pinned host arrays"},
        "gpu_launches": int(launches),
        "clocks": clk,
        "pipeline": {"stages": stats["stages"], "tiles": stats["tiles"]},
        "pods_per_s": P / (dev_ms / args.steps * 1e-3),
    }
    if not args.no_sub:
        configs = {}
        try:
            if args.config != "c3":
                configs["c3"], c3_rate = sub_record_c3(eng, syn, flush, max(1, min(args.steps, 3)), peak)
                configs["c3"]["roofline"]["physical"] = physical_roofline(
                    c3_rate, 0 if nw == 0 else 1, clk.get("sm_mhz"), configs["c3"]["roofline"]["kernel_ms_per_step"], CONFIGS["c3"][0])
            configs["c5"] = sub_record_c5(eng, syn, flush, peak)
            if args.config == "c2":
                line["e2e"]["python_surface"] = python_surface(eng, syn, c)
        except Exception as e:  # a sub-record must never take the headline down
            configs["error"] = "%s: %s" % (type(e).__name__, e)
        line["configs"] = configs
    if not args.no_cpu_baseline:
        if P * N <= 2 * 10 ** 9:
            decisions, times = time_oracle(c, 1, 0)
            assert decisions == res["decisions"], (decisions, res["decisions"])
            sample = "the full %s tick once (%.1f s)" % (args.config, times[0])
        else:  # bounded sample: the same generator at 1/8 of the pods and nodes (decisions/s is size-stable)
            cs = syn.make_cluster(P // 8, N // 8, D, T, seed=SEED)
            decisions, times = time_oracle(cs, 1, 0)
            sample = "%s scaled to %d pods x %d nodes (%.1f s)" % (args.config, P // 8, N // 8, times[0])
        line["cpu_baseline"] = {"value": decisions / times[0], "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": sample + " on 1 of %d host cores (%s), plain-C port of the reference loops"
                                          % (os.cpu_count(), cpu_model()),
                                "python": python_reference(((1000, 100), (2000, 200), (4000, 400)))}
    print(json.dumps(line))


def run_cluster(args):
    """N > 1: one cluster on all ranks (cluster mode), strong scaling."""
    import torch
    import torch.distributed as dist
    from kubernetes_acs_engine_autoscaler_b200 import build as acs_build
    from kubernetes_acs_engine_autoscaler_b200 import distributed as acs_dist
    from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
    from kubernetes_acs_engine_autoscaler_b200.engine import Engine
    rank, world, local_rank = acs_dist.env_rank()
    torch.cuda.set_device(local_rank)
    acs_dist.init("nccl")
    if rank == 0:
        acs_build.build()
    acs_dist.barrier()
    name = args.config if args.config in ("c3", "small") else "c3"
    P, N, D, T = CONFIGS[name]
    run_c4 = not args.no_c4  # configs[3] (10M x 1M): the shape where the scan outweighs the placement chain
    Pmax, Nmax = (CONFIGS["c4"][0], CONFIGS["c4"][1]) if run_c4 else (P, N)
    eng = Engine(local_rank)
    eng.cluster_connect(max_pods=Pmax, max_nodes=Nmax, max_dims=8)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    peak, peak_src = load_peaks()

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def counts_agree(r, c):
        """the north-star's single NCCL all-reduce of the per-pool integer counts: every rank computed the whole
        answer, so MIN and MAX over the ranks must both equal it"""
        v = np.concatenate([np.asarray(r["new_size"], np.int64) - c["pool_actual"].astype(np.int64),
                            np.array([r["n_to_schedule"], r["n_pending"], r["num_unaccounted"], r["decisions"]], np.int64)])
        t = torch.from_numpy(np.concatenate([v, -v])).to(eng.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.cpu().numpy()
        assert np.array_equal(t[:len(v)], v) and np.array_equal(-t[len(v):], v), "ranks disagree on the pool counts"

    def measure(cname, steps, warmup, verify=True, solo_steps=2, dump_dir=None):
        Pc, Nc, Dc, Tc = CONFIGS[cname]
        c = syn.make_cluster(Pc, Nc, Dc, Tc, seed=SEED)  # identical on every rank
        w = Workload(eng, c, pinned=(cname != "c4"))

        def step():
            r = w.step_device()
            counts_agree(r, c)
            return r
        res, dev_ms, launches = timed(step, steps, warmup, flush, barrier, lambda: eng.launch_count)
        if dump_dir and rank == 0:  # every rank holds the whole (replicated) result
            dump_outputs(dump_dir, w.outputs(res))
        plan = eng.cluster_last_plan()
        host_ms = None
        if w.h is not None:
            def step_h():
                r = w.step_host()
                counts_agree(r, c)
                return r
            res_h, host_ms, _ = timed(step_h, steps, 1, flush, barrier, lambda: eng.launch_count)
            assert res_h["decisions"] == res["decisions"]
        k_ms, k_dec, k_bytes = w.pipeline_leg(flush, 1)
        t = torch.tensor([dev_ms, host_ms or 0.0, k_ms], dtype=torch.float64, device=eng.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, host_ms2, k_ms = float(t[0]), float(t[1]), float(t[2])
        rec = {"workload": workload_name(cname, Pc, Nc, Dc, Tc, world), "steps": steps, "warmup": warmup,
               "ms_per_step": dev_ms / steps, "value": res["decisions"] * steps / (dev_ms * 1e-3), "unit": UNIT,
               "decisions_per_step": int(res["decisions"]), "pods_to_schedule": res["n_to_schedule"],
               "pending": res["n_pending"], "bins_opened": [int(x) for x in res["bins_opened"]],
               "cluster_plan": plan, "gpu_launches": int(launches),
               "roofline": {"bound": "hbm", "achieved": k_bytes / (k_ms * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s",
                            "frac": k_bytes / (k_ms * 1e-3) / 1e9 / (peak * world), "traffic": None,
                            "peak_source": peak_src + " x %d GPUs" % world, "kernel_ms_per_step": k_ms,
                            "note": "SURVEY 8(d) algorithmic bytes over the slowest rank's pipeline time (nodes pass + "
                                    "bin passes, barriers and merges between them included)"}}
        if host_ms is not None:
            rec["e2e"] = {"value": res["decisions"] * steps / (host_ms2 * 1e-3), "unit": UNIT, "ms_per_step": host_ms2 / steps,
                          "h2d_bytes_per_step": int(w.h2d) * world, "d2h_bytes_per_step": int(w.d2h) * world,
                          "path": "every rank: occupancy_host + scale_up_host (cluster mode) + maintain_host from pinned arrays"}
        if verify:
            # the single-GPU answer of the same snapshot, on rank 0, in the same run: must be identical
            ok = torch.ones(1, dtype=torch.int64, device=eng.device)
            solo_ms = torch.zeros(1, dtype=torch.float64, device=eng.device)
            if rank == 0:
                solo = Engine(local_rank)
                ws = Workload(solo, c, pinned=False)
                r1, ms1, _ = timed(ws.step_device, solo_steps, 1, flush, lambda: torch.cuda.synchronize(),
                                   lambda: solo.launch_count)
                solo_ms[0] = ms1 / solo_steps
                same = (torch.equal(r1["placed"], res["placed"]) and torch.equal(r1["acc_pool"], res["acc_pool"])
                        and torch.equal(ws.used.view(torch.int64), w.used.view(torch.int64))
                        and np.array_equal(r1["new_size"], res["new_size"]) and r1["decisions"] == res["decisions"]
                        and np.array_equal(r1["bins_opened"], res["bins_opened"]))
                ok[0] = 1 if same else 0
                solo.close()
                del ws
            # every rank holds the same replicated result as rank 0
            h = torch.stack([res["placed"].to(torch.int64).sum(), (res["placed"].to(torch.int64) * 31 % 1000003).sum(),
                             w.used.view(torch.int64).sum(), res["acc_pool"].to(torch.int64).sum()])
            hmax, hmin = h.clone(), h.clone()
            dist.all_reduce(hmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(hmin, op=dist.ReduceOp.MIN)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            dist.all_reduce(solo_ms, op=dist.ReduceOp.MAX)
            assert torch.equal(hmax, hmin), "ranks hold different results"
            assert int(ok[0]) == 1, "cluster-mode result differs from the single-GPU result"
            rec["verified"] = "placements, used bits, accounted pools, pool sizes and decision count equal the " \
                              "single-GPU tick of the same snapshot (rank 0, same run); identical on all ranks"
            rec["strong_scaling"] = {"n1_ms_per_step": float(solo_ms[0]), "ms_per_step": dev_ms / steps,
                                     "speedup": float(solo_ms[0]) / (dev_ms / steps), "n_gpus": world}
        del w
        torch.cuda.empty_cache()
        return rec, c

    with ClockSampler(local_rank) as clocks:
        head, c = measure(name, args.steps, args.warmup, dump_dir=args.dump_outputs)
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": head["workload"], "seed": SEED, "decisions_per_step": head["decisions_per_step"],
                   "pods_to_schedule": head["pods_to_schedule"], "pending": head["pending"],
                   "bins_opened": head["bins_opened"], "l2": "flushed between timed iterations (256 MiB fill)",
                   "python_gc": "paused over the timed steps",
                   "tick": "occupancy (K1, replicated) + scale_up in cluster mode (node / bin axis split over the ranks, "
                           "stage pipeline continued over NVLink peer memory) + NCCL all-reduce of the per-pool counts "
                           "+ node_states (K6) + maintain (replicated)",
                   "parallelism": "one cluster on %d ranks: node ranges per rank, %s" % (world, json.dumps(head["cluster_plan"]))},
        "roofline": head["roofline"], "e2e": head.get("e2e"), "gpu_launches": head["gpu_launches"],
        "clocks": clocks.summary(), "verified": head.get("verified"), "strong_scaling": head.get("strong_scaling"),
        "pods_per_s": P / (head["ms_per_step"] * 1e-3),
    }
    configs = {}
    if run_c4:
        try:
            configs["c4"], _ = measure("c4", 2, 1, verify=not args.no_c4_verify, solo_steps=1)
        except Exception as e:
            configs["c4"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if configs:
        line["configs"] = configs
    if not args.no_fleet:
        # secondary: the round-1 weak-scaling measurement (independent c2 cluster shards, one all-reduce of the counts)
        fleet_eng = Engine(local_rank)
        Pf, Nf, Df, Tf = CONFIGS["c2"]
        cf = syn.make_cluster(Pf, Nf, Df, Tf, seed=SEED + 1000 * rank)
        wf = Workload(fleet_eng, cf, pinned=False)

        def fstep():
            r = wf.step_device()
            r["fleet"] = acs_dist.fleet_scale_up(r, cf["pool_actual"])
            return r
        rf, f_ms, _ = timed(fstep, 5, 2, flush, barrier, lambda: fleet_eng.launch_count)
        t = torch.tensor([f_ms, float(rf["decisions"])], dtype=torch.float64, device=eng.device)
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        line["fleet"] = {"workload": "%d independent c2 clusters (weak scaling, one all-reduce of the counts)" % world,
                         "value": float(t[1]) * 5 / (float(tm[0]) * 1e-3), "unit": UNIT, "ms_per_step": float(tm[0]) / 5}
    if rank == 0:
        print(json.dumps(line))
    acs_dist.barrier()
    acs_dist.shutdown()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the configs.c3 / configs.c5 sub-records")
    ap.add_argument("--no-c4", action="store_true", help="N > 1: skip the configs.c4 sub-record (10M x 1M, ~1 minute)")
    ap.add_argument("--no-c4-verify", action="store_true", help="skip the single-GPU check of c4 (tens of seconds)")
    ap.add_argument("--no-fleet", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup not negative")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU tick (--impl ours)")
    sys.dont_write_bytecode = True  # the tree may be read-only: nothing imported from here leaves a cache in it
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the pod-fit path has no CPU fallback")
    if world > 1:
        run_cluster(args)
    else:
        run_single(args)


if __name__ == "__main__":
    main()
