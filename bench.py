#!/usr/bin/env python3
"""bench.py -- BLS12-381 G1 multi-scalar-multiplication throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--logn 20] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one MSM of 2^logn (scalar, point) pairs (configs[2]: BLS12-381 G1, N = 2^20, uniform 255-bit scalars not
reduced mod r, points in the prime-order subgroup).  Prints ONE JSON line on rank 0.

  value   MSMs/s, inputs resident in HBM when the timed region starts (ctt_b200_msm_device), CUDA events on the stream
          the kernels are launched on, max over ranks.  N > 1: ONE MSM per step, inputs replicated, windows sharded over the ranks
          (strong scaling): window digits stay on the device, ONE NCCL all_gather + one host pass, inside the timed region.
  e2e     same metric through the reference's own C symbol ctt_bls12_381_g1_jac_multi_scalar_mul_big_coefs_vartime_parallel
          with HOST (pinned) buffers: H2D of scalars+points and D2H of the window digits inside the timed region; e2e.pageable is
          the same call with ordinary malloc'd buffers.  Every leg's result is checked against the closed form (closed_form_check).
  roofline  accumulation phase (batched-affine levels + k_accumulate): algorithmic 32x32->64 integer MACs (3300 per bucket
          point-add, SURVEY.md 8d) / its CUDA-event duration, against the measured IMAD.WIDE.X issue peak (profiles/ubench_r1.jsonl,
          profiles/sass_integer_pipe_r2.txt) -- may exceed 1, see frac_note; frac_executed counts the multiplications really issued.
          The HBM fraction (algorithmic bytes / step time vs MEASURED_PEAKS.json) is reported beside it.
  cpu_baseline  the oracle's restatement of the reference's CPU algorithm (kind "port": the Nim reference cannot be
          built in this image) on all host cores, bounded sample.
--impl reference times that same CPU restatement as the reference arm.
--dump-outputs DIR writes what the last timed step of each leg returned (dump_outputs), so that two builds can be compared
          output for output: the inputs depend on the arguments only.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the benchmark writes nothing into the tree (it may be read-only)

CURVE = "bls12_381_g1"                   # default workload; --curve selects another BASELINE config (same harness)
INT_MACS_PER_POINT_ADD = 3300            # SURVEY.md 8d: 11 field mults x (2*12^2 + 12) MACs, BLS12-381 G1
ALGO_BYTES_PER_TERM = 128                # 32 B scalar + 96 B affine point
# SURVEY.md 8d per-unit figures for the other groups: (int-MACs per point-add, algorithmic bytes per term)
UNIT_FIGURES = {"bls12_381_g1": (3300, 128), "bn254_snarks_g1": (1496, 96), "pallas_ec": (1496, 96), "vesta_ec": (1496, 96),
                "bls12_381_g2": (9000, 224), "bn254_snarks_g2": (4080, 160)}
# Measured on this pool's B200 (tools/ubench.cu, profiles/ubench_r1.jsonl): the integer multiplier issues 63.4 IMAD /clk/SM,
# i.e. one 32-bit result half per lane per pass; a full 32x32->64 multiply-accumulate (IMAD.WIDE.U32 with 64-bit addend
# or carry, what mad.lo.cc/madc.hi.cc pairs compile to) takes two passes: measured 31.65 MAC/clk/SM
# => 148 SMs x 31.65 x 1.965 GHz = 9.2e12 MACs/s.  (A carry-free reduced-radix multiplier was prototyped and is slower:
# profiles/ubench_r1b.jsonl.)
INT_MAC_PEAK_PER_S = 9.205e12
# dram__bytes_read.sum + dram__bytes_write.sum of the accumulation phase of one MSM at N = 2^20, c = 16 (three k_affine_pairs launches +
# k_accumulate) from the committed `ncu --set full` capture (profiles/ncu_accumulate_and_reduce_r2.txt): 6.334 GB + 2.224 GB. The
# algorithmic gather is 1.61 GB: the batched-affine levels trade DRAM traffic (pair lists, two operand reads per pair and pass, prefix
# products, level results; 24 % of the DRAM peak) for multiplications. Round 1 (XYZZ only, profiles/ncu_k_accumulate_r1.txt): 1.51 GB.
NCU_TRAFFIC_BYTES_N20 = 8.558e9


def workload_string(curve, logn):
    """config.workload, identical in both arms (the driver compares them)."""
    from constantine_b200.curves import CURVES
    cv = CURVES[curve]
    return (f"BLS12-381 G1 MSM N=2^{logn} (BASELINE configs[2]), uniform 255-bit scalars, subgroup points" if curve == "bls12_381_g1"
            else f"{curve} MSM N=2^{logn}, uniform {cv.scalar_bits}-bit scalars, subgroup points")


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler(threading.Thread):
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self._halt = threading.Event()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def make_inputs(n, seed):
    """Synthetic inputs: scalars uniform in [0, 2^255) (not reduced mod r, like reference
    benchmarks/bench_elliptic_parallel_template.nim:90); points P_i = [k_i]G with random 64-bit k_i, computed on the GPU
    by the library's generator hook (prime-order subgroup by construction). Returns numpy uint8 arrays + the k_i."""
    import numpy as np
    from constantine_b200 import _lib
    from constantine_b200.curves import CURVES
    cv = CURVES[CURVE]
    rng = np.random.default_rng(seed)
    scal = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    scal[:, 31] &= (1 << (cv.scalar_bits - 248)) - 1
    k = rng.integers(1, 2**63, size=n, dtype=np.uint64)
    gen = np.frombuffer(_gen_bytes(cv), dtype=np.uint8).copy()
    pts = np.empty((n, cv.aff_bytes), dtype=np.uint8)
    lib = _lib.load()
    rc = lib.ctt_b200_scalar_mul_u64(cv.curve_id, gen.ctypes.data, k.ctypes.data, n, pts.ctypes.data)
    assert rc == 0
    return scal, pts, k


def _gen_bytes(cv):
    f = cv.fp
    out = b""
    for coord in cv.gen:
        for c in coord:
            out += f.to_mont(c).to_bytes(f.nbytes, "little")
    return out


def effective_cores():
    """Host cores this process may actually use: min(affinity mask, cgroup CPU quota). os.cpu_count() reports the
    machine, not the container."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def algorithmic_point_adds(n, c, bits=255):
    """SURVEY.md 8d: W*(N + 2*2^(c-1)) + W*(c+1), W = floor(b/c)+1."""
    W = bits // c + 1
    return W * (n + 2 * (1 << (c - 1))) + W * (c + 1)


def time_oracle(n_full, budget_s=20.0, max_logn=20):
    """CPU baseline: the oracle's signed-window one-task-per-window MSM with batched-affine bucket sums (restatement of the
    reference's parallel MSM: its window choice, its MSM-level split, its arithmetic for c >= 9 -- 6 multiplications per bucket
    addition around a shared inversion) on all host cores, on a bounded sample."""
    import numpy as np
    from constantine_b200.curves import CURVES
    from oracle import oracle
    cv = CURVES[CURVE]
    cores = effective_cores()
    lib = oracle.load()                  # built by __graft_entry__.build(); no rebuild from a possibly read-only tree
    cvt = oracle.curve_t(cv)
    # points for the CPU sample: multiples of G generated by the oracle itself is not needed -- timing does not depend on
    # the values, so reuse a small pool of valid points produced by the exact tier.
    from oracle import pyref
    import random
    rnd = random.Random(99)
    pool = np.frombuffer(b"".join(pyref.aff_to_bytes(pyref.ec_mul_fast(rnd.getrandbits(64) | 1, cv.gen, cv), cv) for _ in range(256)),
                         dtype=np.uint8).reshape(256, cv.aff_bytes)
    rng = np.random.default_rng(5)

    def run(logn, threads):
        n = 1 << logn
        pts = pool[rng.integers(0, 256, size=n)]
        scal = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        scal[:, 31] &= 0x7F
        out = ctypes.create_string_buffer(cv.jac_bytes)
        pts = np.ascontiguousarray(pts)
        t0 = time.perf_counter()
        c = lib.oracle_msm(ctypes.byref(cvt), out, scal.ctypes.data, pts.ctypes.data, n, 0, oracle.IMPL_SIGNED_AFFINE, 0, threads)
        return time.perf_counter() - t0, c

    # containers often expose more CPUs than their quota allows: probe a few thread counts and keep the fastest
    best = None
    for th in sorted({cores, max(1, cores // 2), min(cores, 32), min(cores, 16)}, reverse=True):
        t, _ = run(15, th)
        t = min(t, run(15, th)[0])
        if best is None or t < 0.9 * best[0]:   # prefer more threads unless fewer are clearly faster
            best = (t, th)
    t15, threads = best
    logn = 15
    while logn < max_logn and (1 << logn) < n_full and t15 * (1 << (logn + 1 - 15)) * 0.8 < budget_s:
        logn += 1
    t, c = run(logn, threads)
    cores = threads
    n = 1 << logn
    padds = algorithmic_point_adds(n, c)
    scale = n_full / n   # MSM cost is ~linear in N at these sizes (window count shrinks slowly): scaled, stated in `sample`
    return {"value": 1.0 / (t * scale), "unit": "MSM/s", "cores": cores, "kind": "port",
            "sample": f"one MSM of 2^{logn} pairs in {t:.2f} s (c={c}, {padds / t / 1e6:.1f} Mop point-adds/s = "
                      f"{padds / t / 1e6 / cores:.2f} per thread), scaled x{scale:g} to N=2^{n_full.bit_length() - 1}; "
                      "C port with batched-affine bucket sums and a MULX/ADX multiplication, NOT Constantine itself: the reference "
                      "publishes 33 Mop/s on 16 Zen4 threads at N=2^18 (BASELINE.md)",
            "point_adds_per_s": padds / t, "seconds": t, "logn": logn}


def dump_outputs(dirname, cv, results):
    """DIR/msm_<leg>_jac.npy: the Jacobian struct each leg's caller received from its last timed step, as its little-endian 32-bit
    words (exact in float64), shape (3, words per coordinate), Montgomery form. DIR/msm_resident_affine.npy: that point in affine
    coordinates, which unlike Jacobian ones are unique, as 32-bit words of the canonical integers, shape (2, extension degree,
    words per field element); zeros for the point at infinity."""
    import numpy as np
    from oracle import pyref
    os.makedirs(dirname, exist_ok=True)
    for leg, raw in results.items():
        words = np.frombuffer(raw[:cv.jac_bytes], dtype="<u4").astype(np.float64).reshape(3, -1)
        np.save(os.path.join(dirname, f"msm_{leg}_jac.npy"), words)
    nw = cv.fp.nbytes // 4
    aff = np.zeros((2, cv.ext_degree, nw), dtype=np.float64)
    P = pyref.jac_bytes_to_affine(results["resident"], cv)
    if P is not None:
        for i, coord in enumerate(P):
            for j, v in enumerate(coord):
                aff[i, j] = [(v >> (32 * w)) & 0xFFFFFFFF for w in range(nw)]
    np.save(os.path.join(dirname, "msm_resident_affine.npy"), aff)


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    n = 1 << args.logn
    vals = []
    info = None
    for i in range(args.warmup + args.steps):
        info = time_oracle(n, budget_s=12.0)
        if i >= args.warmup:
            vals.append(info["seconds"] * (n / (1 << info["logn"])))
    ms = 1e3 * sum(vals) / len(vals)
    v = 1e3 / ms
    line = {"impl": "reference", "metric": "bls12_381_g1_msm_throughput", "value": v, "unit": "MSM/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_string(CURVE, args.logn), "note":
                       "C restatement (oracle port, NOT Constantine itself) of the reference's parallel MSM on all host cores: its window "
                       "choice, MSM-level split, batched-affine bucket sums and a MULX/ADX Montgomery multiplication; the Nim reference "
                       "cannot be built in this image"},
            "cpu_baseline": {"value": v, "unit": "MSM/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]},
            "e2e": {"value": v, "unit": "MSM/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--logn", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--curve", default="bls12_381_g1", help="bls12_381_g1 (default, BASELINE metric) | pallas_ec | bls12_381_g2 | ...")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of each leg's last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    global CURVE, INT_MACS_PER_POINT_ADD, ALGO_BYTES_PER_TERM
    CURVE = args.curve
    INT_MACS_PER_POINT_ADD, ALGO_BYTES_PER_TERM = UNIT_FIGURES[CURVE]
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    from constantine_b200 import _lib, msm as M, sharded
    from constantine_b200.curves import CURVES

    rank, world, local = dist_env()
    cv = CURVES[CURVE]
    # NCCL prints its version banner on stdout at the first collective: keep stdout clean for the ONE JSON line by
    # pointing fd 1 at stderr until the result is printed
    sys.stdout.flush()
    saved_stdout_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    n = 1 << args.logn
    lo, hi = sharded.balanced_chunk(n, world, rank)
    n_loc = hi - lo
    # Every rank generates the same global instance (same seed). Resident leg, N > 1: the (scalar, point) arrays are
    # replicated in every GPU's HBM and the MSM is sharded by WINDOW RANGE (north star: "sharded by scalar-window ... final
    # NCCL exchange of <= 8 partial points"). End-to-end leg: the host arrays are sharded by POINTS, so each rank moves only
    # its N/world pairs over PCIe. Both end in one all_gather of <= world partial points + host adds.
    scal_all_seed = 0xC770003
    scal, pts, k_dlog = make_inputs(n, scal_all_seed)
    d_scal = torch.from_numpy(scal).to(dev)
    d_pts = torch.from_numpy(pts).to(dev)
    h_scal = torch.from_numpy(np.ascontiguousarray(scal[lo:hi])).pin_memory()
    h_pts = torch.from_numpy(np.ascontiguousarray(pts[lo:hi])).pin_memory()
    # ordinary (pageable) heap buffers, what a C / Rust / Nim caller of the reference symbol passes
    pg_scal = np.ascontiguousarray(scal[lo:hi]).copy()
    pg_pts = np.ascontiguousarray(pts[lo:hi]).copy()
    torch.cuda.synchronize()
    # run the engine on a torch-owned (non-default) stream so that torch.cuda.Event brackets exactly the launches
    bench_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(bench_stream)
    lib.ctt_b200_set_stream(ctypes.c_void_p(bench_stream.cuda_stream))
    c_plan, W_plan = M.plan(cv, n)
    wb, we = sharded.window_range(W_plan, world, rank)

    def step_resident():
        if world == 1:
            return M.msm_device_ptrs(cv, d_scal.data_ptr(), d_pts.data_ptr(), n, out=M.OUT_JAC)
        return sharded.msm_window_sharded_device(cv, d_scal.data_ptr(), d_pts.data_ptr(), n, c_plan, W_plan, device=dev)

    symbol = f"ctt_{cv.cprefix}_jac_multi_scalar_mul_big_coefs_vartime_parallel"
    named = _lib.named_msm(symbol)
    named_xyzz = lib.ctt_b200_msm_host
    tp = M.Threadpool.new(1)
    r_buf = ctypes.create_string_buffer(4 * cv.coord_bytes)

    def step_e2e():
        if world == 1:
            named(tp._h, r_buf, h_scal.data_ptr(), h_pts.data_ptr(), n_loc)
            return r_buf.raw[:cv.jac_bytes]
        named_xyzz(cv.curve_id, M.OUT_XYZZ, r_buf, h_scal.data_ptr(), h_pts.data_ptr(), n_loc, 0)
        return sharded.msm_point_sharded(cv, r_buf.raw, device=dev)

    def step_e2e_pageable():
        if world == 1:
            named(tp._h, r_buf, pg_scal.ctypes.data, pg_pts.ctypes.data, n_loc)
            return r_buf.raw[:cv.jac_bytes]
        named_xyzz(cv.curve_id, M.OUT_XYZZ, r_buf, pg_scal.ctypes.data, pg_pts.ctypes.data, n_loc, 0)
        return sharded.msm_point_sharded(cv, r_buf.raw, device=dev)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, collect=None):
        """(ms per step on the stream, wall ms per step, what the last step returned)"""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            last = fn()
            if collect is not None:
                collect(M.last_stats())
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ev_ms = e0.elapsed_time(e1)
        ms = max(ev_ms, 0.0)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms, wall_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall_ms = t[0].item(), t[1].item()
        return ms / steps, wall_ms / steps, last

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    stats = []
    ms_res, wall_res, out_res = timed(step_resident, args.steps, args.warmup, collect=stats.append)
    e2e_stats = []
    ms_e2e, wall_e2e, out_e2e = timed(step_e2e, args.steps, args.warmup, collect=e2e_stats.append)
    ms_e2e_pg, wall_e2e_pg, out_e2e_pg = timed(step_e2e_pageable, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    # the engine launches strictly in order on one stream, so the CUDA events it records around the accumulation phase bracket
    # those kernels alone
    serial_stats = stats
    ms_serial = ms_res

    # Extra (not the headline): two host threads calling concurrently, as the reference's callers may (KZG batch
    # verification issues three MSMs at once). Each thread leases its own engine slot (streams + scratch), so the
    # latency-bound reduce / host tail of one MSM overlaps the accumulate phase of the other. Wall clock, synchronised.
    concurrent = None
    if world == 1:
        import threading as _th
        def _worker(k):
            for _ in range(k):
                M.msm_device_ptrs(cv, d_scal.data_ptr(), d_pts.data_ptr(), n, out=M.OUT_JAC)
        for _ in range(2):
            ths = [_th.Thread(target=_worker, args=(2,)) for _ in range(2)]
            [t.start() for t in ths]; [t.join() for t in ths]
        torch.cuda.synchronize()
        per_thread = max(1, args.steps // 2)
        t0 = time.perf_counter()
        ths = [_th.Thread(target=_worker, args=(per_thread,)) for _ in range(2)]
        [t.start() for t in ths]; [t.join() for t in ths]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        concurrent = {"threads": 2, "msms": 2 * per_thread, "value": 2 * per_thread / dt, "unit": "MSM/s",
                      "note": "two concurrent callers, two engine slots; wall clock"}

    # correctness of what was timed: every leg against the closed form  MSM = [sum s_i k_i mod r] G  (the points are k_i G)
    ra, rb, rc_ = step_resident(), step_e2e(), step_e2e_pageable()
    from oracle import pyref
    s_int = [int.from_bytes(scal[i].tobytes(), "little") for i in range(n)]
    expect = pyref.ec_mul_fast(sum(a * int(b) for a, b in zip(s_int, k_dlog)) % cv.fr.modulus, cv.gen, cv)
    legs_ok = [pyref.jac_bytes_to_affine(x, cv) == expect for x in (ra, rb, rc_)]
    same = all(legs_ok)

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cv, {"resident": out_res, "e2e_pinned": out_e2e, "e2e_pageable": out_e2e_pg})

    st = stats[-1]
    if world > 1:
        # the window-digit leg returns without per-rank timing (no synchronisation inside the engine): take the phase times of
        # this rank's window range from three extra calls of the synchronous device entry
        serial_stats = []
        for _ in range(3):
            M.msm_device_ptrs(cv, d_scal.data_ptr(), d_pts.data_ptr(), n, out=M.OUT_XYZZ, force_c=c_plan, win_begin=wb, win_end=we)
            serial_stats.append(M.last_stats())
        st = serial_stats[-1]
    acc_ms = max(1e-6, sum(s["ms_accumulate"] for s in serial_stats) / len(serial_stats))
    madds = st["entries"]      # bucket point-adds issued by k_accumulate per launch (one per sorted entry, minus run heads)
    macs = madds * INT_MACS_PER_POINT_ADD
    achieved = macs / (acc_ms * 1e-3)
    # executed MACs: an XYZZ mixed add runs 6 products + 2 squarings + 1 two-product multiplication (2710 MACs for 12 limbs, 8.2 field
    # multiplications), a batched-affine addition 6 field multiplications; after AL levels ~2^-AL of the entries are left for XYZZ
    n32 = cv.fp.nbytes // 4
    fmul = 2 * n32 * n32 + n32
    al = st["affine_levels"]
    xyzz_macs = 8.2 * fmul * (3 if cv.ext_degree == 2 else 1)
    aff_macs = 6.0 * fmul * (3 if cv.ext_degree == 2 else 1)
    executed = madds * ((1.0 - 2.0 ** -al) * aff_macs + 2.0 ** -al * xyzz_macs) if al else madds * xyzz_macs
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    algo_bytes = n * ALGO_BYTES_PER_TERM
    hbm_achieved = algo_bytes / (ms_res * 1e-3) / 1e9
    padds = algorithmic_point_adds(n, st["c"], cv.scalar_bits)
    line = {
        "metric": f"{CURVE}_msm_throughput", "value": 1e3 / ms_res, "unit": "MSM/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": workload_string(CURVE, args.logn),
                   "parallelism": "1 GPU" if world == 1 else (f"resident leg: inputs replicated, {W_plan} windows sharded over {world} GPUs, one NCCL all_gather of the window "
                                                                  f"digits + one host pass; e2e leg: points sharded over {world} GPUs + all_gather of partial points"),
                   "window_c": st["c"], "windows": st["num_windows"],
                   "l2": "no flush needed: inputs (128 MiB) + sort/bucket scratch (~470 MiB) exceed the 126 MB L2"},
        "point_adds_per_s": padds / (ms_res * 1e-3), "Mop_point_adds_per_s": padds / (ms_res * 1e-3) / 1e6,
        "wall_ms_per_step": wall_res,
        "e2e": {"value": 1e3 / ms_e2e, "unit": "MSM/s", "ms_per_step": ms_e2e, "wall_ms_per_step": wall_e2e,
                "h2d_bytes_per_step": int(n_loc * ALGO_BYTES_PER_TERM), "d2h_bytes_per_step": int(st["num_windows"] * 4 * cv.coord_bytes),
                "api": symbol + " (pinned host buffers)", "input_chunks_in_flight": "engine default (ctt_b200_set_input_chunks)",
                "pageable": {"value": 1e3 / ms_e2e_pg, "unit": "MSM/s", "ms_per_step": ms_e2e_pg, "wall_ms_per_step": wall_e2e_pg,
                             "note": "same call with ordinary malloc'd (pageable) host buffers, as an unmodified caller of the reference symbol passes"}},
        "gpu_launches": int(sum(s["kernel_launches"] for s in stats)),
        "phases_ms_serial_launch_order": {k: round(sum(s[k] for s in serial_stats) / len(serial_stats), 4) for k in
                                          ("ms_digits", "ms_sort", "ms_accumulate", "ms_fixup", "ms_reduce", "ms_d2h_tail", "ms_total")},
        "ms_per_step_serial_launch_order": ms_serial, "window_groups": st["groups"], "slice_len": st["slice_len"],
        "roofline": {"bound": "int32-mad (neither hbm nor tensor: see roofline_hbm)",
                     "kernel": ("bucket accumulation phase: k_affine_pairs x%d levels + k_accumulate over the survivors" % st["affine_levels"]
                                if st["affine_levels"] else "k_accumulate"),
                     "achieved": achieved / 1e12, "peak": INT_MAC_PEAK_PER_S / 1e12, "unit": "TMAC/s (32x32->64)",
                     "frac": achieved / INT_MAC_PEAK_PER_S,
                     "frac_note": "ALGORITHMIC fraction: the unit is the reference's 11-multiplication Jacobian mixed add (3300 MACs, SURVEY.md 8d) per "
                                  "sorted entry; batched-affine additions execute ~6 multiplications (+ a shared inversion), so the figure may exceed 1",
                     "frac_executed": executed / (acc_ms * 1e-3) / INT_MAC_PEAK_PER_S, "executed_macs_per_entry": executed / max(1, madds),
                     "traffic": (NCU_TRAFFIC_BYTES_N20 if (world == 1 and args.logn == 20 and st["c"] == 16 and CURVE == "bls12_381_g1") else None),
                     "traffic_note": "DRAM bytes (read + write) of the phase's four launches from the committed ncu --set full capture "
                                     "(profiles/ncu_accumulate_and_reduce_r2.txt); algorithmic gather = entries x 96 B = 1.61e9 B -- the affine levels "
                                     "re-read operands per pass and park prefix products, 24 % of the DRAM peak",
                     "fmaheavy_pipe_busy_ncu": 0.71,
                     "peak_source": "measured 32x32->64 MAC rate of the register-resident Montgomery multiplier loop (IMAD.WIDE.U32.X carry chains, 2 "
                                    "issue slots each: 31.65 MAC/clk/SM x 148 SM x 1.965 GHz), tools/ubench.cu -> profiles/ubench_r1.jsonl, SASS in profiles/",
                     "algorithmic_work": f"{madds} bucket point-adds x {INT_MACS_PER_POINT_ADD} MACs per step, {acc_ms:.3f} ms"},
        "roofline_hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                         "traffic": None, "peak_source": hbm_src, "algorithmic_bytes": algo_bytes},
        "clocks": clocks, "paths_agree": bool(same), "closed_form_check": {"resident": legs_ok[0], "e2e_pinned": legs_ok[1], "e2e_pageable": legs_ok[2]},
        "concurrent_callers": concurrent,
    }
    if not args.no_cpu_baseline and world == 1 and CURVE == "bls12_381_g1":
        line["cpu_baseline"] = {k: v for k, v in time_oracle(n).items() if k in ("value", "unit", "cores", "kind", "sample")}
    sys.stdout.flush()
    os.dup2(saved_stdout_fd, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def make_inputs_shard(n, seed, lo, hi):
    """Rank-local shard of the global instance: the global scalar / multiplier streams are generated with the same seed on
    every rank and sliced, so the instance does not depend on the world size."""
    import numpy as np
    from constantine_b200 import _lib
    from constantine_b200.curves import CURVES
    cv = CURVES[CURVE]
    rng = np.random.default_rng(seed)
    scal = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    scal[:, 31] &= 0x7F
    k = rng.integers(1, 2**63, size=n, dtype=np.uint64)
    scal, k = np.ascontiguousarray(scal[lo:hi]), np.ascontiguousarray(k[lo:hi])
    gen = np.frombuffer(_gen_bytes(cv), dtype=np.uint8).copy()
    pts = np.empty((hi - lo, cv.aff_bytes), dtype=np.uint8)
    rc = _lib.load().ctt_b200_scalar_mul_u64(cv.curve_id, gen.ctypes.data, k.ctypes.data, hi - lo, pts.ctypes.data)
    assert rc == 0
    return scal, pts, k


if __name__ == "__main__":
    main()
