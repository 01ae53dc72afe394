#!/usr/bin/env python
"""bench.py -- BN254 G1 MSM points/s (+ Fr NTT elements/s) at 2^24 on B200, one process per GPU.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm: oracle port timed on the host cores

A "step" is one pass of the hot path over one batch of synthetic input: one 2^24-point BN254 G1 MSM
(BASELINE.json metric, fits one GPU).  `value` = points/s with bases and scalars resident in HBM;
`e2e` = the same MSM through the reference-facing C-ABI call with HOST scalars (pinned) and resident
bases (the proving key is fixed across proofs), host<->device copies inside the timed region.  The Fr NTT
half of the metric (2^24 forward + inverse) is timed in its own K-step loop and reported under "ntt".

Multi-GPU (weak scaling): every rank owns its own 2^24-point shard of one (N * 2^24)-point MSM, reduces
it to one XYZZ partial sum, NCCL all-gathers the 128-byte partials and folds them -- the all-gather + local
fold is the "allreduce of partial sums" (NCCL has no elliptic-curve reduction).  Timing: CUDA events on
the launching stream, barrier + synchronize on both sides, max over ranks.

Beside the headline, the same JSON line carries the other configurations BASELINE.json names:
  "g2"      2^24-point G2 MSM on one GPU (value, e2e, roofline on n x 160 B)                          [config 4, N=1]
  "strong"  ONE 2^24-point G1 MSM and ONE 2^24-point G2 MSM point-split over the N ranks (strong scaling),
            with the one-GPU time of the same MSM measured in the same run on rank 0                   [config 4]
  "ntt"     2^24 forward + inverse                                                                    [config 3]
  "proof"   Groth16-shaped prove at domain 2^24 through B200Backend.prove (one b200zk_groth16_commit call per
            proof on one GPU; dealt NTTs + one all_gather on N), with the CPU oracle's wall time of the
            same pipeline on a stated smaller domain                                                   [config 5]
Every roofline side field is measured in this run or read from profiles/r2_ncu_kernels.json (written from an
ncu capture by tools/ncu_to_profile_json.py); the file's figures are used only while its source hash equals the
hash of the sources the loaded libb200zk.so was built from, else they are null.
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
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, torchrun notices) also write to fd 1,
# so keep a private handle on the real stdout for the result line and point fd 1 at stderr for everything else.
# Done in main() only: importing bench (tests, tools) leaves the importer's stdout alone.
_RESULT_OUT = None


def claim_stdout():
    global _RESULT_OUT
    if _RESULT_OUT is None:
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def ntt_products_per_element(log_n: int, full_table_max_log: int = 26) -> float:
    """Modular products one forward transform spends per element -- the host-side count of csrc/ntt.cu's schedule (default
    plan of make_ntt_plan; radix-4 rounds whose w^0 twiddles are skipped; one inter-pass product per element when the pass's
    twiddle comes from one lookup -- L <= 16, or the last pass's direct table -- else two)."""
    k = log_n
    if k <= 12:
        passes = [k]
    elif k <= 20:
        passes = [(k + 1) // 2, k - (k + 1) // 2]
    else:
        s0 = (k + 2) // 3
        s1 = (k - s0 + 1) // 2
        passes = [s0, s1, k - s0 - s1]
    total, done = 0.0, 0
    for i, s in enumerate(passes):
        q = 0
        if s & 1:  # one radix-2 stage: half a product per element, none for jj = 0
            total += 0.5 * (1 - 1 / (1 << (s - 1)))
            q = 1
        while q < s:  # radix-4 round: 4 products per quad, 1 when jj = 0 (one quad in m/2)
            m2 = 1 << (s - 2 - q)
            total += 1 - 0.75 / m2
            q += 2
        done += s
        if i > 0:
            last = i == len(passes) - 1
            total += 1 if (done <= 16 or (last and 16 < k <= full_table_max_log)) else 2
    return total


def emit_result(line: dict):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


SEED_SCALARS, SEED_POINTS, SEED_NTT = 0xB2000001, 0xB2000002, 0xB2000003
R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
# --dump-outputs keeps a fixed, seeded sample of DUMP_ELEMS elements of a long vector (a 2^24-element Fr vector is 512 MiB)
SEED_DUMP, DUMP_ELEMS = 0xB2000004, 1 << 16


def dump_outputs(out_dir: str, outputs: dict):
    """--dump-outputs: out_dir/<name>.npy for every output of the last timed step, so that two builds run with the same
    arguments can be compared output for output.  Each output is the bytes a caller receives (encoded points, proof
    bytes, field elements as little-endian limbs), one float32 per byte: exact, so a difference in any bit shows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, raw in outputs.items():
        a = np.frombuffer(raw, dtype=np.uint8) if isinstance(raw, bytes) else raw
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def source_hash() -> str:
    """sha256 over the sources libb200zk.so is built from (csrc/*.cu, *.cuh, Makefile, include/b200zk.h): the "build
    hash" that ties profiles/r2_ncu_kernels.json to the code that was profiled."""
    import glob
    import hashlib
    h = hashlib.sha256()
    files = sorted(glob.glob(os.path.join(ROOT, "ethrex_b200", "csrc", "*.cu")) + glob.glob(os.path.join(ROOT, "ethrex_b200", "csrc", "*.cuh")))
    files += [os.path.join(ROOT, "ethrex_b200", "csrc", "Makefile"), os.path.join(ROOT, "include", "b200zk.h")]
    for f in files:
        h.update(os.path.basename(f).encode() + b"\0")
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_profile(kernel_key: str):
    """entry of profiles/r2_ncu_kernels.json for `kernel_key` if the file was captured on THIS source tree, else None"""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_kernels.json")) as f:
            doc = json.load(f)
    except Exception:  # noqa: BLE001
        return None
    if doc.get("source_hash") != source_hash():
        return None
    return doc.get("kernels", {}).get(kernel_key)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU arm
def cpu_msm_sample(log_sample: int, threads: int = 0):
    """(points/s, seconds, cores) of the CPU oracle's Pippenger on a 2^log_sample slice of the same workload."""
    import cpu_oracle as orc
    import pyref
    n = 1 << log_sample
    k, d = pyref.chain_scalar(SEED_POINTS)
    pts = orc.g1_chain(n, k, d)
    s = orc.rand_fr(SEED_SCALARS, 0, n)
    t0 = time.perf_counter()
    out = orc.g1_msm(pts, s, 0, threads)
    dt = time.perf_counter() - t0
    return n / dt, dt, (threads or orc.num_threads()), out, (pts, s, k, d)


def cpu_ntt_sample(log_sample: int, threads: int = 0):
    import cpu_oracle as orc
    n = 1 << log_sample
    a = orc.fr_to_mont(orc.rand_fr(SEED_NTT, 0, n))
    t0 = time.perf_counter()
    orc.fr_ntt(a, log_sample, 0, threads=threads)
    dt = time.perf_counter() - t0
    return n / dt, dt


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the box's host cores.  The reference's own
    (third-party, Rust/Go) MSM cannot be built here (no cargo/go, sources not vendored: SURVEY.md 8c), so this
    is the oracle port (ark-ec 0.5.0 Pippenger rule, OpenMP over windows/chunks)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import cpu_oracle as orc
    log_sample = args.cpu_log_n
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_msm_sample(min(log_sample, 16))
    times, rate = [], 0.0
    for _ in range(args.steps):
        rate, dt, cores, out, _ = cpu_msm_sample(log_sample)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"g1_msm": out})
    ms = 1e3 * sum(times) / len(times)
    value = (1 << log_sample) / (ms / 1e3)
    ntt_rate, ntt_dt = cpu_ntt_sample(min(22, args.log_n))
    one_log = min(log_sample, 17)
    r1, dt1, _, _, _ = cpu_msm_sample(one_log, threads=1)  # ethrex's lockfile builds ark-ec WITHOUT rayon (SURVEY.md 0.4)
    line = {
        "impl": "reference", "metric": "bn254_g1_msm_points_per_sec", "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32x8 Montgomery (254-bit modular integer)", "data": "synthetic",
        "config": {"workload": f"2^{args.log_n}-point BN254 G1 MSM per GPU (chain bases P_i=(k+i*d)G, uniform Fr scalars), bases+scalars resident in HBM",
                   "points_per_gpu": 1 << args.log_n, "total_points": args.gpus << args.log_n,
                   "reference_arm": f"rank 0 times a 2^{log_sample}-point slice of that workload per step on the host cores (points/s does not depend on the slice length beyond 2^20)"},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": orc.num_threads(), "kind": "port",
                         "sample": f"2^{log_sample}-point slice of the 2^{args.log_n} workload, Pippenger c={orc.lib().orc_msm_window(1 << log_sample)} (ark-ec rule), all host threads",
                         "single_thread": {"value": r1, "unit": "points/s", "sample": f"2^{one_log} points, {dt1:.2f} s (the reference's lockfile configuration: ark-ec without rayon)"},
                         "note": "the reference has no MSM of its own and its third-party ones cannot be built here (no cargo / go, sources not vendored): this is the "
                                 "oracle port of ark-ec 0.5.0's Pippenger; it gets no precomputed window tables (ark has none), the GPU arm does (one-off, outside its timed region)"},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ntt": {"metric": "fr_ntt_elems_per_sec", "value": ntt_rate, "unit": "elements/s", "sample": f"2^{min(22, args.log_n)} forward, {ntt_dt:.3f} s"},
        "gpu_launches": 0,
    }
    emit_result(line)


# ---------------------------------------------------------------------------------------------- GPU arm
def cpu_proof_pipeline(log_n: int, threads: int = 0):
    """The Groth16-shaped pipeline of config 5 on the CPU oracle at domain 2^log_n: 7 NTTs, pointwise quotient, 4 G1 MSMs
    + 1 G2 MSM over chain proving-key columns (the proving key is generated OUTSIDE the timed region, like the GPU arm's
    resident key).  -> (seconds, threads, breakdown)"""
    import numpy as np
    import cpu_oracle as orc
    from ethrex_b200.groth16 import COSET_GEN, SyntheticWrapCircuit, _chain_kd
    n = 1 << log_n
    T = threads or orc.num_threads()
    cols = {}
    for name, is_g2 in SyntheticWrapCircuit.QUERIES:
        k, d = _chain_kd(name.encode())
        cols[name] = (orc.g2_chain if is_g2 else orc.g1_chain)(n, k, d, T)
    w = orc.rand_fr(SEED_SCALARS, 0, n)
    a = orc.fr_to_mont(orc.rand_fr(SEED_NTT, 0, n))
    b = orc.fr_to_mont(orc.rand_fr(SEED_NTT + 1, 0, n))
    c = orc.field_mul("fr", a, b)
    t0 = time.perf_counter()
    cos = []
    for poly in (a, b, c):
        cos.append(orc.fr_ntt(orc.fr_ntt(poly, log_n, orc.NTT_INVERSE, threads=T), log_n, orc.NTT_COSET, threads=T))
    zinv = pow((pow(COSET_GEN, n, R_MOD) - 1) % R_MOD, -1, R_MOD)
    hq = orc.fr_quotient(cos[0], cos[1], cos[2], zinv, T)
    h = orc.fr_from_mont(orc.fr_ntt(hq, log_n, orc.NTT_INVERSE | orc.NTT_COSET, threads=T))
    t_ntt = time.perf_counter() - t0
    t1 = time.perf_counter()
    for name, is_g2 in SyntheticWrapCircuit.QUERIES:
        sc, cnt = (h, n - 1) if name == "h_g1" else (w, n)
        (orc.g2_msm if is_g2 else orc.g1_msm)(cols[name][:cnt], sc[:cnt], 0, T)
    t_msm = time.perf_counter() - t1
    return t_ntt + t_msm, T, {"ntt_quotient_s": t_ntt, "msm_s": t_msm}


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import ethrex_b200 as eb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = eb.Context(local)
    n, log_n = 1 << args.log_n, args.log_n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic workload, generated on the device (deterministic: SURVEY.md section 8d)
    import pyref
    k, d = pyref.chain_scalar(SEED_POINTS)
    start = rank * n
    d_points = torch.empty(8 * n, dtype=torch.int64, device="cuda")
    d_scalars = torch.empty(4 * n, dtype=torch.int64, device="cuda")
    ctx.g1_chain_device(d_points, start, n, k, d)
    ctx.fr_random_device(d_scalars, n, SEED_SCALARS, start)
    d_partial = torch.zeros(16, dtype=torch.int64, device="cuda")
    # the proving key is loaded once: resident bases, expanded to their window multiples (b200zk_bases_precompute)
    handle = ctx.g1_bases_from_device(d_points, n)
    table_setup_s = None
    if not args.no_precompute:
        t0 = time.perf_counter()
        ctx.bases_precompute(handle, args.window)
        ctx.synchronize()
        table_setup_s = time.perf_counter() - t0  # one-off per proving key, OUTSIDE every timed region (reported, not hidden)
    elif args.window:
        ctx.set_msm_window(args.window)
    result, dumps = {}, {}

    from ethrex_b200.dist import msm_sharded, shard_range

    def msm_step():
        if world == 1:
            result["out"] = ctx.g1_msm_resident_device(handle, d_scalars, n)
        else:
            result["out"] = msm_sharded(ctx, d_points, d_scalars, n, handle=handle)

    def timed_loop(fn, steps, warmup, stats=None):
        for _ in range(warmup):
            fn()
        # start the clock sampler BEFORE the barrier: forking nvidia-smi from a process that maps gigabytes of pinned
        # memory takes ~100 ms, and with it after the barrier every other rank's timed region absorbed that wait at the
        # first all_gather (measured at N=8: 61.7 ms "per step" max-over-ranks against 39.9 ms on every rank)
        sampler = ClockSampler(local) if rank == 0 else None
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        l0 = ctx.launch_count
        evs[0].record()
        for i in range(steps):
            fn()
            evs[i + 1].record()  # per-step marks inside the one timed region (min / median / max below)
        barrier()
        ms = evs[0].elapsed_time(evs[steps]) / steps
        per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
        if stats is not None:
            stats.update({"min": per[0], "median": per[len(per) // 2], "max": per[-1]})
        return max_over_ranks(ms), ctx.launch_count - l0, (sampler.stop() if sampler else None)

    def wall_loop(fn, steps, warmup):
        """host wall clock around `steps` synchronous public-API calls (each returns bytes: the D2H read is inside)"""
        for _ in range(warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        return max_over_ranks((time.perf_counter() - t0) / steps)

    msm_step_stats = {}
    ms_step, launches, clocks = timed_loop(msm_step, args.steps, args.warmup, msm_step_stats)
    dumps["g1_msm"] = result["out"]
    value = world * n / (ms_step / 1e3)

    # ---- correctness of what was timed: closed form of the chain MSM (rank 0, outside the timed region)
    import cpu_oracle as orc  # the checker (and the cpu_baseline leg): never inside a timed GPU region

    def closed_form(total_points, seed, g2=False):
        tot = 0
        for lo in range(0, total_points, 1 << 24):
            m = min(1 << 24, total_points - lo)
            s = torch.empty(4 * m, dtype=torch.int64, device="cuda")
            ctx.fr_random_device(s, m, seed, lo)
            tot = (tot + orc.chain_dot(s.cpu().numpy().view(np.uint64).reshape(m, 4), (k + lo * d) % R_MOD, d)) % R_MOD
            del s
        if g2:
            return orc.g2_mul_be(pyref.g2_to_be(pyref.G2_GEN), tot.to_bytes(32, "big"))[1]
        return orc.g1_mul_be(pyref.g1_to_be(pyref.G1_GEN), tot.to_bytes(32, "big"))[1]

    verified = None
    if rank == 0 and not args.no_verify:
        verified = bool(closed_form(world * n, SEED_SCALARS) == result["out"])
        if not verified:
            raise SystemExit("bench.py: GPU MSM result differs from the oracle's closed form -- refusing to report a number")

    # ---- the binding ceiling, measured in THIS run: 254-bit Montgomery products per second of the chip
    # (b200zk_field_mul_device: out = out * b chained `repeat` times per element, one element per thread)
    def modmul_ceiling():
        m = ctx_sm * 2048 * 4
        xa = torch.empty(4 * m, dtype=torch.int64, device="cuda")
        xb = torch.empty(4 * m, dtype=torch.int64, device="cuda")
        ctx.fr_random_device(xa, m, 11, 0)
        ctx.fr_random_device(xb, m, 12, 0)
        rep = 512
        ctx.field_mul_device(xa, xb, xa, m, 0, 8)
        sampler = ClockSampler(local)
        best = 1e30
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ctx.field_mul_device(xa, xb, xa, m, 0, rep)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        clk = sampler.stop()
        return m * rep / (best / 1e3), {"elements": m, "repeat": rep, "ms": best, "sm_mhz": clk.get("sm_mhz")}

    ctx_sm = torch.cuda.get_device_properties(local).multi_processor_count
    modmul_peak, modmul_how = modmul_ceiling()

    # ---- per-kernel time of the dominant kernel (bucket accumulation), live, CUDA events on the launch stream
    def phase_times(fn, reps):
        ctx.set_profiling(True)
        acc, ph = [], None
        for _ in range(reps):
            fn()
            ph = ctx.last_msm_phase_ms()
            acc.append(ph["accumulate"])
        ctx.set_profiling(False)
        return sum(acc) / len(acc), ph

    acc, phases = phase_times(lambda: ctx.g1_msm_partial_resident_device(handle, d_scalars, n, d_partial), max(2, min(args.steps, 5)))
    peak, peak_src = _peaks()
    algo_bytes = n * 96 + 64  # SURVEY.md 8(d): n x (32 B scalar + 64 B affine base) read + 64 B written
    achieved = algo_bytes / (acc / 1e3) / 1e9
    default_cfg = log_n == 24 and not args.no_precompute and not args.window
    prof = ncu_profile("msm_accumulate_g1") if default_cfg else None
    adds = n * 13 if (not args.no_precompute and not args.window and log_n >= 20) else None
    # multiply instructions of one XYZZ mixed addition, in units of one Montgomery product (136 IMAD-type
    # instructions): 6 products + one two-product/one-reduction mul2 (200) + 2 dedicated squarings (108 each)
    PE = (6 * 136 + 200 + 2 * 108) / 136.0
    roofline = {"bound": "hbm", "kernel": "msm_accumulate<Fq>", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (prof["dram_bytes_read"] + prof["dram_bytes_write"]) if prof else None,
                "traffic_source": "profiles/r2_ncu_kernels.json (ncu --set full of this source tree)" if prof else "no ncu capture of this source tree: null",
                "peak_source": peak_src, "kernel_ms": acc, "phases_ms": phases,
                "binding_roofline": {"bound": "fmaheavy pipe (IMAD.WIDE): 254-bit modular products", "peak_products_per_s": modmul_peak,
                                     "peak_measured": modmul_how,
                                     "achieved_products_per_s": (adds * PE / (acc / 1e3)) if adds else None,
                                     "frac": (adds * PE / (acc / 1e3) / modmul_peak) if adds else None,
                                     "ncu_sm__pipe_fmaheavy_cycles_active_pct": (prof.get("fmaheavy_pct") or prof.get("fmaheavy_pct_elapsed")) if prof else None},
                "note": "integer-compute-bound kernel (n*13 XYZZ mixed additions of 9.06 product-equivalents: 6 products, one mul2, 2 squarings): the HBM fraction is small by "
                        "construction, see DESIGN.md section 4; kernel_ms is measured in the one-shot schedule"}

    # ---- the same MSM over PLAIN resident bases (no window table): what a caller gets without the one-off precompute
    plain = None
    if not args.no_plain and world == 1 and not args.no_precompute:
        hp = ctx.g1_bases_from_device(d_points, n)
        st = {}
        pms, _, _ = timed_loop(lambda: result.__setitem__("plain", ctx.g1_msm_resident_device(hp, d_scalars, n)), args.steps, 2, st)
        ctx.bases_free(hp)
        assert result["plain"] == result["out"]
        plain = {"value": n / (pms / 1e3), "unit": "points/s", "ms_per_step": pms,
                 "note": "resident bases WITHOUT b200zk_bases_precompute (c=17, 15 windows + Horner); the headline uses the 13x window table, whose one-off build is outside the timed region"}

    # ---- e2e: C-ABI call with HOST scalars (pinned), resident bases, result read back -- rank-local shard
    e2e = None
    if not args.no_e2e:
        h_scalars = torch.empty(4 * n, dtype=torch.int64).pin_memory()
        h_scalars.copy_(d_scalars)

        def e2e_step():
            if world == 1:
                result["e2e"] = ctx.g1_msm_resident(handle, h_scalars, n)
            else:  # every rank ships its own shard of scalars (pipelined upload), then partial -> all_gather -> fold
                result["e2e"] = msm_sharded(ctx, None, h_scalars, n, handle=handle)
        wall = wall_loop(e2e_step, args.steps, max(1, args.warmup // 2))
        assert result["e2e"] == result["out"]
        e2e = {"value": world * n / wall, "unit": "points/s", "h2d_bytes_per_step": world * n * 32, "d2h_bytes_per_step": world * 64,
               "ms_per_step": wall * 1e3,
               "api": "b200zk_g1_msm_resident (pinned host scalars -> result bytes; bases resident in HBM)" if world == 1 else
                      "pinned host scalars -> ethrex_b200.dist.msm_sharded (b200zk_g1_msm_partial_resident, NCCL all_gather, fold) -> result bytes"}
        del h_scalars
    ctx.bases_free(handle)
    del d_points
    torch.cuda.empty_cache()

    # ---- G2 MSM at 2^log_n on one GPU (config 4's G2 half at N=1): value, e2e, roofline on n x 160 B
    g2 = None
    if not args.no_g2 and world == 1:
        g2n = n
        k2, d2 = k, d
        pts2 = torch.empty(16 * g2n, dtype=torch.int64, device="cuda")
        ctx.g2_chain_device(pts2, 0, g2n, k2, d2)
        h2 = ctx.g2_bases_from_device(pts2, g2n)
        del pts2
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        ctx.bases_precompute(h2, 0)
        ctx.synchronize()
        g2_setup = time.perf_counter() - t0
        st2 = {}
        g2_steps = args.steps
        g2ms, g2l, _ = timed_loop(lambda: result.__setitem__("g2", ctx.g2_msm_resident_device(h2, d_scalars, g2n)), g2_steps, 2, st2)
        dumps["g2_msm"] = result["g2"]
        g2_ok = None
        if not args.no_verify:
            g2_ok = bool(closed_form(g2n, SEED_SCALARS, g2=True) == result["g2"])
            if not g2_ok:
                raise SystemExit("bench.py: GPU G2 MSM result differs from the oracle's closed form")
        d_partial2 = torch.zeros(32, dtype=torch.int64, device="cuda")
        acc2, ph2 = phase_times(lambda: ctx.g2_msm_partial_resident_device(h2, d_scalars, g2n, d_partial2), 2)
        g2_bytes = g2n * 160 + 128
        prof2 = ncu_profile("msm_accumulate_g2") if default_cfg else None
        # multiply instructions of one G2 mixed addition in units of one Fq product (136 instructions):
        # 6 Fq2 mul (2 mul2_add each) + 2 Fq2 sqr (2 Fq mul each) + 1 mul2_sub over Fq2 (2 mul4_add: 2 x 328/136)
        PE2 = (6 * 2 * 200 + 2 * 2 * 136 + 2 * 328) / 136.0
        g2e = None
        if not args.no_e2e:
            hs = torch.empty(4 * g2n, dtype=torch.int64).pin_memory()
            hs.copy_(d_scalars)
            wall = wall_loop(lambda: result.__setitem__("g2e", ctx.g2_msm_resident(h2, hs, g2n)), g2_steps, 1)
            assert result["g2e"] == result["g2"]
            g2e = {"value": g2n / wall, "unit": "points/s", "ms_per_step": wall * 1e3, "h2d_bytes_per_step": g2n * 32, "d2h_bytes_per_step": 128,
                   "api": "b200zk_g2_msm_resident (pinned host scalars -> 128 result bytes; bases resident)"}
            del hs
        g2 = {"metric": "bn254_g2_msm_points_per_sec", "value": g2n / (g2ms / 1e3), "unit": "points/s", "ms_per_step": g2ms, "step_ms": st2, "points": g2n,
              "verified_vs_oracle": g2_ok, "gpu_launches": g2l, "table_setup_s": g2_setup, "e2e": g2e,
              "roofline": {"bound": "hbm", "kernel": "msm_accumulate<Fq2>", "achieved": g2_bytes / (acc2 / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": g2_bytes / (acc2 / 1e3) / 1e9 / peak, "kernel_ms": acc2, "phases_ms": ph2,
                           "traffic": (prof2["dram_bytes_read"] + prof2["dram_bytes_write"]) if prof2 else None,
                           "binding_roofline": {"bound": "fmaheavy pipe", "peak_products_per_s": modmul_peak,
                                                "achieved_products_per_s": g2n * 13 * PE2 / (acc2 / 1e3), "frac": g2n * 13 * PE2 / (acc2 / 1e3) / modmul_peak,
                                                "ncu_sm__pipe_fmaheavy_cycles_active_pct": (prof2.get("fmaheavy_pct") or prof2.get("fmaheavy_pct_elapsed")) if prof2 else None},
                           "note": "algorithmic bytes n x (32 + 128) B (SURVEY.md 8d); one G2 mixed addition = 26.5 Fq product-equivalents (3600 multiply instructions)"}}
        ctx.bases_free(h2)
        torch.cuda.empty_cache()

    # ---- config 4: ONE 2^log_n-point G1 MSM and ONE G2 MSM point-split over the N ranks (strong scaling)
    strong = None
    if not args.no_strong and world > 1:
        lo, hi = shard_range(n, rank, world)
        m = hi - lo
        strong = {"total_points": n, "points_per_rank": m, "n_gpus": world, "scaling": "strong",
                  "partitioning": "point split; every rank reduces its shard to one XYZZ partial, ONE NCCL all_gather of 128 B (G1) / 256 B (G2) per rank, local fold"}
        for is_g2 in (False, True):
            w = 16 if is_g2 else 8
            tag = "g2" if is_g2 else "g1"
            pts = torch.empty(w * m, dtype=torch.int64, device="cuda")
            (ctx.g2_chain_device if is_g2 else ctx.g1_chain_device)(pts, lo, m, k, d)
            hs_ = (ctx.g2_bases_from_device if is_g2 else ctx.g1_bases_from_device)(pts, m)
            del pts
            ctx.bases_precompute(hs_, 0)
            sc = torch.empty(4 * m, dtype=torch.int64, device="cuda")
            ctx.fr_random_device(sc, m, SEED_SCALARS, lo)
            sms, _, _ = timed_loop(lambda: result.__setitem__("s" + tag, msm_sharded(ctx, None, sc, m, g2=is_g2, handle=hs_)), args.steps, 2)
            dumps[f"strong_{tag}_msm"] = result["s" + tag]
            ctx.bases_free(hs_)
            del sc
            torch.cuda.empty_cache()
            strong[tag + "_ms"] = sms
            strong[tag + "_points_per_s"] = n / (sms / 1e3)
            # the same MSM on ONE GPU, in the same run (rank 0 alone; the other ranks wait at the barrier)
            if not args.no_strong_n1:
                one = None
                if rank == 0:
                    pts = torch.empty(w * n, dtype=torch.int64, device="cuda")
                    (ctx.g2_chain_device if is_g2 else ctx.g1_chain_device)(pts, 0, n, k, d)
                    h1 = (ctx.g2_bases_from_device if is_g2 else ctx.g1_bases_from_device)(pts, n)
                    del pts
                    ctx.bases_precompute(h1, 0)
                    sc1 = torch.empty(4 * n, dtype=torch.int64, device="cuda")
                    ctx.fr_random_device(sc1, n, SEED_SCALARS, 0)
                    fn1 = ctx.g2_msm_resident_device if is_g2 else ctx.g1_msm_resident_device
                    for _ in range(2):
                        result["one" + tag] = fn1(h1, sc1, n)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    reps = args.steps
                    e0.record()
                    for _ in range(reps):
                        fn1(h1, sc1, n)
                    e1.record()
                    torch.cuda.synchronize()
                    one = e0.elapsed_time(e1) / reps
                    ctx.bases_free(h1)
                    del sc1
                    torch.cuda.empty_cache()
                    strong[tag + "_one_gpu_ms_same_run"] = one
                    strong[tag + "_speedup_vs_one_gpu"] = one / sms
                    strong[tag + "_equals_one_gpu_result"] = bool(result["one" + tag] == result["s" + tag])
                barrier()
            if rank == 0 and not args.no_verify:
                ok = bool(closed_form(n, SEED_SCALARS, g2=is_g2) == result["s" + tag])
                strong[tag + "_verified_vs_oracle"] = ok
                if not ok:
                    raise SystemExit(f"bench.py: sharded {tag} MSM differs from the oracle's closed form")

    # ---- NTT half of the metric: forward + inverse at 2^log_n, resident, K steps each
    ntt = None
    if not args.no_ntt:
        d_ntt = torch.empty(4 * n, dtype=torch.int64, device="cuda")
        ctx.fr_random_device(d_ntt, n, SEED_NTT, start, eb.SCALARS_MONT)
        ref = d_ntt.clone()
        rows = torch.from_numpy(np.sort(np.random.default_rng(SEED_DUMP).choice(n, min(n, DUMP_ELEMS), replace=False)))

        def sample(t):
            return t.view(n, 4)[rows.to(t.device)].cpu().numpy().view(np.uint8)
        fwd_ms, fl, _ = timed_loop(lambda: ctx.fr_ntt_device(d_ntt, log_n, 0), args.steps, args.warmup)
        dumps["ntt_forward"] = sample(d_ntt)
        d_ntt.copy_(ref)
        ctx.fr_ntt_device(d_ntt, log_n, 0)
        inv_ms, _, _ = timed_loop(lambda: ctx.fr_ntt_device(d_ntt, log_n, eb.NTT_INVERSE), args.steps, args.warmup)
        dumps["ntt_inverse"] = sample(d_ntt)
        # round trip check on fresh data
        d_ntt.copy_(ref)
        ctx.fr_ntt_device(d_ntt, log_n, 0)
        ctx.fr_ntt_device(d_ntt, log_n, eb.NTT_INVERSE)
        ok = bool(torch.equal(d_ntt, ref))
        if not ok:
            raise SystemExit("bench.py: iNTT(NTT(a)) != a")
        ntt_bytes = 64 * n
        profn = ncu_profile("ntt_forward_2_24") if log_n == 24 else None
        ntt = {"metric": "fr_ntt_elems_per_sec", "value": world * n / (fwd_ms / 1e3), "unit": "elements/s", "forward_ms": fwd_ms, "inverse_ms": inv_ms,
               "inverse_value": world * n / (inv_ms / 1e3), "roundtrip_ok": ok, "launches_per_transform": fl // max(1, args.steps),
               "roofline": {"bound": "hbm", "achieved": ntt_bytes / (fwd_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": ntt_bytes / (fwd_ms / 1e3) / 1e9 / peak,
                            "traffic": (profn["dram_bytes_read"] + profn["dram_bytes_write"]) if profn else None,
                            "binding_roofline": {"bound": "fmaheavy pipe: modular products per element counted from the schedule (at 2^24: 3 passes x 3.0 stage-twiddle products after the trivial ones + 1 inter-pass product in passes 2 and 3 = 11; 12 without the last pass's direct twiddle table)", "peak_products_per_s": modmul_peak,
                                                 "products_per_element": ntt_products_per_element(log_n, int(os.environ.get("B200ZK_NTT_FULL_TW") or 26)), "frac": ntt_products_per_element(log_n, int(os.environ.get("B200ZK_NTT_FULL_TW") or 26)) * n / (fwd_ms / 1e3) / modmul_peak,
                                                 "ncu_sm__pipe_fmaheavy_cycles_active_pct": (profn.get("fmaheavy_pct") or profn.get("fmaheavy_pct_elapsed")) if profn else None},
                            "note": "whole transform (all passes); algorithmic bytes = 64*n; traffic = sum of the passes' dram bytes (profiles/r2_ncu_kernels.json) or null"}}
        # end to end through the host-buffer C-ABI call: pinned host buffer in, transformed in place, copies included
        if not args.no_e2e and world == 1:
            h_ntt = torch.empty(4 * n, dtype=torch.int64).pin_memory()
            h_ntt.copy_(ref)
            wall = wall_loop(lambda: ctx.fr_ntt(h_ntt, log_n, 0), args.steps, 1)
            dumps["ntt_forward_e2e"] = sample(h_ntt)
            ntt["e2e"] = {"value": n / wall, "unit": "elements/s", "ms_per_step": wall * 1e3, "h2d_bytes_per_step": 32 * n, "d2h_bytes_per_step": 32 * n,
                          "api": "b200zk_fr_ntt (pinned host buffer, in place): PCIe-bound, 2 x 512 MiB per transform"}
            del h_ntt
        del d_ntt, ref
    del d_scalars
    torch.cuda.empty_cache()

    # ---- config #5: Groth16-shaped wrap (7 NTT + quotient + 4 G1 MSM + 1 G2 MSM) through B200Backend.prove
    proof = None
    if not args.no_proof:
        from ethrex_b200.backend import B200Backend, ProofFormat, log_proved
        from ethrex_b200.groth16 import SyntheticWrapCircuit
        t0 = time.perf_counter()
        circuit = SyntheticWrapCircuit(ctx, args.proof_log_n, precompute=True, rank=rank, world=world)
        ctx.synchronize()
        setup_s = time.perf_counter() - t0
        backend = B200Backend(ctx, circuit)
        backend.prove({"batch": 0})  # warm-up (workspaces, twiddles)
        times, digests, pl0 = [], [], ctx.launch_count
        reps = args.steps
        for i in range(reps):
            barrier()
            pr, dt = backend.prove_timed({"batch": i + 1}, ProofFormat.GROTH16)
            times.append(max_over_ranks(dt))
            digests.append(pr.proof.hex()[:16])
        dumps["groth16_proof"] = pr.proof
        proof_launches = (ctx.launch_count - pl0) // reps
        # same bytes on every rank (the fold is replicated)
        if world > 1:
            got = [None] * world
            dist.all_gather_object(got, digests[-1])
            if len(set(got)) != 1:
                raise SystemExit("bench.py: ranks disagree on the proof bytes")
        sep_ms = None
        if world == 1 and not args.no_proof_separate:  # the pre-ABI-v2 sequence (five read-back MSMs, host assembly), same circuit
            ser = backend.serialize_input({"batch": reps})
            circuit.prove_separate(ser)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            p2, _ = circuit.prove_separate(ser)
            sep_ms = 1e3 * (time.perf_counter() - t1)
            assert p2.hex()[:16] == digests[-1]
        circuit.close()
        med = sorted(times)[len(times) // 2]
        proof = {"metric": "groth16_wrap_prove_wall_ms", "value": 1e3 * med, "unit": "ms", "higher_is_better": False,
                 "domain_log2": args.proof_log_n, "proving_key_setup_s": setup_s, "n_gpus": world, "proof_prefix": digests[-1], "gpu_launches_per_proof": proof_launches,
                 "api": "B200Backend.prove -> ONE b200zk_groth16_commit call (device inputs), one synchronisation" if world == 1 else
                        "B200Backend.prove -> dealt NTTs (3 broadcasts), b200zk_groth16_commit_partial, ONE all_gather of 768-byte blocks, b200zk_groth16_fold",
                 "separate_calls_ms": sep_ms, "timed_log_line": log_proved(reps, med),
                 "work": "3 iNTT + 3 coset NTT + quotient + 1 coset iNTT, 4 G1 MSM + 1 G2 MSM (synthetic R1CS, chain proving key, no blinding; STARK stage excluded)",
                 "real_input_leg": "absent: decoding fixtures/cache/rpc_prover/cache_hoodi_1265656.json into a witness needs the Rust ProgramInput types and the zkVM's "
                                   "wrap circuit, neither available here; the witness is derived deterministically from the serialized input instead"}
        if rank == 0 and world == 1 and not args.no_cpu:
            cs, ct, cb = cpu_proof_pipeline(args.cpu_proof_log_n)
            proof["cpu"] = {"wall_s": cs, "cores": ct, "domain_log2": args.cpu_proof_log_n, "kind": "port", "breakdown": cb,
                            "sample": f"the same pipeline on the CPU oracle at domain 2^{args.cpu_proof_log_n} (proving key generated outside the timed region); "
                                      f"the GPU line above is domain 2^{args.proof_log_n}"}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only), bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, dt, cores, _, (cpts, cs_, ck, cd) = cpu_msm_sample(args.cpu_log_n)
        ntt_rate, ntt_dt = cpu_ntt_sample(min(22, log_n))
        one_log = min(args.cpu_log_n, 18)
        r1, dt1, _, _, _ = cpu_msm_sample(one_log, threads=1)
        n1_rate, n1_dt = cpu_ntt_sample(min(20, log_n), threads=1)
        g2_log = min(args.cpu_log_n, 20)
        g2pts = orc.g2_chain(1 << g2_log, ck, cd)
        t0 = time.perf_counter()
        orc.g2_msm(g2pts, cs_[: 1 << g2_log], 0, 0)
        g2dt = time.perf_counter() - t0
        cpu = {"value": rate, "unit": "points/s", "cores": cores, "kind": "port",
               "sample": f"2^{args.cpu_log_n}-point slice of the same workload, {dt:.2f} s, Pippenger c={orc.lib().orc_msm_window(1 << args.cpu_log_n)} (ark-ec 0.5.0 rule), "
                         "window x chunk parallel over all host threads",
               "single_thread": {"value": r1, "unit": "points/s", "sample": f"2^{one_log} points, {dt1:.2f} s; ethrex's lockfile builds ark-ec WITHOUT rayon (SURVEY.md 0.4): this is the reference's real configuration",
                                 "ntt": {"value": n1_rate, "unit": "elements/s", "sample": f"2^{min(20, log_n)} forward NTT, {n1_dt:.2f} s"}},
               "g2": {"value": (1 << g2_log) / g2dt, "unit": "points/s", "sample": f"2^{g2_log}-point G2 MSM, {g2dt:.2f} s, all host threads"},
               "ntt": {"value": ntt_rate, "unit": "elements/s", "sample": f"2^{min(22, log_n)} forward NTT, {ntt_dt:.2f} s"}}

    if rank == 0:
        line = {
            "metric": "bn254_g1_msm_points_per_sec", "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "step_ms": msm_step_stats, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 Montgomery (254-bit modular integer)", "data": "synthetic",
            "config": {"workload": f"2^{log_n}-point BN254 G1 MSM per GPU (chain bases P_i=(k+i*d)G, uniform Fr scalars), bases+scalars resident in HBM",
                       "points_per_gpu": n, "total_points": world * n, "l2": "inputs (1.6 GB/GPU) larger than L2; no flush needed",
                       "multi_gpu": "point-split, NCCL all_gather of 128-B XYZZ partials + local fold" if world > 1 else "single GPU",
                       "bases": "resident 13-window table (b200zk_bases_precompute, one-off per proving key: table_setup_s; the table-free figure is plain_bases)" if not args.no_precompute else "plain resident bases",
                       "table_setup_s": table_setup_s, "source_hash": source_hash()},
            "verified_vs_oracle": verified, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "e2e": e2e, "plain_bases": plain,
            "g2": g2, "strong": strong, "ntt": ntt, "proof": proof, "cpu_baseline": cpu,
        }
        emit_result(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=24)
    ap.add_argument("--cpu-log-n", type=int, default=22, help="size of the CPU-arm sample (2^k points)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ntt", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-proof", action="store_true")
    ap.add_argument("--proof-log-n", type=int, default=24, help="domain size of the synthetic Groth16 wrap (config #5)")
    ap.add_argument("--cpu-proof-log-n", type=int, default=18, help="domain of the CPU-oracle run of the same pipeline (bounded sample)")
    ap.add_argument("--no-g2", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-strong-n1", action="store_true", help="skip the one-GPU run of the strong-scaling MSM on rank 0")
    ap.add_argument("--no-plain", action="store_true")
    ap.add_argument("--no-proof-separate", action="store_true")
    ap.add_argument("--no-precompute", action="store_true", help="plain resident bases (no 2^(cw) P_i table)")
    ap.add_argument("--window", type=int, default=0, help="force the MSM window bits (0 = automatic)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each timed path computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
