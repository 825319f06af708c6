#!/usr/bin/env python
"""bench.py -- fp64 block-matmul GFLOP/s at N=16384 (BASELINE.json metric), 1..8 B200.

  python bench.py --gpus N --steps K --warmup W            our arm  (CUDA, through the C ABI)
  python bench.py --impl reference --gpus N ...            reference arm: the reference algorithm
                                                           restated on the box's host cores (oracle/)
  python bench.py --steps K --warmup W --dump-outputs DIR  also writes a fixed sample of blocks of the
                                                           last timed step's product to DIR/*.npy

A "step" is one full C = A * B over the whole block matrix.  `value` is measured with the inputs
resident in HBM; `e2e` is the same multiply through the public Dataset API with HOST buffers
(host->device copies of every A and B block and device->host copies of every C block inside the
timed region).  Prints ONE JSON line on rank 0.
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

N_DEFAULT, BLK_DEFAULT = 16384, 1024
METRIC = "fp64 block-matmul GFLOP/s at N=16384"
UNIT = "GFLOP/s"


def fp64_peak_tflops():
    """Roofline denominator for the fp64 tensor pipe: MEASURED_PEAKS.json has no fp64 entry, so the
    measured DMMA peak of tools/fp64_peak.cu (profiles/fp64_peaks_r01.jsonl) is used."""
    path = os.path.join(ROOT, "profiles", "fp64_peaks_r01.jsonl")
    best, src = None, None
    try:
        for line in open(path):
            d = json.loads(line)
            if d.get("bench") == "dmma_sustained":
                best, src = d["tflops"], "profiles/fp64_peaks_r01.jsonl dmma_sustained (measured on this pool's B200; MEASURED_PEAKS.json has no fp64 entry)"
    except OSError:
        pass
    if best is None:
        best, src = 37.2, "nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz (fallback: no measured file)"
    return best, src


def dram_traffic_per_launch(n: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the GEMM kernel at this N from the committed ncu capture
    (profiles/gemm_traffic_r01.json), or None when no capture exists for this size."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic_r01.json")))
        e = d.get(str(n))
        return None if e is None else {"bytes": e["dram_read_bytes"] + e["dram_write_bytes"], "algorithmic_bytes": 3 * n * n * 8,
                                       "unit": "bytes per launch", "source": e.get("source", "ncu")}
    except (OSError, ValueError, KeyError):
        return None


def tc_traffic_per_launch(n: int, moduli: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one ozaki2_gemm_2sm_kernel launch at this N and moduli count, from the
    committed `ncu --set full` capture (profiles/gemm_traffic_r02.json), or None when no capture exists for this configuration.
    Algorithmic bytes of the launch: the int8 residues of both operands read once (2 x T x N^2) + the residue planes written (T x N^2)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic_r02.json")))
        e = d.get(f"{n}x{moduli}")
        if e is None:
            return None
        scale = e.get("total_tiles", 1) / e.get("captured_tiles", 1)   # the capture holds one piece of the multiply's tile list
        return {"bytes": (e["dram_read_bytes"] + e["dram_write_bytes"]) * scale, "algorithmic_bytes": 3 * moduli * n * n,
                "captured_launch_bytes": e["dram_read_bytes"] + e["dram_write_bytes"], "captured_tiles": e.get("captured_tiles"),
                "total_tiles": e.get("total_tiles"), "l2_hit_rate_pct": e.get("l2_hit_rate_pct"),
                "unit": "bytes per step (all pieces of the multiply's tile list)", "source": e.get("source", "ncu")}
    except (OSError, ValueError, KeyError, TypeError, ZeroDivisionError):
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.mark_at = index, None, [], 0

    def mark(self):
        """Call at the start of the timed region: only samples from here on are reported (the sampler is
        started earlier so that nvidia-smi is already streaming when a short timed region begins)."""
        self.mark_at = len(self.lines)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines[self.mark_at:]
        note = None
        if not lines and self.lines:   # timed region shorter than one sampling period: report the closest samples
            lines, note = self.lines[-3:], "timed region shorter than the 100 ms sampling period; last warm-up samples reported"
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
               "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference ALGORITHM restated on host cores (oracle/)
#
# Both legs run in a SUBPROCESS (`bench.py --_cpu-worker ...`) whose environment pins every BLAS / OpenMP pool to one
# thread BEFORE numpy loads, and whose parallelism is one forked worker PROCESS per host core.  (Round 1 ran 128 Python
# threads into the numpy-bundled OpenBLAS, which is built for 64: "precompiled NUM_THREADS exceeded" -> heap corruption
# -> rc 134 / 139 on the 128-thread GPU hosts, and a 4.5x swing of the reported baseline.)  The GPU process itself never
# runs the CPU legs.
# ------------------------------------------------------------------------------------------------
_W = {}


def host_cores() -> int:
    """Cores this process may actually use: the affinity mask, capped by the cgroup CPU quota (a 1-GPU lease of the 128-thread
    GPU host gets a fraction of its CPUs: round 1 read 353 GFLOP/s there and 1600 on the 8-GPU lease of the same host class)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]           # cgroup v2
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())   # cgroup v1
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def _cpu_task(ij):
    """One Spark task of matrixMultiplyGeneral = one output block (i, j): for every k the MLMatrixSerializer copy-in of
    A(i,k) and B(k,j) (:50-69), a fresh C + dgemm per pair (MLMatrix.multiply :100-104 -> BLAS.gemm), the pairwise
    LocalMatrix.add of reduceByKey (:255), and the serializer copy-out (:26-48)."""
    O, nb, A, B = _W["O"], _W["nb"], _W["A"], _W["B"]
    i, j = ij
    acc = None
    for k in range(nb):
        a = O.deserialize(O.serialize(A[(i + k) % nb]))
        b = O.deserialize(O.serialize(B[(k + j) % nb]))
        p = O.matrixMultiplication(a, b)
        acc = p if acc is None else O.add(acc, p)
    return float(O.serialize(acc)[5][0])


def _cpu_worker_main(mode: str, n: int, blk: int, steps: int, warmup: int, budget_s: float):
    """Runs inside the subprocess; prints one JSON document."""
    import numpy as np
    nb = n // blk
    cores = host_cores()
    if mode == "f2j":
        from oracle import c_port
        if not c_port.available():
            print(json.dumps({"error": "oracle/liboracle.so not built"}))
            return
        threads = c_port.max_threads()
        ntasks = min(nb * nb, threads)
        rng = np.random.default_rng(7)
        uniq = [rng.random(blk * blk) for _ in range(2 * nb)]          # block values do not change dgemm's speed
        A = [uniq[(i + k) % nb] for i in range(nb) for k in range(nb)]
        B = [uniq[nb + (k + j) % nb] for k in range(nb) for j in range(nb)]
        t0 = time.perf_counter()
        c_port.block_multiply_f2j(A, B, nb, blk, 1, 1, 1)              # calibrate: one block pair, one thread
        t_pair = time.perf_counter() - t0
        nk = max(1, min(nb, int(budget_s / max(t_pair * 6.0, 1e-3))))   # all-core runs are ~3x slower per pair than one thread alone
        t0 = time.perf_counter()
        c_port.block_multiply_f2j(A, B, nb, blk, ntasks, threads, nk)
        wall = time.perf_counter() - t0
        fl = ntasks * 2.0 * blk ** 3 * nk
        print(json.dumps({"value": fl / wall / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                          "sample": f"{ntasks} of {nb * nb} output blocks x first {nk} of {nb} k-blocks in {wall:.1f} s, reference-BLAS "
                                    f"(F2J-equivalent) dgemm loop nest, {threads} OpenMP threads (oracle/oracle.c)"}))
        return
    import multiprocessing as mp
    from oracle import matrel_oracle as O
    rng = np.random.default_rng(42)
    # timing inputs: U(0,1) like DenseMatrix.rand (values do not change dgemm's speed); 2 nb distinct blocks are shared
    # copy-on-write by the forked workers and rotated so that every task touches nb different A and nb different B blocks
    _W.update(O=O, nb=nb,
              A=[O.DenseMatrix(blk, blk, rng.random(blk * blk)) for _ in range(nb)],
              B=[O.DenseMatrix(blk, blk, rng.random(blk * blk)) for _ in range(nb)])
    task_flops = 2.0 * blk * blk * blk * nb
    _cpu_task((0, 0))                                          # warm-up (untimed)
    t0 = time.perf_counter()
    _cpu_task((0, 0))
    t1 = time.perf_counter() - t0                              # one single-threaded task on an otherwise idle host
    # under full load a task runs ~2-4x slower than alone (shared L3 / DRAM bandwidth): size the sample for that
    waves = max(1, int(budget_s / max(t1 * 3.0, 1e-3)))
    ntasks = min(nb * nb, cores * waves)
    nproc = min(cores, ntasks)
    todo = [(t // nb, t % nb) for t in range(ntasks)]
    out = []
    with mp.get_context("fork").Pool(nproc) as pool:
        pool.map(_cpu_task, todo[:nproc])                      # every worker process has started and touched its pages
        for s in range(warmup + steps):
            t0 = time.perf_counter()
            res = pool.map(_cpu_task, todo, chunksize=1)
            wall = time.perf_counter() - t0
            if s >= warmup:
                out.append({"seconds": wall, "flops": ntasks * task_flops, "checksum": res[0]})
    tot_f = sum(r["flops"] for r in out)
    tot_t = sum(r["seconds"] for r in out)
    print(json.dumps({"value": tot_f / tot_t / 1e9, "unit": UNIT, "cores": int(nproc), "kind": "port",
                      "sample": f"{ntasks} of {nb * nb} output blocks of the {n}x{n}/{blk} multiply per step, {len(out)} timed step(s) "
                                f"of {tot_t / max(1, len(out)):.1f} s: one single-threaded task (process) per output block, {nproc} in flight "
                                f"(host cores={cores}); per pair: serializer copy-in, fresh C + OpenBLAS dgemm (1 thread), LocalMatrix.add; "
                                f"a single task on the idle host = {t1:.2f} s ({task_flops / t1 / 1e9:.1f} GFLOP/s/core)",
                      "seconds": tot_t, "flops": tot_f, "steps": len(out), "checksum": out[0]["checksum"] if out else None}))


def _run_cpu_worker(mode: str, n: int, blk: int, steps: int, warmup: int, budget_s: float, timeout_s: float = 1500.0):
    env = dict(os.environ)
    cores = host_cores()
    one = "1" if mode != "f2j" else str(cores)
    for k in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS", "VECLIB_MAXIMUM_THREADS"):
        env[k] = one
    if mode != "f2j":
        env["OPENBLAS_NUM_THREADS"] = "1"
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):   # not a torchrun rank
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--_cpu-worker", mode, "--n", str(n), "--blk", str(blk),
           "--steps", str(steps), "--warmup", str(warmup), "--cpu-budget", str(budget_s)]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout_s, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"cpu worker ({mode}) rc={r.returncode}: {(r.stderr or r.stdout)[-400:]}")
    return json.loads(lines[-1])


def cpu_reference_sample(n: int, blk: int, budget_s: float = 20.0, steps: int = 1, warmup: int = 0):
    """matrixMultiplyGeneral restated on the host cores the way Spark local[*] runs it: one task per output block (i, j),
    one single-threaded worker process per host core.  Bounded sample of the N x N workload (as many output blocks as fit
    the time budget, the whole multiply on a 128-core host); GFLOP/s = sample flops / wall seconds.  Upper bound on the
    reference's speed: no Spark scheduling, shuffle, Kryo or GC is modelled, and dgemm is OpenBLAS (the best case a
    netlib-native install reaches)."""
    return _run_cpu_worker("port", n, blk, steps, warmup, budget_s)


def cpu_f2j_sample(n: int, blk: int, budget_s: float = 8.0):
    """Same algorithm with the pure-loop reference-BLAS dgemm (what netlib-java's F2jBLAS runs when no native BLAS is
    installed = stock Spark 2.1.0), oracle/oracle.c, OpenMP threads = host cores; one wave of output blocks."""
    return _run_cpu_worker("f2j", n, blk, 1, 0, budget_s)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, blk = args.n, args.blk
    # each step = a bounded sample of the workload; the whole --steps/--warmup run is sized to end within ~2.5 minutes
    per_step_budget = max(2.0, 150.0 / max(1, args.steps + args.warmup))
    r = cpu_reference_sample(n, blk, budget_s=per_step_budget, steps=args.steps, warmup=args.warmup)
    v = r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * (2.0 * n ** 3 / (v * 1e9)), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{n}x{n} fp64 dense multiply, {blk}-block (reference algorithm on host cores)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def tc_peaks():
    """Measured tcgen05 peaks of tools/tc_peak.cu (profiles/tc_peaks_r02.jsonl): {bench: value}."""
    out = {}
    try:
        for line in open(os.path.join(ROOT, "profiles", "tc_peaks_r02.jsonl")):
            if line.startswith("{"):
                d = json.loads(line)
                out[d["bench"]] = d["value"]
    except (OSError, ValueError, KeyError):
        pass
    return out


def int8_peak_tops():
    pk = tc_peaks()
    if "tcgen05_i8_sustained" in pk:
        return pk["tcgen05_i8_sustained"], ("profiles/tc_peaks_r02.jsonl tcgen05_i8_sustained (tools/tc_peak.cu: back-to-back 128x256x32 kind::i8 MMAs "
                                            "on shared-memory operands, all SMs, ~3 s; MEASURED_PEAKS.json has no int8 entry)")
    try:
        bf16 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]
        return 2.0 * bf16, "2 x MEASURED_PEAKS.json bf16_tflops_sustained (int8 dense = 2 x bf16 dense on this part; no int8 microbenchmark file)"
    except (OSError, ValueError, KeyError):
        return 2.0 * 1400.0, "2 x the profiling guide's sustained bf16 fallback (1.4 PFLOP/s)"


def time_multiply(torch, stream, A, B, n, blk, steps, keep_last=False):
    """Mean ms per step over `steps` timed multiplies; with keep_last, also the product of the last step (else None)."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    last = None
    for i, (e0, e1) in enumerate(evs):
        e0.record(stream)
        C = A.matrixMultiply(n, n, B, n, n, blk)
        e1.record(stream)
        if keep_last and i == steps - 1:
            last = C
        del C
    torch.cuda.synchronize()
    ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    return sum(ms) / len(ms), last


DUMP_BUDGET_BYTES = 64 * 10 ** 6


def dump_outputs(C, out_dir):
    """Writes a fixed sample of the blocks of the product C, as a caller collects them, to out_dir/C_<rid>_<cid>.npy
    (float64, numRows x numCols): the first and the last block, then blocks in an order drawn by a generator with a fixed
    seed, as many as fit DUMP_BUDGET_BYTES in all.  The same arguments dump the same blocks.  Returns the written
    [rid, cid] list and the bytes written."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    ids = sorted(C.block_ids())
    order = [ids[0], ids[-1]] + [ids[k] for k in np.random.default_rng(0).permutation(len(ids))]
    written, total = [], 0
    for rid, cid in dict.fromkeys(order):
        m = np.ascontiguousarray(C.get_block(rid, cid).to_numpy(), dtype=np.float64)
        if total + m.nbytes + 128 > DUMP_BUDGET_BYTES:    # 128: the .npy header
            if written:
                break
            m = np.ascontiguousarray(m[:, :max(1, (DUMP_BUDGET_BYTES - 128) // (8 * m.shape[0]))])   # one block over budget: its leading columns
        path = os.path.join(out_dir, f"C_{rid}_{cid}.npy")
        np.save(path, m)
        written.append([rid, cid])
        total += os.path.getsize(path)
    return written, total


def run_ours(args):
    import numpy as np
    import torch
    import matrel_b200 as mb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    n, blk = args.n, args.blk
    nb = n // blk
    flops = 2.0 * n ** 3

    if world > 1:
        from matrel_b200 import distributed as dist_mm
        line = dist_mm.bench_main(args, METRIC, UNIT, fp64_peak_tflops, ClockSampler, cpu_reference_sample, int8_peak_tops)
        if line is not None:   # rank 0
            # the per-rank sampled blocks are checked against numpy fp64 on the host (= the oracle's dgemm), MAX over ranks
            line["max_rel_err_vs_oracle"] = line["check"]["max_rel_err_vs_host_fp64"]
            print(json.dumps(line), flush=True)
        return

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        s = mb.MatfastSession(device=local_rank, stream=stream.cuda_stream)
        s.set_option("gemm_algo", args.algo)
        s.set_option("crt_moduli", args.crt_moduli)
        A = s.rand(n, n, blk, 42)
        B = s.rand(n, n, blk, 43)
        s.sync()

        # ---- device-resident: value (CUDA events on the launching stream around whole operator calls)
        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(args.warmup):
            C = A.matrixMultiply(n, n, B, n, n, blk)
            del C
        s.sync()
        s.reset_stats()
        torch.cuda.synchronize()
        sampler.mark()
        t_wall0 = time.perf_counter()
        ms_per_step, C_last = time_multiply(torch, stream, A, B, n, blk, args.steps, keep_last=bool(args.dump_outputs))
        t_wall = time.perf_counter() - t_wall0
        clocks = sampler.stop()
        st = s.stats()
        dump = None
        if args.dump_outputs:
            blocks, nbytes = dump_outputs(C_last, args.dump_outputs)
            dump = {"dir": args.dump_outputs, "blocks": blocks, "bytes": nbytes, "of": "C = A * B of the last timed step"}
            del C_last
        launches_per_step = st["kernel_launches"] / args.steps
        on_tc = st["tc_gemm_launches"] > 0

        # ---- the dominant kernel alone (events inside the library, around its launches)
        s.set_option("time_kernels", 1)
        s.reset_stats()
        reps = max(3, min(args.steps, 10))
        for _ in range(reps):
            C = A.matrixMultiply(n, n, B, n, n, blk)
            del C
        st2 = s.stats()
        moduli_used = int(st2.get("tc_moduli", 0))
        s.set_option("time_kernels", 0)
        dpeak, dpeak_src = fp64_peak_tflops()
        if on_tc:
            kern_ms = st2["tc_gemm_ms_total"] / reps
            ipeak, ipeak_src = int8_peak_tops()
            ach = st2["tc_int8_ops"] / (kern_ms * 1e-3) / 1e12
            tct = tc_traffic_per_launch(n, moduli_used)
            # the engine's plane-capacity rule (csrc/abi_multiply.cpp: plane_cap_tiles, rounded up to an even tile count)
            plane_cap = max(64, (2 << 30) // (max(1, moduli_used) * 128 * 256))
            plane_cap += plane_cap & 1
            tiles_total = (-(-n // 128)) * (-(-n // 256))
            pieces = -(-tiles_total // plane_cap)
            roofline = {"bound": "tensor", "achieved": ach, "peak": ipeak, "unit": "TFLOP/s", "frac": ach / ipeak,
                        "traffic": (tct or {}).get("bytes"), "traffic_detail": tct,
                        "op": "int8 multiply-add x 2 (TOPS) on tcgen05.mma kind::i8, s32 accumulators in TMEM",
                        "kernel": "ozaki2_gemm_2sm_kernel (persistent CTA pairs, TMA -> 6-stage smem ring -> UTCIMMA cta_group::2 256x256x32 -> TMEM -> residue epilogue)",
                        "kernel_ms": kern_ms, "launches_per_step": 1.0,
                        "algorithmic": f"{st2['tc_moduli']} moduli x 2*N^3 = {st2['tc_int8_ops']:.4g} int8 ops per step (all moduli x all tiles; the 2 GiB residue-plane "
                                       f"buffer holds {plane_cap} of the {tiles_total} 128x256 tiles at {moduli_used} moduli, so the step's GEMM is {pieces} back-to-back "
                                       "launch(es) of this kernel and kernel_ms is their sum)",
                        "peak_source": ipeak_src,
                        "fp64_equivalent": {"achieved": flops / (ms_per_step * 1e-3) / 1e12, "dmma_peak": dpeak, "x_dmma_roof": flops / (ms_per_step * 1e-3) / 1e12 / dpeak,
                                            "note": "whole multiply (absmax + residues + int8 GEMM + CRT) as fp64 flop/s against the measured native-fp64 (DMMA) roof"}}
        else:
            kern_ms = st2["gemm_ms_total"] / max(1, st2["gemm_launches"])
            ach = flops / (kern_ms * 1e-3) / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": dpeak, "unit": "TFLOP/s", "frac": ach / dpeak,
                        "traffic": (dram_traffic_per_launch(n) or {}).get("bytes"), "traffic_detail": dram_traffic_per_launch(n),
                        "kernel": "gemm_f64_dmma_kernel<128,128,2,4,5>", "kernel_ms": kern_ms, "launches_per_step": 1.0,
                        "algorithmic": f"2*N^3 = {flops:.4g} flop per launch (whole block multiply, K reduction fused)", "peak_source": dpeak_src}

        # ---- host-side check of the timed configuration: one output block against numpy fp64 on the host
        check = None
        try:
            from threadpoolctl import threadpool_limits
            Ck = A.matrixMultiply(n, n, B, n, n, blk)
            i_, j_ = nb // 2, nb // 3
            with threadpool_limits(limits=16, user_api="blas"):
                want = sum(A.get_block(i_, k).to_numpy() @ B.get_block(k, j_).to_numpy() for k in range(nb))
            got = Ck.get_block(i_, j_).to_numpy()
            check = {"block": [i_, j_], "max_rel_err_vs_host_fp64": float(np.max(np.abs(got - want)) / np.max(np.abs(want)))}
            del Ck
        except Exception as e:
            check = {"error": str(e)[-200:]}

        # ---- the exact native-fp64 kernel (gemm_algo 1, DMMA) beside the headline, with its own roofline fraction
        dmma = None
        if on_tc:
            try:
                s.set_option("gemm_algo", 1)
                for _ in range(2):
                    C = A.matrixMultiply(n, n, B, n, n, blk)
                    del C
                s.sync()
                d_steps = max(3, min(args.steps, 5))
                d_ms, _ = time_multiply(torch, stream, A, B, n, blk, d_steps)
                Cd = A.matrixMultiply(n, n, B, n, n, blk)
                s.set_option("gemm_algo", args.algo)
                Ct = A.matrixMultiply(n, n, B, n, n, blk)
                worst = 0.0
                for key in [(0, 0), (nb // 2, nb // 3), (nb - 1, nb - 1)]:
                    a_, b_ = Cd.get_block(*key).values, Ct.get_block(*key).values
                    worst = max(worst, float(np.max(np.abs(a_ - b_)) / np.max(np.abs(a_))))
                del Cd, Ct
                tr = dram_traffic_per_launch(n)
                dmma = {"algo": "gemm_algo 1: gemm_f64_dmma_kernel (TMA -> 5-stage ring -> mma.sync m8n8k4 f64)", "value": flops / (d_ms * 1e-3) / 1e9,
                        "unit": UNIT, "ms_per_step": d_ms, "steps": d_steps,
                        "roofline": {"bound": "tensor", "achieved": flops / (d_ms * 1e-3) / 1e12, "peak": dpeak, "unit": "TFLOP/s",
                                     "frac": flops / (d_ms * 1e-3) / 1e12 / dpeak, "traffic": (tr or {}).get("bytes"), "peak_source": dpeak_src},
                        "max_rel_dev_tcgen05_vs_dmma": worst}
            except Exception as e:
                dmma = {"error": str(e)[-200:]}
            finally:
                s.set_option("gemm_algo", args.algo)

        # ---- end to end through the public API with pinned HOST buffers
        hostA = {k: A.get_block(*k) for k in A.block_ids()}
        hostB = {k: B.get_block(*k) for k in B.block_ids()}
        pin = lambda m: torch.from_numpy(m.values).pin_memory().numpy()  # noqa: E731
        pA = [mb.MatrixBlock(i, j, mb.DenseMatrix(m.numRows, m.numCols, pin(m), m.isTransposed)) for (i, j), m in hostA.items()]
        pB = [mb.MatrixBlock(i, j, mb.DenseMatrix(m.numRows, m.numCols, pin(m), m.isTransposed)) for (i, j), m in hostB.items()]
        outbuf = {(i, j): torch.empty(blk * blk, dtype=torch.float64).pin_memory().numpy() for i in range(nb) for j in range(nb)}
        del hostA, hostB
        h2d = sum(b.matrix.values.nbytes for b in pA) + sum(b.matrix.values.nbytes for b in pB)
        d2h = sum(v.nbytes for v in outbuf.values())

        rowsA = {}
        colsB = {}
        for b_ in pA:
            rowsA.setdefault(b_.rid, []).append(b_)
        for b_ in pB:
            colsB.setdefault(b_.cid, []).append(b_)

        def e2e_step():
            # block row t of A and block column t of B are uploaded alternately; every put_block is an async copy on
            # the ingest stream tagged with an event, the multiply launches chunk after chunk as the operands each
            # chunk needs have landed (residues of a block row / column as soon as it is complete, then the int8 GEMM
            # + CRT of the output blocks it unlocks), and finished blocks of C stream back on the egress stream meanwhile
            dbg = os.environ.get("MATREL_E2E_DEBUG")
            tq = [time.perf_counter()]
            dA, dB = s.emptyDataset(), s.emptyDataset()
            for t_ in range(nb):
                dA.put_blocks(rowsA[t_])
                dB.put_blocks(colsB[t_])
            tq.append(time.perf_counter())
            dC = dA.matrixMultiply(n, n, dB, n, n, blk)
            tq.append(time.perf_counter())
            first = True
            for (i, j) in sorted(dC.block_ids(), key=lambda ij: (max(ij), ij)):   # the order the chunks complete in
                dC.get_block(i, j, out=outbuf[(i, j)])
                if first:
                    tq.append(time.perf_counter())
                    first = False
            tq.append(time.perf_counter())
            if dbg:
                print("e2e host timeline ms: puts %.1f  multiply-call %.1f  first-block %.1f  all-blocks %.1f  launches %d" % (
                    (tq[1] - tq[0]) * 1e3, (tq[2] - tq[1]) * 1e3, (tq[3] - tq[2]) * 1e3, (tq[4] - tq[2]) * 1e3,
                    s.stats()["kernel_launches"]), file=sys.stderr, flush=True)
            return dC

        def e2e_time():
            for _ in range(min(args.warmup, 2)):
                e2e_step()
            torch.cuda.synchronize()
            k_ = max(1, min(args.steps, 5))
            t0 = time.perf_counter()
            for _ in range(k_):
                e2e_step()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / k_ * 1e3, k_

        e2e_ms, e2e_steps = e2e_time()
        # the PCIe floor of the step on this box: the same uploads alone
        t0 = time.perf_counter()
        for _ in range(2):
            dA, dB = s.emptyDataset(), s.emptyDataset()
            dA.put_blocks(pA)
            dB.put_blocks(pB)
            dA.wait_ingest()               # host-blocking
            dB.wait_ingest()
            del dA, dB
        ingest_only_ms = (time.perf_counter() - t0) / 2 * 1e3
        checksum = float(outbuf[(0, 0)][0])
        e2e_blk = outbuf[(nb // 2, nb // 3)].copy()
        if isinstance(check, dict) and "error" not in check:
            try:   # the end-to-end result is the same product: compare the same block with the resident run's
                Ck = A.matrixMultiply(n, n, B, n, n, blk)
                ref_blk = Ck.get_block(nb // 2, nb // 3).values
                check["e2e_block_equals_resident"] = bool(np.array_equal(ref_blk, e2e_blk))
                check["e2e_block_max_rel_dev"] = float(np.max(np.abs(ref_blk - e2e_blk)) / np.max(np.abs(ref_blk)))
                del Ck
            except Exception as e:
                check["e2e_error"] = str(e)[-200:]
        if isinstance(dmma, dict) and "error" not in dmma:
            try:
                s.set_option("gemm_algo", 1)
                d_e2e_ms, _ = e2e_time()
                dmma["e2e"] = {"value": flops / (d_e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": d_e2e_ms,
                               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
            except Exception as e:
                dmma["e2e"] = {"error": str(e)[-200:]}
            finally:
                s.set_option("gemm_algo", args.algo)
        s.stop()

    try:
        cpu = cpu_reference_sample(n, blk, budget_s=args.cpu_budget)
        for k_ in ("seconds", "flops", "checksum", "steps"):
            cpu.pop(k_, None)
    except Exception as e:  # the CPU leg runs in its own process; whatever happens there, the GPU line is printed
        cpu = {"value": None, "unit": UNIT, "cores": host_cores(), "kind": "port", "sample": "cpu worker failed", "error": str(e)[-300:]}
    try:
        cpu["f2j"] = cpu_f2j_sample(n, blk)
    except Exception as e:  # the secondary baseline must never take the bench line down
        cpu["f2j"] = {"error": str(e)[-300:]}
    algo_name = ("auto -> Ozaki-II on tcgen05 (int8 residue GEMMs modulo %d coprime moduli%s + CRT; device-side guard, DMMA fallback)"
                 % (moduli_used, "" if args.crt_moduli else ", count chosen from K: operand truncation 2^-alpha x sqrt(K) <= K 2^-54") if on_tc else "dmma_fp64")
    line = {
        "metric": METRIC, "value": flops / (ms_per_step * 1e-3) / 1e9, "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{n}x{n} fp64 dense multiply, {blk}-block, 1xB200 (BASELINE metric size)",
                   "inputs": "U(0,1) java.util.Random streams, every block present, column-major",
                   "l2": f"inputs 2 x {n * n * 8 / 2**30:.0f} GiB + output {n * n * 8 / 2**30:.0f} GiB >> 126 MB L2; no flush needed",
                   "gemm_algo": algo_name, "wall_ms_per_step": t_wall / args.steps * 1e3, "c00": checksum,
                   "oz2_ksplit_env": os.environ.get("MATREL_OZ2_KSPLIT")},
        "e2e": {"value": flops / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms, "steps": e2e_steps, "ingest_only_ms": ingest_only_ms,
                "note": "ingest_only_ms = the step's host->device copies alone on this box: the PCIe floor of the step"},
        "gpu_launches": int(round(launches_per_step * args.steps)),
        "gpu_launches_per_step": launches_per_step,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "check": check,
        "dmma_fp64": dmma,
    }
    if dump is not None:
        line["dump_outputs"] = dump
    print(json.dumps(line), flush=True)



# ------------------------------------------------------------------------------------------------
# --workload cfg5: BASELINE configs[4] -- 32768^2 sparse(1 %) x dense fp64, CSR 1024-blocks, on 1 GPU or sharded over N GPUs
# ------------------------------------------------------------------------------------------------
def run_cfg5(args):
    import numpy as np
    import torch
    import matrel_b200 as mb
    from matrel_b200.dataset import grid_multiply_rows, memcpy_d2h, sprand
    from matrel_b200.distributed import GridPlan, ShardedMatrix, stream_barrier

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    n, blk, density = args.n5, 1024, 0.01
    nb = n // blk
    plan = GridPlan(world, n, n, blk)
    r, c = plan.coords(rank)

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    stream = torch.cuda.Stream(device=device)
    with torch.cuda.stream(stream):
        s = mb.MatfastSession(device=local_rank, stream=stream.cuda_stream)
        # A: every block SparseMatrix.sprand(1024, 1024, 0.01, new java.util.Random(seed)) in CSR form, generated on the device.
        # The thin operand is replicated where it is needed (the reference's duplicateCrossPartitions): every rank generates the
        # block rows it owns -- all k of them -- from the same seeds, so no sparse block crosses NVLink.
        Afull = sprand(s, n, n, blk, density, 1000, csr=True)
        A_rows = Afull.filter_blocks(plan.pr, r)
        nnz_total = nb * nb * int(np.ceil(blk * blk * density))
        B = ShardedMatrix.rand(s, plan, rank, 43, device)
        s.sync()
        peers = B.peer_slabs()
        colB = [peers[plan.rank_of(rr, c)] for rr in range(plan.pr)]
        barrier()
        flops = 2.0 * nnz_total * n

        def step():
            return grid_multiply_rows(s, A_rows, n, n, B.sharded, colB)

        for _ in range(args.warmup):
            out = step()
            del out
        barrier()
        s.reset_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local_rank)
        sampler.start()
        sampler.mark()
        e0.record(stream)
        for _ in range(args.steps):
            out = step()
            del out
        e1.record(stream)
        barrier()
        clocks = sampler.stop()
        ms = allmax(e0.elapsed_time(e1) / args.steps)
        st = s.stats()
        s.set_option("time_kernels", 1)
        s.reset_stats()
        for _ in range(3):
            out = step()
            del out
        kern_ms = allmax(s.stats()["gemm_ms_total"] / 3.0)
        s.set_option("time_kernels", 0)
        # correctness: one output block per rank against scipy on the host
        import scipy.sparse as sp
        dC = step()
        mine = plan.owned(rank)
        i, j = mine[len(mine) // 2]
        want = np.zeros((blk, blk))
        buf = np.empty(blk * blk)
        for k in range(nb):
            a = A_rows.get_block(i, k)                       # CSR: colPtrs = row pointers, rowIndices = column indices
            csr = sp.csr_matrix((a.values, a.rowIndices, a.colPtrs), shape=(blk, blk))
            memcpy_d2h(s, peers[plan.owner(k, j)] + plan.slot(k, j) * plan.slot_elems * 8, buf)
            want += csr @ buf.reshape(blk, blk).T
        got = dC.get_block(i, j).to_numpy()
        err = allmax(float(np.max(np.abs(got - want)) / np.max(np.abs(want))))
        del dC
        # end to end: the dense operand and the result cross PCIe (A is 0.13 GB of CSR arrays, ingested once)
        hostB = [(k, B.dataset.get_block(*k)) for k in B.dataset.block_ids()]
        pB = [mb.MatrixBlock(i_, j_, mb.DenseMatrix(m.numRows, m.numCols, torch.from_numpy(m.values).pin_memory().numpy(), False)) for (i_, j_), m in hostB]
        del hostB
        outbuf = {k: torch.empty(blk * blk, dtype=torch.float64).pin_memory().numpy() for k in plan.owned(rank)}
        eB = ShardedMatrix(plan, rank, torch.zeros_like(B.slab), None, s)
        epeers = eB.peer_slabs()
        ecolB = [epeers[plan.rank_of(rr, c)] for rr in range(plan.pr)]
        barrier()

        def e2e_step():
            eB.sharded.put_blocks(pB)
            s.wait_ingest()
            stream_barrier(device)
            dC_ = grid_multiply_rows(s, A_rows, n, n, eB.sharded, ecolB)
            for k in sorted(dC_.block_ids()):
                dC_.get_block(*k, out=outbuf[k])
            stream_barrier(device)

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        k_e2e = max(1, min(args.steps, 3))
        for _ in range(k_e2e):
            e2e_step()
        barrier()
        e2e_ms = allmax((time.perf_counter() - t0) / k_e2e * 1e3)
        h2d = sum(b.matrix.values.nbytes for b in pB) * world
        d2h = sum(v.nbytes for v in outbuf.values()) * world
        s.stop()
    if rank == 0:
        hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
        alg_bytes = (12.0 * nnz_total + 4.0 * (n + nb) * nb + 2 * 8.0 * n * n) / world     # SURVEY 8d compulsory bytes, per rank
        fma_roof = 148 * 16 * 2 * 1.9e9 / 1e12      # shared-memory port: 16 fp64 FMA / clk / SM at ~1.9 GHz
        ach_tf = (flops / world) / (kern_ms * 1e-3) / 1e12
        line = {"metric": f"fp64 sparse(1%) x dense block-matmul GFLOP/s at N={n}", "value": flops / (ms * 1e-3) / 1e9, "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"BASELINE configs[4]: {n}x{n} sparse(1%) x dense fp64, CSR {blk}-blocks, {plan.pr}x{plan.pc} grid over {world}xB200",
                           "inputs": "A blocks SparseMatrix.sprand(1024, 1024, 0.01, java.util.Random(1000 + rid*nb + cid)) as CSR, generated on the device; "
                                     "B U(0,1) java.util.Random streams, column-major",
                           "parallelism": "C-stationary grid; sparse block rows replicated where needed (duplicateCrossPartitions), dense B pulled from the grid column over NVLink",
                           "nnz": nnz_total, "l2": "B panel per rank >> 126 MB L2"},
                "e2e": {"value": flops / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_ms, "steps": k_e2e},
                "gpu_launches": int(st["kernel_launches"] * world), "gpu_launches_per_step_per_rank": st["kernel_launches"] / args.steps,
                "roofline": {"bound": "hbm", "achieved": alg_bytes / (kern_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                             "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / hbm, "traffic": None, "kernel": "spmm2_kernel", "kernel_ms": kern_ms,
                             "algorithmic": f"{alg_bytes:.4g} compulsory bytes per rank per launch (12 nnz + 4 (rows + nb) nb + 16 N^2, SURVEY 8d) / world",
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs",
                             "smem_port": {"achieved_tflops": ach_tf, "roof_tflops": fma_roof, "frac": ach_tf / fma_roof,
                                           "note": "every FMA needs its own 8-byte B element from shared memory: 128 B/clk/SM = 16 FMA/clk/SM is the binding roof"}},
                "clocks": clocks, "check": {"max_rel_err_vs_host_fp64": err, "blocks_checked": world}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_DEFAULT)
    ap.add_argument("--blk", type=int, default=BLK_DEFAULT)
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--ozaki-slices", type=int, default=7)
    ap.add_argument("--algo", type=int, default=0, choices=(0, 1, 2, 4),
                    help="gemm_algo of the headline: 0 = auto (tcgen05 Ozaki-II with the device-side guard), 1 = DMMA fp64")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="N > 1: pieces of block rows / block columns the pipelined end-to-end step uploads and pulls")
    ap.add_argument("--crt-moduli", type=int, default=0, help="Ozaki-II residue moduli (6..16); 0 = chosen by the library from K")
    ap.add_argument("--workload", default="metric", choices=("metric", "cfg5"), help="metric = BASELINE metric (dense N=16384); cfg5 = configs[4]")
    ap.add_argument("--n5", type=int, default=32768, help="matrix size of --workload cfg5")
    ap.add_argument("--pull-chunks", type=int, default=4, help="N > 1: pieces the peer pull of A is cut into")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of blocks of the last step's product C to DIR/C_<rid>_<cid>.npy "
                         "(float64, at most 64 MB in all); single-GPU metric workload")
    ap.add_argument("--_cpu-worker", dest="cpu_worker", default=None, choices=("port", "f2j"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "metric" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is supported for the single-GPU metric workload of --impl ours")
    if args.cpu_worker:
        return _cpu_worker_main(args.cpu_worker, args.n, args.blk, args.steps, args.warmup, args.cpu_budget)
    if args.workload == "cfg5":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the reference arm times the metric workload only (dense N=16384)"}))
            return
        return run_cfg5(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
