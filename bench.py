#!/usr/bin/env python3
"""bench.py -- Groth16 proofs/sec on BLS12-381 at 2^20 constraints (BASELINE.json's metric and configs[2]).

One "step" = one complete proof of the synthetic R1CS (SURVEY.md section 8d): witness map (row evaluation + 7 NTTs) and the
five MSMs (A, B-in-G1, B-in-G2, H, L) plus the O(1) final assembly, through the C ABI of libg16b200.so.

  python bench.py --gpus 1 --steps K --warmup W            own arm (CUDA path)
  python bench.py --impl reference ...                      reference arm: the restated ark CPU path (oracle/) on the host
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   N GPUs: every MSM's (scalar, base) pairs
      are sharded by index range over the ranks (SURVEY.md section 8e), 5 partial points per rank are all-gathered over NCCL,
      every rank assembles the same proof.  Strong scaling: the proof size is fixed as N grows.

Output: ONE JSON line on rank 0 (contract in the task statement) with `roofline`, `cpu_baseline`, `e2e`, `clocks`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA is initialised: see groth16_b200/__init__.py

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def metric_name(a):
    return f"groth16_proofs_per_sec_{a.curve}_2^{a.log_n}"



def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--curve", default="bls12_381")
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads for the CPU arm / cpu_baseline (0 = all)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="synthetic", choices=["synthetic", "dummy"],
                    help="synthetic = non-degenerate R1CS of SURVEY 8d (default, the BASELINE configs); dummy = the reference's "
                         "own benchmark circuit, DummyCircuit with 2^log_n - 100 variables and constraints "
                         "(benches/bench.rs:17-20,41-64): constant witness, a/b queries almost all identity")
    ap.add_argument("--inflight", type=int, default=0, choices=[0, 1, 2],
                    help="proofs in flight per GPU: 1 = one proof at a time; 2 = software pipeline over the two proof slots of a "
                         "context (g16_prove_submit / g16_prove_wait); 0 (default) = 2 up to 2^20 constraints (the next proof fills "
                         "the latency-bound tail of the previous one; single-proof latency is reported next to it), 1 above")
    ap.add_argument("--mode", default="auto", choices=["auto", "shard", "replicas"],
                    help="N > 1: 'shard' splits every MSM of ONE proof over the GPUs (strong scaling, NCCL gather of partial "
                         "points) and is what `value` reports; 'replicas' lets every GPU prove its own proofs (weak scaling, no "
                         "communication: BASELINE config 5) and reports that as `value`; 'auto' (default) = 'shard' for `value` "
                         "and additionally measures the replicas, reported under the secondary key \"replicas\"")
    ap.add_argument("--check-oracle", action="store_true",
                    help="N > 1: rank 0 also proves once with the CPU oracle and compares bit for bit (N = 1 always does, as its cpu_baseline)")
    ap.add_argument("--record", default="", help="also append the JSON line to this file (profiles/r02_bench_*.json)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the proof of the last timed step as DIR/a.npy, b.npy, c.npy (see dump_outputs); the inputs "
                         "depend only on the arguments, so two builds can be compared output for output")
    return ap.parse_args()


def workload_name(a):
    if a.workload == "dummy":
        return (f"{a.curve} DummyCircuit 2^{a.log_n}-100 variables and constraints (the reference's own benchmark, "
                "benches/bench.rs:17-20,41-64: constant witness, near-empty a/b queries), full prover path")
    return f"{a.curve} synthetic R1CS 2^{a.log_n} constraints (non-degenerate, SURVEY 8d), full A/B(G1,G2)/H/L MSM path + witness map"


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe).

    The nvidia-smi process is started BEFORE the warm-up steps: its start-up (process spawn, NVML attaching to every GPU of
    the box) takes driver-wide locks for hundreds of milliseconds, which inside a 0.3 s timed region of an 8-GPU sharded
    run stalled kernel launches on all ranks (profiles/r02_bench_h_bls12_381_20_n8.json: `value` 77 proofs/s under the
    sampler against 137 for the unsampled host-input run of the same process).  Every sample is stamped on arrival and only
    those that fall between mark_begin() and mark_end() are reported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.proc = None
        self.lines = []          # (arrival time, text)
        self.t_begin = self.t_end = None

    def start(self):
        if self.proc:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def wait_ready(self, timeout=5.0):
        """block until the first sample has arrived (nvidia-smi is past its start-up)"""
        t = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t < timeout:
            time.sleep(0.02)

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)   # the sample taken at the end of the region is printed up to one period later
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.proc = None
        t0 = self.t_begin if self.t_begin is not None else 0.0
        t1 = (self.t_end if self.t_end is not None else time.perf_counter()) + 0.12
        inside = [ln for t, ln in self.lines if t0 <= t <= t1]
        window = "timed region"
        if not inside:   # region shorter than one sampling period: the nearest samples (warm-up steps: same load)
            inside = [ln for _, ln in self.lines[-3:]]
            window = "nearest samples (timed region shorter than the 100 ms sampling period)"
        sm, smax, reasons, pw = [], [], set(), []
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(pw), "samples": len(sm),
                "window": window, "reasons": sorted(reasons)}


def host_threads(requested=0):
    """Threads for the CPU arm: min(affinity, cgroup CPU quota) -- the GPU boxes expose 128 logical CPUs under a 16-CPU quota,
    and oversubscribing a quota only adds contention."""
    if requested > 0:
        return requested
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(p) + 0.5)))
    except Exception:
        pass
    return n


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def ncu_summary():
    """Per-launch DRAM traffic / pipe utilisation of the dominant kernel from the committed ncu capture, if present."""
    p = os.path.join(ROOT, "profiles", "accum_kernel_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------------------------
def build_workload(a):
    from groth16_b200.workload import dummy_r1cs, synthetic_r1cs
    t = time.time()
    if a.workload == "dummy":
        k = (1 << a.log_n) - 100
        m, z, pub = dummy_r1cs(a.curve, k, k, seed=a.seed)
    else:
        m, z, pub = synthetic_r1cs(a.curve, a.log_n, seed=a.seed)
    return m, z, pub, time.time() - t


TOXIC = (0x1111111111111111111111, 0x2222222222222222222223, 0x3333333333333333333335, 0x4444444444444444444447,
         0x5555555555555555555559)  # alpha, beta, gamma, delta, tau -- fixed, so every rank mints the same key


def cpu_prove_once(a, g_codec, nq, pk, m, z, r, s, threads):
    """cpu_baseline / reference arm: the oracle's restated ark CPU prover (test infrastructure used as the CPU yardstick)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    t = time.time()
    proof, tms = orc.prove(g_codec.c.cid, nq, pk, m, z, r, s, threads=threads)
    return proof, time.time() - t, tms


def cpu_setup(a, m, threads):
    """Valid CRS for the reference arm minted WITHOUT the CUDA library: the oracle's CPU trusted setup (generator.rs:47-208
    restated in oracle/oracle.cpp) from the same toxic waste and generators as the CUDA arm, hence the very same key."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    from groth16_b200.api import ProvingKey, VerifyingKey     # plain dataclasses; libg16b200.so is NOT loaded by this import
    from groth16_b200.codec import CurveCodec
    from groth16_b200.params import GENERATORS, get_curve
    cp = get_curve(a.curve)
    cd = CurveCodec(cp)
    G = GENERATORS[cp.name]
    k = orc.generate_parameters(cp.cid, cd.nq, m, cd.fr.enc(list(TOXIC)), cd.enc_g1([G["g1"]])[0], cd.enc_g2([G["g2"]])[0], threads)
    vk = VerifyingKey(k["alpha_g1"], k["beta_g2"], k["gamma_g2"], k["delta_g2"], k["gamma_abc_g1"])
    return ProvingKey(vk, k["beta_g1"], k["delta_g1"], k["a_query"], k["b_g1_query"], k["b_g2_query"], k["h_query"], k["l_query"])


# ------------------------------------------------------------------------------------------------------------------
def run_reference(a):
    """`--impl reference`: the reference's CPU implementation of the path.  ark-groth16 itself cannot be built in this
    image (no Rust toolchain, dependencies un-vendored), so the arm times oracle/oracle.cpp, the multi-threaded
    restatement of the ark CPU prover, on all host cores; one step = one full proof of the same workload.  Nothing of the
    CUDA library is loaded in this process: the key comes from the oracle's own CPU setup."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    from groth16_b200.codec import CurveCodec
    from groth16_b200.params import get_curve
    threads = host_threads(a.cpu_threads)
    cp = get_curve(a.curve)
    cd = CurveCodec(cp)
    m, z, pub, _ = build_workload(a)
    t = time.time()
    pk = cpu_setup(a, m, threads)
    t_setup = time.time() - t
    r = cd.fr.enc1(123456789)
    s = cd.fr.enc1(987654321)
    for _ in range(a.warmup):
        cpu_prove_once(a, cd, cd.nq, pk, m, z, r, s, threads)
    t0 = time.time()
    for _ in range(a.steps):
        proof, _, _ = cpu_prove_once(a, cd, cd.nq, pk, m, z, r, s, threads)
    dt = time.time() - t0
    val = a.steps / dt
    # the other CPU schedule, once, outside the timed region: ark-ec parallelises msm_bigint across windows
    old = orc.set_msm_mode(1)
    try:
        proof_w, sec_w, _ = cpu_prove_once(a, cd, cd.nq, pk, m, z, r, s, threads)
    finally:
        orc.set_msm_mode(old)
    assert np.array_equal(proof, proof_w), "window-parallel and chunk-parallel CPU proofs differ"
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, proof, cd.nq)
    line = {
        "impl": "reference", "metric": metric_name(a), "value": val, "unit": "proofs/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64 limbs (255-bit Fr / 381-bit Fq Montgomery integers)", "data": "synthetic",
        "config": {"workload": workload_name(a), "curve": a.curve, "log_n": a.log_n,
                   "pk": "valid CRS minted by the oracle's CPU setup (same toxic waste and generators as the CUDA arm: same key)",
                   "threads": threads, "cpu_setup_s": t_setup},
        "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": threads, "kind": "port",
                         "sample": f"{a.steps} full proofs (restated ark CPU path: chunk-parallel Pippenger, radix-2 FFT)",
                         "threads": threads, "chunk_parallel_s_per_proof": dt / a.steps,
                         "ark_window_parallel_s_per_proof": sec_w,
                         "note": "ark-ec 0.5 parallelises msm_bigint across windows (<= 256/c-way); the timed default is the "
                                 "chunk-parallel schedule, the stronger baseline on many-core hosts; both give the same proof"},
        "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(a, line)


def dump_outputs(d, proof, nq):
    """What a caller of g16_prove receives -- A (G1), B (G2), C (G1) as affine coordinates of nq Montgomery u64 limbs each --
    as float64 arrays a (2, 2*nq), b (4, 2*nq), c (2, 2*nq): one row per coordinate (B: x.c0, x.c1, y.c0, y.c1), every u64
    limb split into its low and high 32-bit word, so that float64 holds every bit exactly."""
    os.makedirs(d, exist_ok=True)
    words = np.ascontiguousarray(proof, dtype="<u8").view("<u4").astype(np.float64).reshape(-1, 2 * nq)
    for name, rows in (("a", slice(0, 2)), ("b", slice(2, 6)), ("c", slice(6, 8))):
        np.save(os.path.join(d, f"{name}.npy"), words[rows])


def emit(a, line):
    out = json.dumps(line)
    print(out, flush=True)
    if a.record:
        os.makedirs(os.path.dirname(os.path.abspath(a.record)) or ".", exist_ok=True)
        with open(a.record, "a") as f:
            f.write(out + "\n")


# ------------------------------------------------------------------------------------------------------------------
def kernel_rev():
    """hash of the kernel sources a committed ncu capture must have been taken with to describe the running code"""
    import hashlib
    h = hashlib.sha256()
    for f in ("fp.cuh", "ec.cuh", "msm.cuh", "msm_ba.cuh", "fp_inv.cuh"):
        with open(os.path.join(ROOT, "groth16_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


INT_PIPE_LANES_PER_CLK_SM = 32      # IMAD.WIDE.U32: one warp instruction per 4 cycles per SM sub-partition (4 per SM)


def run_cuda(a):
    import torch
    import torch.distributed as dist
    from groth16_b200 import Groth16, _lib
    from groth16_b200.params import GENERATORS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (own arm) needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m, z_np, pub, t_work = build_workload(a)
    g = Groth16(a.curve, local)
    cd = g.codec
    nq = g.nq
    G = GENERATORS[g.curve.name]
    want_shard = world > 1 and a.mode != "replicas"
    # ---- residency plan: precomputed multiples of every base as far as HBM allows (DESIGN.md section 2) ----
    nvars = m.num_instance_variables + m.num_witness_variables
    key_bytes = nvars * 8 * nq * (4 * 2 + 4)              # a, b_g1, h, l (G1) + b_g2, packed affine, one copy
    mem_total = torch.cuda.get_device_properties(dev).total_memory
    share = world if want_shard else 1
    ne = 1
    while ne < 16 and key_bytes * ((16 + ne - 1) // ne) / share > 0.5 * mem_total:
        ne *= 2
    big = key_bytes * 16 > 0.5 * mem_total                # the unsharded key with all copies does not fit one GPU
    if os.environ.get("G16_BENCH_FORCE_BIG"):              # exercise the large-key path (mint without copies, re-load) at any size
        big = True
    residency = {"key_bytes_one_copy": int(key_bytes), "msm_ne": ne, "copies": (16 + ne - 1) // ne,
                 "resident_key_bytes_per_gpu": int(key_bytes * ((16 + ne - 1) // ne) / share)}
    t = time.time()
    if big:
        g.set_option("msm_ne", 0)                         # mint the key without precomputed multiples, re-load it with the plan
        g.set_option("proof_slots", 1)
    pk = g.generate_parameters_with_qap(m, *TOXIC, G["g1"], G["g2"], export=(want_shard or big or not a.no_cpu_baseline))
    if big:
        g.set_option("msm_ne", ne)
        if not want_shard:
            g.load_proving_key(pk, 0, 1)
    t_setup = time.time() - t
    r = np.ascontiguousarray(cd.fr.enc1(123456789))
    s = np.ascontiguousarray(cd.fr.enc1(987654321))
    z_pinned = torch.from_numpy(z_np.view(np.int64)).pin_memory()
    z_dev = z_pinned.to(dev)
    proof = np.zeros(8 * nq, dtype=np.uint64)
    ON_DEV = _lib.ASSIGNMENT_ON_DEVICE

    class Arm:
        """one way of running a step: 'single' (this GPU proves alone) or 'shard' (one proof split over all ranks)"""

        def __init__(self, kind, inflight):
            self.kind, self.inflight = kind, inflight
            self.sp = None
            if kind == "shard":
                from groth16_b200.dist import ShardedProver
                self.sp = ShardedProver(g, pk, None, rank, world, dev)   # keeps this rank's round-robin share of every query

        def step(self, zptr, flags):
            if self.kind == "single":
                g.prove_raw(r, s, zptr, flags, proof)
            else:
                pf = self.sp.prove(r, s, zptr, flags)   # partial MSMs -> NCCL all-gather of 5 points per rank -> assemble
                proof[:2 * nq] = pf.a; proof[2 * nq:6 * nq] = pf.b; proof[6 * nq:] = pf.c
            return proof

        def _submit(self, slot, zptr, flags):
            if self.kind == "single":
                g.prove_submit_raw(slot, r, s, zptr, flags)
            else:
                self.sp.submit(slot, r, zptr, flags, s=s)

        def _finish(self, slot):
            if self.kind == "single":
                g.prove_wait_raw(slot, proof)
            else:
                pf = self.sp.finish(slot, r, s)
                proof[:2 * nq] = pf.a; proof[2 * nq:6 * nq] = pf.b; proof[6 * nq:] = pf.c

        def run_steps(self, zptr, flags, steps):
            """`steps` complete proofs; with inflight 2 proof i+1 is submitted before proof i is waited for"""
            dev_ms, launches = [], 0
            if self.inflight == 1:
                for _ in range(steps):
                    self.step(zptr, flags)
                    tm = g.timings()
                    dev_ms.append(tm["total_ms"]); launches += tm["launches"]
                return dev_ms, launches
            self._submit(0, zptr, flags)
            for i in range(1, steps + 1):
                if i < steps:
                    self._submit(i & 1, zptr, flags)
                self._finish((i - 1) & 1)
                tm = g.timings()
                dev_ms.append(tm["total_ms"]); launches += tm["launches"]
            return dev_ms, launches

        def timed(self, zptr, flags, steps, sampler=None):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            if sampler:
                sampler.mark_begin()
            t0 = time.perf_counter()
            dev_ms, launches = self.run_steps(zptr, flags, steps)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            dt = time.perf_counter() - t0
            if sampler:
                sampler.mark_end()
            clocks = sampler.stop() if sampler else None
            if world > 1:
                tt = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
            return dt, dev_ms, launches, clocks

        def latency(self, zptr, flags, reps=5):
            """one proof at a time (no pipelining): wall-clock latency per proof"""
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                self.step(zptr, flags)
            torch.cuda.synchronize()
            return 1e3 * (time.perf_counter() - t0) / reps

        def measure(self, units, sampler=None):
            """warm-up, resident-input run, single-proof latency, host-input (e2e) run"""
            if sampler:
                sampler.start()   # before the warm-up: nvidia-smi's start-up must not fall into the timed region
                sampler.wait_ready()
            # warm-up through the SAME path as the timed steps: with two proofs in flight the second proof slot's workspaces
            # (GBs of cudaMalloc) are allocated on first use -- in round-2 records taken before this fix that happened inside
            # the first timed region (`value` of the inflight-2 runs was understated; their `e2e` run came after and was not)
            self.run_steps(z_dev.data_ptr(), ON_DEV, max(a.warmup, 3))
            first = self.step(z_dev.data_ptr(), ON_DEV).copy()
            dt, dev_ms, launches, clocks = self.timed(z_dev.data_ptr(), ON_DEV, a.steps, sampler)
            last = proof.copy()                  # the proof of the last timed step
            lat = self.latency(z_dev.data_ptr(), ON_DEV)
            self.run_steps(z_pinned.data_ptr(), 0, 2)
            assert np.array_equal(first, proof), "resident-input and host-input proofs differ"
            dt_e, _, _, _ = self.timed(z_pinned.data_ptr(), 0, a.steps)
            tm_e = g.timings()
            return {"proof": first, "last": last, "value": units * a.steps / dt, "ms_per_step": 1e3 * dt / a.steps,
                    "device_ms_per_step": statistics.mean(dev_ms), "latency_ms_single_proof": lat, "launches": int(launches),
                    "clocks": clocks, "inflight": self.inflight,
                    "e2e": {"value": units * a.steps / dt_e, "unit": "proofs/s", "h2d_bytes_per_step": int(tm_e["h2d_bytes"]),
                            "d2h_bytes_per_step": int(tm_e["d2h_bytes"]), "ms_per_step": 1e3 * dt_e / a.steps}}

    sampler = ClockSampler(local) if rank == 0 else None
    secondary = None
    # Two proofs in flight (software pipeline over the two proof slots of a context) up to 2^20: the next proof's sort and
    # first rounds fill the latency-bound tail of the previous one (bucket reduction, host finish) -- +3.7 % on one GPU
    # (gpurun_out/bench_r02p_*.json: 35.8 vs 34.5 proofs/s), more on the small per-rank shards.  Larger circuits keep one proof
    # in flight: the second slot's work lists would compete with the precomputed multiples for HBM.
    auto_inflight = 1 if (big or a.log_n > 20) else 2
    if want_shard:
        arm = Arm("shard", a.inflight or auto_inflight)
        main = arm.measure(1, sampler)
        main["library"] = g.config()              # launch geometry of this rank's shard (before the replicas reload the full key)
        par = (f"msm-shard{world}: one proof per step, pair i of every MSM on rank i mod {world}, the witness map's three a/b/c chains spread over the "
               "ranks (ncclSend/Recv, h broadcast), "
               "3 partial points per rank (768 B) all-gathered by ONE ncclAllGather issued inside the library "
               "(g16_prove_sharded), every rank finishes the same proof")
        scaling = "strong"
        if a.mode == "auto" and not big:
            g.load_proving_key(pk, 0, 1)          # full key resident again: every rank proves on its own
            rep = Arm("single", a.inflight or auto_inflight).measure(world)
            assert np.array_equal(rep["proof"], main["proof"]), "sharded and single-GPU proofs differ"
            secondary = {"mode": f"replicas{world}: one independent proof per GPU per step, no communication", "scaling": "weak",
                         "value": rep["value"], "unit": "proofs/s", "ms_per_step": rep["ms_per_step"], "e2e_value": rep["e2e"]["value"],
                         "proof_equals_sharded_proof": True}
    else:
        arm = Arm("single", a.inflight or auto_inflight)
        main = arm.measure(world, sampler)
        par = f"replicas{world} (one independent proof per GPU per step, no communication)" if world > 1 else "single-gpu"
        scaling = "weak" if world > 1 else "strong"
    first = main["proof"]

    if rank == 0:
        # ---- kernel-level numbers: serialised MSMs so that CUDA events bracket one bucket-accumulation stage at a time ----
        roof, kern, cpu = None, {}, None
        if world == 1:
            acc = {k: [] for k in ("h", "l", "a", "b_g1", "b_g2")}
            for _ in range(3):
                g.prove_raw(r, s, z_dev.data_ptr(), ON_DEV | _lib.SERIAL_MSMS, proof)
                tm = g.timings()
                for k in acc:
                    acc[k].append(tm["msm_accum_ms"][k])
            assert np.array_equal(first, proof), "serialised-stream proof differs"
            pairs, entries, wm_ms = tm["msm_pairs"], tm["msm_entries"], tm["witness_map_ms"]
            g1_bytes = 32 + 2 * 8 * nq          # scalar + packed affine G1 base  (SURVEY 8d: 128 B on BLS12-381)
            g2_bytes = 32 + 4 * 8 * nq          # 224 B
            g1k = [k for k in ("h", "l", "a", "b_g1") if pairs[k]]
            t_g1 = sum(statistics.median(acc[k]) for k in g1k)
            b_g1 = sum(pairs[k] for k in g1k) * g1_bytes
            t_g2 = statistics.median(acc["b_g2"])
            b_g2 = pairs["b_g2"] * g2_bytes
            peak, peak_src = measured_peak_hbm()
            summ = ncu_summary() or {}
            cfg = g.config()
            # the capture describes ONE workload: same kernel sources, same launch geometry, same curve / size / circuit
            same_code = (summ.get("kernel_rev") == kernel_rev() and summ.get("config") == cfg and summ.get("curve") == a.curve
                         and summ.get("log_n") == a.log_n and summ.get("workload", "synthetic") == a.workload)
            ach = b_g1 / (t_g1 * 1e-3) / 1e9 if t_g1 > 0 else 0.0
            # honest bound: the integer-multiply pipe.  IMAD.WIDE per bucket entry from the SASS (cuobjdump, DESIGN.md section 3)
            nl = 2 * nq                          # 32-bit limbs of Fq
            mul = 2 * nl * nl                    # IMAD.WIDE per Montgomery product (288 for 12 limbs, 128 for 8)
            per_entry = cfg["imad_per_g1_entry_mul"] * mul
            e_g1 = sum(entries[k] for k in g1k)
            sm_clk = (main["clocks"] or {}).get("sm_mhz") or 1965.0
            pipe_peak = torch.cuda.get_device_properties(dev).multi_processor_count * INT_PIPE_LANES_PER_CLK_SM * sm_clk * 1e6
            imad_rate = e_g1 * per_entry / (t_g1 * 1e-3) if t_g1 > 0 else 0.0
            roof = {"kernel": cfg["g1_accum_stage"], "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": summ.get("g1_dram_bytes_per_launch") if same_code else None,
                    "algorithmic_bytes_per_launch": b_g1 / max(1, len(g1k)), "avg_launch_ms": t_g1 / max(1, len(g1k)),
                    "launches_averaged": len(g1k), "peak_source": peak_src,
                    "int_pipe_frac": imad_rate / pipe_peak, "int_pipe_imad_wide_per_s": imad_rate, "int_pipe_peak_per_s": pipe_peak,
                    "int_pipe_model": f"{e_g1} bucket entries x {cfg['imad_per_g1_entry_mul']:.2f} field products x {mul} IMAD.WIDE "
                                      f"per product; peak = SMs x 32 lanes/clk x {sm_clk:.0f} MHz",
                    "note": "integer-multiply bound, not HBM bound: algorithmic bytes are 128 B per pair against ~2-3 thousand "
                            "IMAD.WIDE; `traffic` is the ncu dram__bytes of the committed capture when it was taken with this "
                            "code and configuration, else null"}
            n_dom = 1 << a.log_n
            kern = {"g2_accum_stage": {"achieved_gbs": b_g2 / (t_g2 * 1e-3) / 1e9 if t_g2 > 0 else None, "launch_ms": t_g2,
                                       "frac": (b_g2 / (t_g2 * 1e-3) / 1e9 / peak) if t_g2 > 0 else None},
                    "witness_map": {"ms": wm_ms, "achieved_gbs": 576 * n_dom / (wm_ms * 1e-3) / 1e9,
                                    "frac": 576 * n_dom / (wm_ms * 1e-3) / 1e9 / peak},
                    "msm_accum_ms": {k: statistics.median(v) for k, v in acc.items()}, "msm_pairs": pairs, "msm_entries": entries}
            # ---- CPU baseline beside it (rank 0, N = 1): one full proof by the restated ark CPU path, also a parity check ----
            if not a.no_cpu_baseline:
                threads = host_threads(a.cpu_threads)
                cproof, csec, tms = cpu_prove_once(a, cd, nq, pk, m, z_np, r, s, threads)
                if not np.array_equal(cproof, first):
                    raise SystemExit("PARITY FAILURE: CUDA proof != CPU oracle proof at full size")
                cpu = {"value": 1.0 / csec, "unit": "proofs/s", "cores": threads, "kind": "port",
                       "sample": f"1 full proof of the same workload ({csec:.2f} s wall: witness map {tms[0]:.0f} ms, MSMs+assembly "
                                 f"{tms[1]:.0f} ms), restated ark CPU path; proof bit-identical to the CUDA proof"}
        oracle_check = None
        if world > 1 and a.check_oracle:
            threads = host_threads(a.cpu_threads)
            cproof, csec, tms = cpu_prove_once(a, cd, nq, pk, m, z_np, r, s, threads)
            if not np.array_equal(cproof, first):
                raise SystemExit("PARITY FAILURE: sharded CUDA proof != CPU oracle proof")
            oracle_check = {"proof_bit_identical_to_cpu_oracle": True, "cpu_seconds": csec, "cores": threads,
                            "witness_map_ms": tms[0], "msm_ms": tms[1]}
        line = {
            "metric": metric_name(a), "value": main["value"], "unit": "proofs/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None,
            "dtype": "u32 limbs (255-bit Fr / 381-bit Fq Montgomery integers)", "data": "synthetic",
            "config": {"workload": workload_name(a), "curve": a.curve, "log_n": a.log_n, "parallelism": par,
                       "inflight": main["inflight"], "library": main.get("library") or g.config(),
                       "l2": "inputs exceed L2: resident proving key with precomputed multiples (GBs) + 32 MiB assignment + "
                             "sorted digit arrays (134 MB per MSM) are streamed every step",
                       "timing": "wall clock around K complete proofs bracketed by barrier+synchronize (host finish/assembly "
                                 "included), max over ranks; with inflight=2 proof i+1 is submitted before proof i is waited "
                                 "for (two proof slots per context); device_span_ms_per_proof = CUDA-event span of one proof's "
                                 "GPU work (with two proofs in flight the spans of successive proofs overlap, so it is about "
                                 "twice ms_per_step); latency_ms_single_proof = one proof at a time"},
            "device_span_ms_per_proof": main["device_ms_per_step"],
            "latency_ms_single_proof": main["latency_ms_single_proof"],
            "e2e": main["e2e"],
            "gpu_launches": main["launches"],
            "proof_sha256": __import__("hashlib").sha256(first.tobytes()).hexdigest(),
            "residency": residency,
            "clocks": main["clocks"],
            "setup_s": {"workload": t_work, "gpu_setup_and_key_residency": t_setup},
        }
        knobs = {k: v for k, v in sorted(os.environ.items()) if k.startswith("G16_")}
        if knobs:                                  # non-default tuning knobs (INTEGRATION.md section 6) are part of the record
            line["config"]["env"] = knobs
        if secondary:
            line["replicas"] = secondary
        if oracle_check:
            line["oracle_check"] = oracle_check
        if roof:
            line["roofline"] = roof
            line["kernels"] = kern
        if cpu:
            line["cpu_baseline"] = cpu
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, main["last"], nq)
        emit(a, line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_cuda(a)


if __name__ == "__main__":
    main()
