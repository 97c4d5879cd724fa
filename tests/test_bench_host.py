"""CPU tests of bench.py's host-side pieces (no GPU, no CUDA library): the clock sampler's timed-region window, the
applicability rule of the committed ncu capture (`roofline.traffic`), the CPU-thread rule, and the JSON contract of the
`--impl reference` arm on a small circuit; on a GPU, the outputs --dump-outputs writes for both arms."""
import json
import os
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _line(sm, reasons=("Not Active",) * 4, smax=1965, pw=500.0):
    return f"0, {sm}, {smax}, {pw}, 0x0000000000000000, " + ", ".join(reasons)


def test_clock_sampler_reports_only_samples_of_the_timed_region():
    s = bench.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    now = time.perf_counter()
    # warm-up samples at a low clock, then the timed region at full clock, then a late sample after the region
    s.lines = [(now - 3.0, _line(1200)), (now - 2.9, _line(1250)),
               (now - 2.0, _line(1965)), (now - 1.5, _line(1965)), (now - 1.05, _line(1950, ("Not Active", "Not Active", "Not Active", "Active"))),
               (now - 0.2, _line(800))]
    s.t_begin, s.t_end = now - 2.05, now - 1.1
    out = s.stop()
    assert out["samples"] == 3 and out["sm_mhz"] == 1965.0 and out["window"] == "timed region"
    assert out["reasons"] == ["sw_power_cap"]          # kept and noted (the contract rejects only the thermal / hw ones)


def test_clock_sampler_short_region_falls_back_to_nearest_samples():
    s = bench.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    now = time.perf_counter()
    s.lines = [(now - 3.0, _line(1965)), (now - 2.9, _line(1965))]
    s.t_begin, s.t_end = now - 1.0, now - 0.99       # 10 ms region: no sample can fall into it
    out = s.stop()
    assert out["samples"] == 2 and out["window"].startswith("nearest samples")


def test_clock_sampler_without_nvidia_smi():
    s = bench.ClockSampler(0)
    assert s.stop()["reasons"] == ["nvidia-smi unavailable"]


def test_committed_ncu_capture_matches_the_kernel_sources():
    """profiles/accum_kernel_summary.json must describe the kernels in the tree (bench.py reports roofline.traffic only then)
    and name the workload it was taken on."""
    summ = bench.ncu_summary()
    assert summ is not None
    assert summ["kernel_rev"] == bench.kernel_rev(), "kernel sources changed after the ncu capture: re-run tools/profile_all.sh"
    assert (summ["curve"], summ["log_n"], summ["workload"]) == ("bls12_381", 20, "synthetic")
    # 16 precomputed multiples of every base are gathered twice: the stage moves far more than the 134 MB of algorithmic bytes
    assert 5e9 < summ["g1_dram_bytes_per_launch"] < 3e10


def test_host_threads_respects_request_and_quota():
    assert bench.host_threads(3) == 3
    n = bench.host_threads(0)
    assert 1 <= n <= (os.cpu_count() or 1)


def _run_bench(args):
    out = subprocess.run([sys.executable, "bench.py"] + args, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def _load_dump(d, nq):
    """bench.py --dump-outputs DIR -> the proof as ABI limbs (a || b || c), after checking the files' format"""
    import numpy as np
    parts = [np.load(os.path.join(d, f"{n}.npy")) for n in ("a", "b", "c")]
    assert [p.shape for p in parts] == [(2, 2 * nq), (4, 2 * nq), (2, 2 * nq)] and all(p.dtype == np.float64 for p in parts)
    words = np.concatenate([p.ravel() for p in parts])
    assert np.all((words >= 0) & (words < 2.0 ** 32) & (words == np.floor(words)))
    return words.astype("<u4").view("<u8")


def test_reference_arm_line_contract_small(tmp_path):
    """`bench.py --impl reference` on a 2^10 circuit: one JSON line with the keys the driver reads, nothing of the CUDA library
    loaded (the arm must work on a box whose libg16b200.so is absent or unloadable); --dump-outputs writes a proof that
    verifies for the benchmark's circuit."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--log-n', '10', '--steps', '2', '--warmup', '1', '--cpu-threads', '2',"
            f" '--dump-outputs', {str(tmp_path)!r}];"
            "runpy.run_path('bench.py', run_name='__main__');"
            "import ctypes; assert not any('libg16b200' in l for l in open('/proc/self/maps')), 'reference arm loaded the CUDA library'")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "proofs/s" and line["higher_is_better"] is True
    assert line["metric"] == "groth16_proofs_per_sec_bls12_381_2^10" and line["steps"] == 2 and line["warmup"] == 1
    assert line["gpu_launches"] == 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 2
    import types
    import pyref as P
    from groth16_b200 import Proof
    from util import pk_from_abi, proof_from_abi
    a = types.SimpleNamespace(curve="bls12_381", log_n=10, seed=1, workload="synthetic")
    m, _, pub, _ = bench.build_workload(a)
    pk = pk_from_abi(a.curve, bench.cpu_setup(a, m, 2))
    nq = 6
    limbs = _load_dump(tmp_path, nq)
    pf = proof_from_abi(a.curve, Proof(limbs[:2 * nq], limbs[2 * nq:6 * nq], limbs[6 * nq:]))
    assert P.verify_proof(pk.vk, P.CURVES[a.curve], pf, pub)


@pytest.mark.gpu
def test_dump_outputs_cuda_equals_reference_arm(tmp_path):
    """The CUDA arm's --dump-outputs (the last timed step) equals the reference arm's for the same arguments."""
    import numpy as np
    common = ["--log-n", "12", "--steps", "3", "--warmup", "1", "--cpu-threads", "4"]
    line = _run_bench(common + ["--no-cpu-baseline", "--dump-outputs", str(tmp_path / "cuda")])
    assert line["steps"] == 3
    _run_bench(common + ["--impl", "reference", "--dump-outputs", str(tmp_path / "ref")])
    assert np.array_equal(_load_dump(tmp_path / "cuda", 6), _load_dump(tmp_path / "ref", 6))


def test_standalone_workload_generator_equals_the_library_copy():
    """groth16_b200/libg16workload.so (csrc/workload.cu built with the host compiler alone) and g16_synthetic_r1cs inside
    libg16b200.so are the same generator: identical matrices and assignment for every curve; the circuit is satisfied."""
    import ctypes as C
    import numpy as np
    import pyref as P
    from groth16_b200 import _lib, workload
    from groth16_b200.codec import CurveCodec
    from groth16_b200.params import get_curve
    assert workload._workload_lib() is not None, "libg16workload.so not built (make -C groth16_b200/csrc)"
    for curve in ("bls12_381", "bn254", "bls12_377"):
        m, z, pub = workload.synthetic_r1cs(curve, 9, seed=5)
        nc = (1 << 9) - 2
        a_col = np.empty(2 * nc, dtype=np.uint32); a_val = np.empty((2 * nc, 4), dtype=np.uint64)
        b_col = np.empty(nc, dtype=np.uint32); c_col = np.empty(nc, dtype=np.uint32); z2 = np.zeros((nc + 3, 4), dtype=np.uint64)
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        assert _lib.load().g16_synthetic_r1cs(get_curve(curve).cid, 9, 5, vp(a_col), vp(a_val), vp(b_col), vp(c_col), vp(z2)) == 0
        assert np.array_equal(z, z2) and np.array_equal(m.a[1], a_col) and np.array_equal(m.a[2], a_val)
        assert np.array_equal(m.b[1], b_col) and np.array_equal(m.c[1], c_col)
        # satisfied: (z_p + k) * z_q == z_new for every row
        c = P.CURVES[curve]
        cd = CurveCodec(get_curve(curve))
        zi = cd.fr.dec(z)
        av = cd.fr.dec(a_val)
        for i in range(nc):
            lhs = (zi[a_col[2 * i]] * av[2 * i] + zi[a_col[2 * i + 1]] * av[2 * i + 1]) % c.r
            assert lhs * zi[b_col[i]] % c.r == zi[c_col[i]]
