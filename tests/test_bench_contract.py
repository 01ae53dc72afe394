"""bench.py contract checks: the reference arm prints ONE JSON line with the keys a caller reads, uses every host CPU
even when torchrun's OMP_NUM_THREADS=1 is in the environment, and non-zero ranks stay silent; --dump-outputs writes what
the last timed step computed (the reference arm here, the GPU arm under the gpu mark)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra, args=("--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-log-n", "14")):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def _dumped(d, names):
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in names)
    out = {n: np.load(os.path.join(d, n + ".npy")) for n in names}
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return {n: a.astype(np.uint8).tobytes() for n, a in out.items()}


def test_reference_arm_line_and_thread_count(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_oracle as orc
    import pyref
    from helpers import expected_chain_msm_g1
    dump = tmp_path / "out"
    out = _run({"OMP_NUM_THREADS": "1"}, ("--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-log-n", "14", "--dump-outputs", str(dump)))
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "bn254_g1_msm_points_per_sec" and d["unit"] == "points/s"
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["cores"] == orc.effective_cpus()  # not 1: OMP_NUM_THREADS=1 came from the launcher, not the user
    assert d["config"]["workload"].startswith("2^24-point BN254 G1 MSM per GPU")
    # the timed step's MSM: the closed form of the 2^14-point chain slice
    k, dd = pyref.chain_scalar(pyref.SEED_POINTS)
    assert _dumped(dump, ["g1_msm"])["g1_msm"] == expected_chain_msm_g1(orc.rand_fr(pyref.SEED_SCALARS, 0, 1 << 14), k, dd)


def test_reference_arm_is_silent_on_other_ranks():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}).strip() == ""


def test_importing_bench_leaves_stdout_alone_and_counts_ntt_products(capsys):
    """Tools and tests import bench for source_hash() / the product count: the import must not redirect the importer's
    stdout (only main() claims it), and the NTT product model must follow csrc/ntt.cu's schedule: three 8-stage passes at
    2^24 = 3 x 3.0 stage products + one inter-pass product in passes 2 and 3 with the last pass's direct table, two there
    without it; 2^26 exceeds one lookup in its second pass."""
    sys.path.insert(0, ROOT)
    import bench
    print("still here")
    assert capsys.readouterr().out == "still here\n"
    assert abs(bench.ntt_products_per_element(24) - 11.012) < 1e-2
    assert abs(bench.ntt_products_per_element(24, 0) - 12.012) < 1e-2
    assert abs(bench.ntt_products_per_element(16) - 7.008) < 1e-2           # (8, 8): one lookup, no table needed
    assert bench.ntt_products_per_element(26) > bench.ntt_products_per_element(24) + 1.9
    assert len(bench.source_hash()) == 16


@pytest.mark.gpu
def test_gpu_arm_dumps_what_its_last_timed_steps_computed(tmp_path):
    """Every output the GPU arm dumps equals the oracle's value for the same seeded inputs: the G1 and G2 MSMs (closed
    forms of the chain bases) and the NTT vectors after warmup + steps in-place transforms (2^12 elements: all rows)."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import cpu_oracle as orc
    import pyref
    from helpers import expected_chain_msm_g1, expected_chain_msm_g2
    log_n, n, warmup, steps = 12, 1 << 12, 1, 2
    dump = tmp_path / "out"
    out = _run({}, ("--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--log-n", str(log_n), "--proof-log-n", "10", "--no-cpu",
                    "--dump-outputs", str(dump)))
    assert json.loads(out)["steps"] == steps
    got = _dumped(dump, ["g1_msm", "g2_msm", "ntt_forward", "ntt_inverse", "ntt_forward_e2e", "groth16_proof"])
    k, d = pyref.chain_scalar(pyref.SEED_POINTS)
    s = orc.rand_fr(pyref.SEED_SCALARS, 0, n)
    assert got["g1_msm"] == expected_chain_msm_g1(s, k, d)
    assert got["g2_msm"] == expected_chain_msm_g2(s, k, d)
    a = orc.fr_to_mont(orc.rand_fr(pyref.SEED_NTT, 0, n))
    fwd = [a]
    for _ in range(warmup + steps):
        fwd.append(orc.fr_ntt(fwd[-1], log_n, 0))
    inv = fwd[1]
    for _ in range(warmup + steps):
        inv = orc.fr_ntt(inv, log_n, orc.NTT_INVERSE)
    assert got["ntt_forward"] == fwd[warmup + steps].tobytes()
    assert got["ntt_forward_e2e"] == fwd[1 + steps].tobytes()  # the host-buffer loop warms up with one call
    assert got["ntt_inverse"] == inv.tobytes()
    assert len(got["groth16_proof"]) == 256
