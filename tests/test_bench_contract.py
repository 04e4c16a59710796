"""Tests of bench.py.  Without a GPU: the reference arm prints one JSON line with the contract's keys, rank 0 alone
prints under a multi-rank launch, the output dump stays within its limit, and the GPU arm refuses to run without a
device.  With one (-m gpu): the GPU arm times exactly --steps passes and dumps what the last one computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=e, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_prints_one_contract_line():
    out = run(["--impl", "reference", "--workload", "small", "--steps", "1", "--warmup", "0"])
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "sclens_cells_per_s" and j["unit"] == "cells/s"
    assert j["higher_is_better"] is True and j["value"] > 0 and j["steps"] == 1 and j["warmup"] == 0
    assert j["steps_requested"] == 1 and j["warmup_requested"] == 0
    assert j["config"]["workload"].startswith("small") and j["data"] == "synthetic" and j["vs_baseline"] is None
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "measured once at FULL size" in cb["sample"]
    # the stages are measured, not modelled: seconds per stage at the full shape of the workload, measured once
    assert cb["frac"] == 1 and cb["measured_at"] == [2000, 3000] and cb["eig_n"] == 2000
    assert set(cb["stage_seconds"]) == {"normalise", "gram_f64", "eigen_vectors", "corr"} and min(cb["stage_seconds"].values()) > 0
    assert j["e2e"] == {"value": j["value"], "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    out = run(["--impl", "reference", "--workload", "small", "--steps", "1", "--warmup", "0", "--gpus", "2"],
              env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_writes_floats_within_the_limit(tmp_path):
    """--dump-outputs: every array as float32 / float64 .npy; past the limit the large ones keep a seeded sample of their
    longest axis (the same one on every run) with the sampled positions beside it."""
    sys.path.insert(0, ROOT)
    from bench import dump_outputs
    rng = np.random.default_rng(0)
    arrays = {"evec": rng.standard_normal((5000, 7)).astype(np.float32), "ids": np.arange(9, dtype=np.int32),
              "lam": np.float64(1.5)}
    assert dump_outputs(str(tmp_path / "a"), arrays) == sum(np.asarray(a).nbytes for a in arrays.values()) + 4 * 9
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert got["ids"].dtype == np.float64 and np.array_equal(got["ids"], np.arange(9))
    assert np.array_equal(got["evec"], arrays["evec"]) and got["lam"] == 1.5
    limit = 40_000
    for d in ("b", "c"):
        assert dump_outputs(str(tmp_path / d), arrays, limit=limit) <= limit
    files = sorted(os.listdir(tmp_path / "b"))
    assert files == ["evec.npy", "evec_index.npy", "ids.npy", "lam.npy"] and sum(os.path.getsize(tmp_path / "b" / f) for f in files) <= limit
    idx = np.load(tmp_path / "b" / "evec_index.npy").astype(np.int64)
    np.testing.assert_array_equal(np.load(tmp_path / "b" / "evec.npy"), arrays["evec"][idx])
    np.testing.assert_array_equal(idx, np.load(tmp_path / "c" / "evec_index.npy"))


def test_gpu_arm_refuses_to_run_without_a_device():
    out = run(["--workload", "small", "--steps", "1", "--warmup", "1"], env={"CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_gpu_arm_times_the_requested_steps_and_dumps_the_last_pass(tmp_path):
    out = run(["--workload", "small", "--steps", "3", "--warmup", "1", "--e2e-steps", "0", "--no-cpu-baseline",
               "--dump-outputs", str(tmp_path)])
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["steps"] == 3 and j["steps_requested"] == 3
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    res = j["result"]
    k = int(got["n_signal"])
    assert k == res["n_signal"] > 0 and got["L"].shape == (2000,) and got["signal_evec"].shape == (2000, k)
    assert got["lambda_c"] == res["lambda_c"] and np.all(got["signal_ev"] > res["lambda_c"])
    assert got["gene_basis"].shape == (k, 3000) and got["m_scores"].shape == (k,) and got["b_"].shape == (k, 190)
    assert got["p_sel"] == res["p_sel"] and got["search_p"].shape == (res["n_search"],)
    assert got["sig_id"].shape == (res["n_robust"],) and got["rec_TGC"].shape == (2000,)
