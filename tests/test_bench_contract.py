"""bench.py's reference arm runs on CPU: check the JSON line the driver parses (keys, units, the cpu_baseline and e2e
objects of the reference arm) without a GPU; and that the device arm refuses to run without CUDA instead of falling back."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "scores/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["config"]["workload"].startswith("C3 dyadic all-pairs")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_ranks_other_than_zero_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_device_arm_does_not_fall_back_to_the_cpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "scores/s" not in r.stdout


def test_bad_arguments_are_refused_before_any_work():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 2 and r.stdout == "" and "error:" in r.stderr


@pytest.mark.gpu
def test_dumped_outputs_are_the_last_timed_step_and_repeat(tmp_path):
    """--dump-outputs writes the top-k lists of the last timed step: 2 and 6 steps both end on query batch 1 of the
    four the benchmark cycles through, so two runs must write the same arrays; the device entry point and the
    host-buffer one must agree."""
    import numpy as np

    def run(steps):
        out = tmp_path / f"s{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--no-cpu-baseline",
                            "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        return {f.stem: np.load(f) for f in out.iterdir()}

    a, b = run(2), run(6)
    assert sorted(a) == ["e2e_topk_dist", "e2e_topk_index", "topk_dist", "topk_index"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name, v in a.items():
        assert v.shape == (1024, 100) and v.dtype == (np.float32 if name.endswith("dist") else np.float64)
        np.testing.assert_array_equal(v, b[name], err_msg=name)
    np.testing.assert_array_equal(a["topk_dist"], a["e2e_topk_dist"])
    np.testing.assert_array_equal(a["topk_index"], a["e2e_topk_index"])
    idx = a["topk_index"]
    assert (idx == np.round(idx)).all() and idx.min() >= 0 and idx.max() < 1_000_000
    assert (np.diff(a["topk_dist"], axis=1) >= 0).all()


def test_smoke_tie_check_accepts_fp32_ties_and_rejects_real_differences():
    """The index-set check of __graft_entry__.smoke(): a swap inside an fp32 tie at the k-th distance passes
    (and leaves smoke()'s helpers callable), a swap with a clearly worse candidate fails."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    D = np.array([[0.1, 0.2, 0.3, 0.3 * (1 + 1e-7), 0.9]])
    want_idx, want_val = np.array([[0, 1, 2]]), np.array([[0.1, 0.2, 0.3]])
    ge.check_topk_sets(D, want_idx, want_val, np.array([[0, 1, 3]]))          # tie: candidate 3 for 2
    ge.check_topk_sets(D, want_idx, want_val, np.array([[0, 1, 2]]))
    with pytest.raises(AssertionError):
        ge.check_topk_sets(D, want_idx, want_val, np.array([[0, 1, 4]]))
