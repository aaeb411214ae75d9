"""bench.py's contract on a box without a GPU: the reference arm (the CPU restatement, `--impl reference`) runs and prints ONE JSON line
with the keys the driver reads; the product arm refuses to run without CUDA instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_json_line():
    r = run_bench("--impl", "reference", "--reads", "2000", "--ref-bases", "150000", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "aligned reads/sec" and d["unit"] == "reads/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


SMALL = ("--ref-bases", "150000", "--steps", "1", "--warmup", "1")


def load_dump(path):
    out = {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}
    assert out and all(v.dtype in (np.float32, np.float64) for v in out.values()), {k: v.dtype for k, v in out.items()}
    assert sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path)) <= 64 << 20
    return out


def check_result_layout(d):
    """The dumped result arrays form the library's CSR layout for the sampled queries."""
    nq = len(d["query_index"])
    assert len(d["q_comp_off"]) == nq + 1 and len(d["q_status"]) == nq
    nc = int(d["q_comp_off"][-1]); nch = int(d["comp_choice_off"][-1]); nsa = int(d["choice_sa_off"][-1]); nb = int(d["sa_block_off"][-1])
    assert (len(d["comp_choice_off"]), len(d["choice_sa_off"]), len(d["sa_block_off"])) == (nc + 1, nch + 1, nsa + 1)
    assert (len(d["choice_f64"]), len(d["choice_inner"]), len(d["sa_f64"]), len(d["sa_contig"]), len(d["sa_reversed"]), len(d["blocks"])) == (
        4 * nch, nch, 2 * nsa, nsa, nsa, 4 * nb)
    assert nb > 0


def test_reference_arm_dumps_the_same_outputs_every_run(tmp_path):
    dumps = []
    for k in range(2):
        r = run_bench("--impl", "reference", "--reads", "2000", *SMALL, "--dump-outputs", str(tmp_path / str(k)))
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append(load_dump(tmp_path / str(k)))
    check_result_layout(dumps[0])
    assert np.array_equal(dumps[0]["query_index"], np.arange(2000))      # a batch this small is dumped whole
    assert dumps[0].keys() == dumps[1].keys()
    for k in dumps[0]:
        assert np.array_equal(dumps[0][k], dumps[1][k]), k


def test_steps_must_be_positive():
    r = run_bench("--impl", "reference", "--reads", "2000", "--ref-bases", "150000", "--steps", "0")
    assert r.returncode != 0 and not r.stdout.strip()


@pytest.mark.gpu
def test_product_arm_dumps_what_the_reference_computes(tmp_path):
    """The product's dump and the reference arm's dump of the same arguments are equal array for array (the device results are
    bit-identical to the CPU restatement)."""
    r = run_bench("--reads", "150000", *SMALL, "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "ours"))
    assert r.returncode == 0, r.stderr[-2000:]
    r = run_bench("--impl", "reference", "--reads", "150000", *SMALL, "--dump-outputs", str(tmp_path / "reference"))
    assert r.returncode == 0, r.stderr[-2000:]
    ours, ref = load_dump(tmp_path / "ours"), load_dump(tmp_path / "reference")
    check_result_layout(ours)
    assert len(ours["query_index"]) == 1 << 17     # sampled from the 150,000 queries
    assert ours.keys() == ref.keys()
    for k in ours:
        assert np.array_equal(ours[k], ref[k]), k


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this box has a GPU: the product arm runs (tests -m gpu, bench.py)")
    r = run_bench("--reads", "2000", "--ref-bases", "150000", "--steps", "1", "--warmup", "1", "--no-cpu-baseline")
    assert r.returncode != 0, "bench.py must not produce a product number without CUDA"
    assert not any(ln.strip().startswith("{") for ln in r.stdout.splitlines()), r.stdout
