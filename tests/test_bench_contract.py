"""bench.py contract on CPU: the reference arm (`--impl reference`) needs no GPU -- it times the reference's own C kernels
(oracle/_ref) or the plain-C port under the restated orchestration -- so its JSON line can be checked here: exactly one
line on stdout, the keys the driver reads, and the tier's reference-arm additions.  --dump-outputs is checked on both arms (the
product arm's on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--steps", "4",
                        "--warmup", "3", "--prompt", "8"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["metric"] == "decode tokens/s" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["steps"] == 4 and d["warmup"] == 3 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_product_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: without a CUDA device the product arm must exit non-zero with a clear message and print no JSON."""
    import pytest
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--steps", "3", "--warmup", "3"], cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + [str(a) for a in args], cwd=ROOT, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_dumps_the_same_tokens_from_run_to_run(tmp_path):
    runs = []
    for i in range(2):
        r = _bench("--impl", "reference", "--model", "tiny", "--steps", 5, "--warmup", 3, "--prompt", 8, "--dump-outputs", tmp_path / str(i))
        assert r.returncode == 0, r.stderr[-2000:]
        runs.append(np.load(tmp_path / str(i) / "tokens.npy"))
    assert runs[0].dtype == np.float64 and runs[0].shape == (5,)
    assert np.array_equal(runs[0], runs[1])


def test_steps_below_one_are_refused():
    r = _bench("--impl", "reference", "--model", "tiny", "--steps", 0)
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_product_arm_times_the_requested_steps_and_dumps_their_tokens(tmp_path, oracle):
    """The dump holds what the timed steps decoded: tokens warmup+1 .. warmup+steps of greedy generation after the prompt (token 0 is
    sampled after the prefill, tokens 1 .. warmup by the warm-up), the same tokens the oracle generates."""
    from jlama_b200 import synth
    steps, warmup, prompt = 4, 3, 12
    r = _bench("--gpus", 1, "--model", "tiny", "--steps", steps, "--warmup", warmup, "--prompt", prompt, "--prefill-tokens", 0,
               "--no-cpu-baseline", "--dump-outputs", tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert d["steps"] == steps and d["value"] > 0
    got = np.load(tmp_path / "tokens.npy")
    assert got.dtype == np.float64 and got.shape == (steps,)
    cfg = synth.get_config("tiny")
    om = oracle.OracleLlama(cfg, synth.make_weights(cfg), act_q8=True)
    want, _ = om.generate(synth.random_prompt(cfg, prompt), 1 + warmup + steps, want_logits=False)
    om.close()
    assert [int(t) for t in got] == [int(t) for t in want[1 + warmup:]]
