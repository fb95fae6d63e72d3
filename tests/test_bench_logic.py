"""CPU: the benchmark's own bookkeeping (bench.py) — the lazy-R1 cadence of the timed loops must not depend on --steps or on
the warm-up count (VERDICT round 1, weak #2: a timed region without any R1 evaluation flattered the rate)."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("sae_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _evaluations(c0, d_steps, every):
    """what swapping_autoencoder_optimizer.py:57-60 / optimizer.train_discriminator_one_step do: the counter is incremented,
    then R1 runs when it is a multiple of R1_once_every"""
    n, c = 0, c0
    for _ in range(d_steps):
        c += 1
        n += (c % every == 0)
    return n


@pytest.mark.parametrize("every", [16, 4, 1])
def test_r1_position_gives_the_cadence_for_every_loop_length(bench, every):
    for d_steps in range(1, 6 * every + 3):
        c0, target = bench.r1_position(d_steps, every)
        assert target == max(1, int(round(d_steps / every)))
        assert 0 <= c0 < every
        assert _evaluations(c0, d_steps, every) == target, (d_steps, every, c0)
    assert bench.r1_position(0, every) == (0, 0)


def test_dump_outputs_writes_losses_and_a_fixed_parameter_sample(bench, tmp_path):
    import numpy as np
    import torch
    params = [("small.weight", torch.arange(6.0).reshape(2, 3)), ("big.weight", torch.randn(3 * bench.DUMP_SAMPLE))]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"D_total": torch.tensor(1.5, dtype=torch.float64)}, params)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["loss.D_total.npy", "param.big.weight.npy", "param.small.weight.npy"]
    loss = np.load(tmp_path / "a" / "loss.D_total.npy")
    assert loss.dtype == np.float64 and float(loss) == 1.5
    small = np.load(tmp_path / "a" / "param.small.weight.npy")
    assert small.dtype == np.float32 and small.tolist() == list(range(6))
    big = np.load(tmp_path / "a" / "param.big.weight.npy")
    assert big.dtype == np.float32 and big.shape == (bench.DUMP_SAMPLE,) and np.isin(big, params[1][1].numpy()).all()
    assert np.array_equal(big, np.load(tmp_path / "b" / "param.big.weight.npy"))      # the same sample every run


def test_the_default_and_the_driver_flags_carry_an_r1_evaluation(bench):
    # default: 32 half-steps = 16 D steps -> exactly one evaluation; the driver's --steps 20 = 10 D steps -> still one
    assert bench.r1_position(16, 16)[1] == 1 and _evaluations(bench.r1_position(16, 16)[0], 16, 16) == 1
    assert bench.r1_position(10, 16)[1] == 1 and _evaluations(bench.r1_position(10, 16)[0], 10, 16) == 1
