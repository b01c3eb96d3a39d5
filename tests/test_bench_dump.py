"""bench.py --dump-outputs: the writer's size budget (CPU) and the files of a real run (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def load(d, name):
    return np.load(os.path.join(d, f'{name}.npy'))


def test_write_outputs_samples_logits_rows_to_stay_within_budget(tmp_path):
    g = torch.Generator().manual_seed(0)
    loss, logits, grad = torch.rand(2, generator=g), torch.randn(1000, 13, generator=g), \
        torch.randn(500, generator=g)
    bench.write_outputs(str(tmp_path / 'all'), loss, logits, grad)
    assert sorted(os.listdir(tmp_path / 'all')) == ['grad.npy', 'logits.npy', 'loss.npy']
    for name, t in (('loss', loss), ('logits', logits), ('grad', grad)):
        a = load(tmp_path / 'all', name)
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy())
    budget = 20_000
    for d in ('a', 'b'):
        bench.write_outputs(str(tmp_path / d), loss, logits, grad, budget=budget)
    rows = load(tmp_path / 'a', 'logits_rows')
    assert rows.dtype == np.float64 and np.array_equal(rows, load(tmp_path / 'b', 'logits_rows'))
    assert 0 < rows.size < 1000 and (np.diff(rows) > 0).all()
    assert np.array_equal(load(tmp_path / 'a', 'logits'), logits.numpy()[rows.astype(np.int64)])
    assert sum(load(tmp_path / 'a', n).nbytes for n in ('loss', 'logits', 'grad', 'logits_rows')) \
        <= budget
    with pytest.raises(AssertionError):                  # the gradient alone is over budget
        bench.write_outputs(str(tmp_path / 'c'), loss, logits, grad, budget=grad.numel() * 4)


def run_tiny_bench(out_dir, steps=2):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'tiny',
                          '--steps', str(steps), '--warmup', '0', '--no-cpu-baseline',
                          '--dump-outputs', str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['steps'] == steps
    assert sorted(os.listdir(out_dir)) == ['grad.npy', 'logits.npy', 'loss.npy']
    return line


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    run_tiny_bench(tmp_path)
    loss, logits, grad = (load(tmp_path, n) for n in ('loss', 'logits', 'grad'))
    cfg = bench.BENCH_CONFIGS['tiny']
    assert loss.dtype == logits.dtype == grad.dtype == np.float32
    assert loss.shape == (1,) and logits.shape == (cfg['levels'][0], bench.NUM_CLASSES)
    # loss and logits come from the same step: the loss is the logits' cross-entropy
    labels = bench.scene_labels(cfg['levels'][0], cfg['seed'])
    ce = torch.nn.functional.cross_entropy(torch.from_numpy(logits).double(), labels).item()
    assert abs(ce - float(loss[0])) <= 1e-5 * max(1.0, abs(ce))
    import superpoint_transformer_b200 as S
    net = S.SPT(mlp_norm=S.nn.GraphNorm, norm=S.nn.GraphNorm,
                **bench.model_kwargs(S, no_ffn=cfg['no_ffn']))
    n_params = sum(p.numel() for p in net.parameters()) + (bench.DIM + 1) * bench.NUM_CLASSES
    assert grad.shape == (n_params,) and np.isfinite(grad).all() and np.abs(grad).max() > 0


@pytest.mark.gpu
def test_bench_outputs_repeat_from_run_to_run(tmp_path):
    """Same arguments, same inputs, same outputs: the forward is bit-identical and the gradient
    differs only by the rounding of its float-atomic reductions."""
    for d in ('a', 'b'):
        run_tiny_bench(tmp_path / d)
    for name in ('loss', 'logits', 'grad'):
        a, b = load(tmp_path / 'a', name), load(tmp_path / 'b', name)
        scale = float(np.abs(a).max())
        assert np.abs(a.astype(np.float64) - b).max() <= 1e-5 * scale, name


@pytest.mark.gpu
def test_bench_steps_sets_the_number_of_timed_steps(tmp_path):
    """The timed window grows with --steps: 8 steps take several times as long as 1 (a fixed
    loop count would give the same window and a per-step time that falls as 1 / steps)."""
    one, eight = (run_tiny_bench(tmp_path / str(k), steps=k) for k in (1, 8))
    assert eight['ms_per_step'] * 8 > 3 * one['ms_per_step']
