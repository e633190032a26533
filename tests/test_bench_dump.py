"""bench.py --dump-outputs: what it writes for the default and the largest configuration, without a GPU."""
import os

import numpy as np
import torch

import bench


def _dump(tmp_path, name, F, H, seed):
    theta = torch.from_numpy(np.random.default_rng(seed).standard_normal(F * H + F + H).astype(np.float32))
    stats = torch.arange(16, dtype=torch.float64)
    d = tmp_path / name
    bench.dump_outputs(str(d), F, H, theta, stats)
    return {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}, theta.numpy(), sum(f.stat().st_size for f in d.iterdir())


def test_dump_outputs_layout_and_size(tmp_path):
    F, H = bench.CONFIGS['C2']['F'], bench.CONFIGS['C2']['H']
    out, theta, _ = _dump(tmp_path, 'c2', F, H, 0)
    assert sorted(out) == ['dec_b', 'enc_b', 'enc_w', 'step_stats']
    assert out['enc_w'].shape == (F, H) and (out['enc_w'].ravel() == theta[:F * H]).all()
    assert (out['enc_b'] == theta[F * H:F * H + H]).all() and (out['dec_b'] == theta[F * H + H:]).all()
    assert out['step_stats'].dtype == np.float64 and (out['step_stats'] == np.arange(16)).all()
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())

    F, H = bench.CONFIGS['C4']['F'], bench.CONFIGS['C4']['H']          # 200 MB of weights: a seeded sample of rows
    a, theta, nbytes = _dump(tmp_path, 'c4a', F, H, 1)
    b, _, _ = _dump(tmp_path, 'c4b', F, H, 1)
    assert nbytes <= 64 * 10 ** 6 and 'enc_w' not in a
    W, S = theta[:F * H].reshape(F, H), a['enc_w_row_sample']
    assert S.shape[1] == H and S.shape[0] > F // 5
    assert (S == b['enc_w_row_sample']).all()
    rows = [int(np.flatnonzero((W[:, 0] == r[0]) & (W[:, 1] == r[1]))[0]) for r in S[:50]]
    assert rows == sorted(rows) and all((W[i] == r).all() for i, r in zip(rows, S[:50]))
