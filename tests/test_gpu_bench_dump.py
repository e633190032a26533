"""bench.py --dump-outputs on the device: two runs with the same arguments train on the same batches and write the same outputs,
up to the rounding of the float atomics."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_runs_dump_the_same_outputs(tmp_path):
    outs = []
    for i in range(2):
        d = tmp_path / ('run%d' % i)
        cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '12', '--warmup', '3', '--rows', '8000',
               '--no-cpu-baseline', '--no-fit-api', '--dump-outputs', str(d)]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
        outs.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = outs
    assert sorted(a) == ['dec_b', 'enc_b', 'enc_w', 'step_stats']
    from dae_rnn_news_recommendation_b200._cabi import STAT
    assert a['step_stats'][STAT['n_valid']] == b['step_stats'][STAT['n_valid']]       # the labels of the batch: same rows
    assert np.allclose(a['step_stats'], b['step_stats'], rtol=1e-5, atol=0)
    for k in ('enc_w', 'enc_b', 'dec_b'):
        assert np.allclose(a[k], b[k], rtol=1e-4, atol=1e-6 * np.abs(a[k]).max()), k
