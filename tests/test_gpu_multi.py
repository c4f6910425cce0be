"""Multi-GPU parity (needs >= 2 GPUs on the box; skipped otherwise)."""

import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_two_ranks_reproduce_single_process_reference(tmp_path):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29517',
           os.path.join(ROOT, 'tests', 'multi_rank_scenario.py'),
           'ppo_small', 'ppo_ragged', 'a2c_small', 'td3_small', 'sac_small', 'ddpg_small']
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=540)
    (tmp_path / 'multi_rank_output.log').write_text(res.stdout + '\n----\n' + res.stderr)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
