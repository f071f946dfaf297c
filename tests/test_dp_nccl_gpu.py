"""Data parallelism over NCCL (SURVEY 8e): a global batch sharded over 2 ranks, one SUM all-reduce of the active net's flat gradient
per step, must give (a) bit-identical parameters on every rank and (b) the single-GPU global-batch result up to the fp32 summation
order of the gradient (each rank reduces its own shard first).  Needs 2 GPUs: skipped on a 1-GPU lease."""
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import params as OP
from unsupervised_detection_b200.step_graph import CISGraph

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_two_rank_nccl_training_equals_single_gpu_global_batch(tmp_path):
    gen = torch.Generator().manual_seed(31)
    GB, H, W, ph, pw = 4, 64, 96, 128, 192
    lo = torch.randn(GB, 3, ph // 16, pw // 16, generator=gen)
    img1 = (F.interpolate(lo, size=(ph, pw), mode='bicubic', align_corners=False) * 0.25).permute(0, 2, 3, 1).contiguous().clamp(-0.5, 0.5)
    img2 = torch.roll(img1, shifts=(1, 2), dims=(1, 2)) + 0.01 * torch.randn(GB, ph, pw, 3, generator=gen)
    p = OP.make_params(seed=12, jitter=0.1)
    modes = 'GGRG'
    torch.save(dict(GB=GB, H=H, W=W, ph=ph, pw=pw, img1=img1, img2=img2, params=p, modes=modes), str(tmp_path / 'inputs.pt'))
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(_free_port()), os.path.join(ROOT, 'tests', 'probes', 'dp_equality_worker.py'), str(tmp_path)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stderr[-2000:]
    ranks = [torch.load(str(tmp_path / ('rank%d.pt' % i))) for i in range(2)]
    diff = [k for k in ranks[0] if not torch.equal(ranks[0][k], ranks[1][k])]
    assert not diff, diff[:5]                                           # every rank applies the same averaged gradient
    g = CISGraph(H, W, GB, with_pwc=True, pwc_hw=(ph, pw))
    g.load_params(p)
    g.img1.copy_(img1)
    g.img2.copy_(img2)
    for mode in modes:
        g.train_step(mode, use_graph=True)
    torch.cuda.synchronize()
    one = {k: v.cpu() for k, v in g.export_params().items() if not k.startswith('pwcnet')}
    worst = max(float((one[k] - ranks[0][k]).abs().max()) for k in one)
    mean = float(torch.cat([(one[k] - ranks[0][k]).abs().reshape(-1) for k in one]).mean())
    moved = float(torch.cat([(one[k] - p[k]).abs().reshape(-1) for k in one]).mean())
    # summation order only: Adam normalises tiny generator gradients, so isolated elements may differ by a step size (lr = 1e-4)
    assert worst <= 2.5e-4 * len(modes) and mean <= 0.02 * moved, (worst, mean, moved)
