"""This library's plugin entry point against the REFERENCE'S OWN native kernel: ``alt_cuda_corr.forward(fmap1, fmap2,
coords, radius)`` -- same tensors in, same tensor out (correlation.cpp:23-33).  What the reference kernel returned on a
B200 for these inputs is stored as samples in op_ref_alt_cuda_corr.npz (oracle/make_golden.py --ref-plugin)."""
import pytest
import torch

from oracle import synth
from helpers import check_sample, load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("b,c,h1,w1,h2,w2,r", [(1, 256, 16, 24, 16, 24, 4), (2, 128, 17, 29, 8, 14, 4), (1, 64, 9, 12, 9, 12, 3), (1, 256, 55, 128, 27, 64, 4)])
def test_forward_matches_the_reference_kernel(b, c, h1, w1, h2, w2, r):
    from ptlflow_b200 import alt_cuda_corr

    _, g = load_golden("op_ref_alt_cuda_corr")
    f1 = torch.from_numpy(synth.synth_normal("rp/f1", (b, h1, w1, c), 21)).to(DEV)
    f2 = torch.from_numpy(synth.synth_normal("rp/f2", (b, h2, w2, c), 21)).to(DEV)
    grid = torch.stack(torch.meshgrid(torch.arange(w1, dtype=torch.float32), torch.arange(h1, dtype=torch.float32), indexing="xy"), dim=-1)  # [h1,w1,2] (x, y)
    coords = (grid[None, None] * (w2 / w1) + torch.from_numpy(synth.synth_normal("rp/c", (b, 1, h1, w1, 2), 21, scale=3.0))).contiguous().to(DEV)
    (ours,) = alt_cuda_corr.forward(f1, f2, coords, r)
    assert ours.dtype == torch.float32
    key = "case_" + "_".join(map(str, (b, c, h1, w1, h2, w2, r)))
    scale = max(1.0, float(g[key + "_sums"][2]))
    check_sample(ours, g, key, 2e-5 * scale)
