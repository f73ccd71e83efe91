"""The reference's renderer, wired as the timed CPU baseline runs it (oracle/ref_runner.py), computes what the oracle computes.  The
reference's outputs are stored in tests/golden/render_ref_small.npz (tests/golden/make_golden.py::ref_small_case); where build() staged
the reference modules under oracle/_ref, they are checked against the same outputs."""
import torch

from oracle import real3d_oracle as orc, ref_runner
from real3dportrait_b200 import synthetic as syn


def test_stock_reference_render_matches_oracle_small(golden):
    g = golden('render_ref_small')
    N, res, S = 1, 16, 12
    planes = syn.make_planes(N, h=32, w=32, seed=0)
    cam = syn.make_cameras(N, seed=1)
    mlp, srp = syn.make_decoder_params(seed=4), syn.make_sr_params(seed=5)
    for S_imp in (0, 12):
        u_c, u_f = syn.make_jitter(N, res * res, S, S_imp, seed=2)
        feat, wsum, valid = g[f'imp{S_imp}.rgb'], g[f'imp{S_imp}.wsum'], g[f'imp{S_imp}.valid']
        c2w, K = syn.split_camera(cam)
        o, d = orc.gen_rays(c2w, K, res)
        ref = orc.render(planes, mlp, o, d, S=S, S_imp=S_imp, u_coarse=u_c, u_fine=u_f)
        assert float((feat - ref[0]).abs().max()) < 2e-5 and float((wsum - ref[2]).abs().max()) < 2e-5
        assert torch.equal(valid, ref[3])
        if ref_runner.available():
            head = ref_runner.Head(mlp, srp, S=S, S_imp=S_imp)
            got = head.render(planes, cam, u_c, u_f, res=res)
            assert float((got[0] - feat).abs().max()) < 2e-5 and float((got[2] - wsum).abs().max()) < 2e-5
            assert torch.equal(got[3], valid)
