"""Generate the golden fixtures by running the REFERENCE's own modules (imported, unmodified, from /root/reference)
on seeded synthetic inputs.  Runs only in the authoring container (the GPU box has no /root/reference); the
fixtures it writes (tests/golden/*.npz) are committed and are what pins the oracle and the CUDA path.

    python tests/golden/make_golden.py            # rewrites every fixture

Stochasticity: the reference draws its jitter with torch.rand_like / torch.rand (renderer.py:226,281).  We patch
those two functions for the duration of a call so they return OUR uniforms (same shapes, same order), which the
fixtures record; nothing else in the reference is touched.
"""
import os
import sys
from contextlib import contextmanager

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, '/root/reference')
sys.path.insert(0, ROOT)

from utils.commons.hparams import hparams  # noqa: E402  (reference)
hparams.update(dict(enable_rescale_plane_regulation=False, triplane_feature_type='triplane', triplane_depth=1))
from modules.eg3ds.volumetric_rendering.renderer import ImportanceRenderer, sample_from_planes, generate_planes  # noqa: E402
from modules.eg3ds.volumetric_rendering.ray_sampler import RaySampler  # noqa: E402
from modules.eg3ds.models.triplane import OSGDecoder  # noqa: E402
from modules.eg3ds.models.superresolution import SuperresolutionHybrid8XDC  # noqa: E402
from modules.eg3ds.models.networks_stylegan2 import SynthesisLayer, ToRGBLayer  # noqa: E402
from modules.eg3ds.torch_utils.ops import upfirdn2d  # noqa: E402
from modules.eg3ds.camera_utils.pose_sampler import UnifiedCameraPoseSampler  # noqa: E402

from real3dportrait_b200 import synthetic as syn  # noqa: E402

torch.set_grad_enabled(False)


@contextmanager
def supplied_uniforms(u_coarse, u_fine):
    """Make torch.rand_like / torch.rand return the supplied tensors, in the order the renderer draws them."""
    orig_like, orig_rand = torch.rand_like, torch.rand
    def rand_like(t, *a, **k):
        assert tuple(t.shape) == tuple(u_coarse.shape), (t.shape, u_coarse.shape)
        return u_coarse.clone()
    def rand(*size, **k):
        assert u_fine is not None and tuple(size) == tuple(u_fine.shape), (size, None if u_fine is None else u_fine.shape)
        return u_fine.clone()
    torch.rand_like, torch.rand = rand_like, rand
    try:
        yield
    finally:
        torch.rand_like, torch.rand = orig_like, orig_rand


def ref_decoder(params):
    dec = OSGDecoder(params['net.0.weight'].shape[1], {'decoder_lr_mul': 1, 'decoder_output_dim': params['net.2.weight'].shape[0] - 1})
    dec.load_state_dict(params, strict=True)
    return dec.eval()


def ref_render(planes, dec, camera, res, S, S_imp, u_c, u_f, box_warp=1.0, white_back=False):
    c2w, K = syn.split_camera(camera)
    o, d = RaySampler()(c2w, K, res)
    opts = dict(syn.RENDERING_OPTIONS, depth_resolution=S, depth_resolution_importance=S_imp, box_warp=box_warp,
                white_back=white_back)
    with supplied_uniforms(u_c, u_f):
        rgb, depth, wsum, valid = ImportanceRenderer(hp=hparams)(planes, dec, o, d, opts)
    return o, d, rgb, depth, wsum, valid


def save(name, **arrays):
    out = {k: (v.numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in arrays.items()}
    path = os.path.join(HERE, name + '.npz')
    np.savez(path, **out)
    print(f'{name}: {os.path.getsize(path) / 1e6:.2f} MB', {k: tuple(v.shape) for k, v in out.items()})


def small_cases():
    """Small tri-planes (3x32x32x32), 16^2 rays; inputs stored.  Second camera is wide-angle so part of its rays
    miss the box: exercises the invalid-ray fill (renderer.py:123-126) and the NaN->inf->clamp depth path."""
    g = torch.Generator().manual_seed(11)
    planes = torch.randn(2, 3, 32, 32, 32, generator=g)
    cam = syn.lookat_camera(torch.tensor([0.1, -0.15]), torch.tensor([-0.3, 0.45]))
    cam[1, 16] = cam[1, 20] = 1.2              # fx, fy: wide FOV -> rays miss the unit box
    cam[1, 17] = 0.05                          # non-zero skew
    mlp = syn.make_decoder_params(seed=12)
    dec = ref_decoder(mlp)
    res, S = 16, 12
    for name, S_imp, wb in (('render_small', 0, False), ('render_small_imp', 12, False), ('render_small_wb', 0, True)):
        u_c, u_f = syn.make_jitter(2, res * res, S, S_imp, seed=13)
        o, d, rgb, depth, wsum, valid = ref_render(planes, dec, cam, res, S, S_imp, u_c, u_f, white_back=wb)
        assert 0 < int(valid.sum()) < valid.numel(), 'want a mix of valid and invalid rays'
        extra = {} if u_f is None else {'u_fine': u_f}
        save(name, planes=planes, camera=cam, u_coarse=u_c, ray_o=o, ray_d=d, rgb=rgb, depth=depth, wsum=wsum,
             valid=valid, res=res, S=S, S_imp=S_imp, white_back=wb, **{'mlp.' + k: v for k, v in mlp.items()}, **extra)

    # stand-alone gather + decoder on points that straddle the box (zero padding) — sample_from_planes / run_model
    pts = (torch.rand(2, 500, 3, generator=g) - 0.5) * 1.3
    feat = sample_from_planes(generate_planes(), planes, pts, padding_mode='zeros', box_warp=1.0)
    out = dec(feat, pts)
    save('sample_small', planes=planes, coords=pts, feat=feat, rgb=out['rgb'], sigma=out['sigma'],
         **{'mlp.' + k: v for k, v in mlp.items()})


def full_cases():
    """BASELINE config 1 (N=1, 64^2 rays, 48 spp, 3x32x256x256) and its 48+48 variant; inputs come from seeds."""
    planes = syn.make_planes(1, seed=0)
    cam = syn.make_cameras(1, seed=1)
    # our look-at restatement must equal the reference's pose sampler
    g = torch.Generator().manual_seed(1)
    pitch = torch.rand(1, generator=g) * 0.6 - 0.2
    yaw = torch.rand(1, generator=g) * 1.2 - 0.6
    ref_cam = UnifiedCameraPoseSampler().get_camera_pose(float(pitch), float(yaw), lookat_location=torch.tensor([0, 0, 0.2]),
                                                         distance_to_orig=2.7)
    assert (ref_cam - cam).abs().max() < 1e-6, (ref_cam - cam).abs().max()
    mlp = syn.make_decoder_params(seed=4)
    dec = ref_decoder(mlp)
    feats = {}
    for name, S_imp in (('render_full48', 0), ('render_full48_48', 48)):
        u_c, u_f = syn.make_jitter(1, 4096, 48, S_imp, seed=2)
        o, d, rgb, depth, wsum, valid = ref_render(planes, dec, cam, 64, 48, S_imp, u_c, u_f)
        assert bool(valid.all())
        feats[name] = rgb
        save(name, rgb=rgb, depth=depth, wsum=wsum, valid=valid, ray_o=o[:, ::97], ray_d=d[:, ::97], res=64, S=48, S_imp=S_imp,
             seeds=np.array([0, 1, 2, 4]))

    # SR on the rendered feature image (BASELINE config 3 at N=1)
    srp = syn.make_sr_params(seed=5)
    sr = SuperresolutionHybrid8XDC(channels=32, img_resolution=512, sr_num_fp16_res=0, sr_antialias=True,
                                   channel_base=32768, channel_max=512, fused_modconv_default='inference_only').eval()
    missing = sr.load_state_dict(srp, strict=True)
    fimg = feats['render_full48'].permute(0, 2, 1).reshape(1, 32, 64, 64).contiguous()
    img = sr(fimg[:, :3], fimg, torch.ones(1, 14, 512), noise_mode='none')
    save('sr_full', image=img, seeds=np.array([5]))


def layer_cases():
    """Single SynthesisLayer / ToRGB / upsample2d at small sizes with per-sample (non-uniform) styles."""
    g = torch.Generator().manual_seed(21)
    N, cin, cout, r = 2, 8, 16, 12
    x = torch.randn(N, cin, r, r, generator=g)
    w = torch.randn(N, 512, generator=g)
    out = {'x': x, 'w': w}
    for name, up in (('up', 2), ('same', 1)):
        lay = SynthesisLayer(cin, cout, w_dim=512, resolution=r * up, up=up).eval()
        sd = {'weight': torch.randn(cout, cin, 3, 3, generator=g), 'bias': 0.1 * torch.randn(cout, generator=g),
              'affine.weight': torch.randn(cin, 512, generator=g), 'affine.bias': 1 + 0.1 * torch.randn(cin, generator=g),
              'noise_strength': torch.zeros([]), 'noise_const': torch.randn(r * up, r * up, generator=g),
              'resample_filter': lay.resample_filter.clone()}
        lay.load_state_dict(sd, strict=True)
        out[name + '.y'] = lay(x, w, noise_mode='none', fused_modconv=True)
        out.update({f'{name}.{k}': v for k, v in sd.items()})
    trgb = ToRGBLayer(cin, 3, w_dim=512).eval()
    sd = {'weight': torch.randn(3, cin, 1, 1, generator=g), 'bias': 0.1 * torch.randn(3, generator=g),
          'affine.weight': torch.randn(cin, 512, generator=g), 'affine.bias': 1 + 0.1 * torch.randn(cin, generator=g)}
    trgb.load_state_dict(sd, strict=True)
    out['torgb.y'] = trgb(x, w, fused_modconv=True)
    out.update({f'torgb.{k}': v for k, v in sd.items()})
    img = torch.randn(N, 3, r, r, generator=g)
    out['img'] = img
    out['img_up'] = upfirdn2d.upsample2d(img, upfirdn2d.setup_filter([1, 3, 3, 1]))
    out['x_resized'] = torch.nn.functional.interpolate(x, size=(2 * r, 2 * r), mode='bilinear', align_corners=False, antialias=True)
    save('sr_layers', **out)


def warp_case(mode='v2'):
    """BASELINE config 5's SR head (SuperresolutionHybrid8XDC_Warp) at N=1 with the reference class; its torso_model child is replaced by
    synthetic.StubTorsoModel (the real warper is an opaque child outside the hot path).  mode = htbsr_head_weight_fuse_mode: 'v2' (the released
    configuration) -> sr_warp_full.npz; 'v1' / 'v3' (sr_with_ref.py:96-104,126-152) -> sr_warp_v1.npz / sr_warp_v3.npz."""
    import types
    sys.modules.setdefault('imageio', types.ModuleType('imageio'))
    hparams.update(dict(syn.WARP_HPARAMS, htbsr_head_weight_fuse_mode=mode))
    from modules.real3d.super_resolution.sr_with_ref import SuperresolutionHybrid8XDC_Warp
    m = SuperresolutionHybrid8XDC_Warp(channels=32, img_resolution=512, sr_num_fp16_res=0, sr_antialias=True, channel_base=32768,
                                       channel_max=512, fused_modconv_default='inference_only').eval()
    m.torso_model = syn.StubTorsoModel()
    res = m.load_state_dict(syn.make_sr_warp_params(seed=6, fuse_mode=mode), strict=True)
    g = load('render_full48')
    feat = torch.from_numpy(g['rgb'])
    fimg = feat.permute(0, 2, 1).reshape(1, 32, 64, 64).contiguous()
    wimg = torch.from_numpy(g['wsum']).permute(0, 2, 1).reshape(1, 1, 64, 64).contiguous()
    if mode != 'v2':
        wimg = (wimg * 3.0).clamp(0, 1)        # the random-density fixture has weights around 0.3: stretch them so that the head threshold and the v3 quantile bite
    inp = syn.make_warp_inputs(1, seed=7)
    with torch.no_grad():
        img, ret = m(fimg[:, :3], fimg, torch.ones(1, 14, 512), inp['ref_torso_rgb'], inp['ref_bg_rgb'], wimg, inp['segmap'], inp['kp_s'], inp['kp_d'],
                     noise_mode='none')
    if mode == 'v2':
        save('sr_warp_full', image=img, seeds=np.array([6, 7]))
    else:
        save('sr_warp_' + mode, image=img, weights_img=wimg, seeds=np.array([6, 7]))
    hparams.update(syn.WARP_HPARAMS)


def trigrid_case():
    """`triplane_feature_type: trigrid_v2`, `triplane_depth: 3` (egs/os_avatar/img2plane.yaml:65-66): sample_from_trigrids stand-alone and the
    whole ImportanceRenderer (12 and 12+12 samples) on [2,3,32*3,32,32] tri-grids; wide-angle second camera as in small_cases()."""
    from modules.eg3ds.volumetric_rendering.renderer import sample_from_trigrids
    g = torch.Generator().manual_seed(31)
    D = 3
    grids = torch.randn(2, 3, 32 * D, 32, 32, generator=g)
    cam = syn.lookat_camera(torch.tensor([0.1, -0.15]), torch.tensor([-0.3, 0.45]))
    cam[1, 16] = cam[1, 20] = 1.2
    mlp = syn.make_decoder_params(seed=12)
    dec = ref_decoder(mlp)
    pts = (torch.rand(2, 400, 3, generator=g) - 0.5) * 1.3
    feat = sample_from_trigrids(generate_planes(), grids, pts, padding_mode='zeros', box_warp=1.0, triplane_depth=D)
    out = {'planes': grids, 'camera': cam, 'coords': pts, 'feat': feat, 'depth_slices': D}
    hp = dict(hparams, triplane_feature_type='trigrid_v2', triplane_depth=D)
    res, S = 16, 12
    c2w, K = syn.split_camera(cam)
    o, d = RaySampler()(c2w, K, res)
    for tag, S_imp in (('a', 0), ('b', 12)):
        u_c, u_f = syn.make_jitter(2, res * res, S, S_imp, seed=33)
        opts = dict(syn.RENDERING_OPTIONS, depth_resolution=S, depth_resolution_importance=S_imp)
        with supplied_uniforms(u_c, u_f):
            rgb, depth, wsum, valid = ImportanceRenderer(hp=hp)(grids, dec, o, d, opts)
        out.update({f'{tag}.rgb': rgb, f'{tag}.depth': depth, f'{tag}.wsum': wsum, f'{tag}.valid': valid, f'{tag}.u_coarse': u_c})
        if u_f is not None:
            out[f'{tag}.u_fine'] = u_f
    save('render_trigrid', res=res, S=S, **out, **{'mlp.' + k: v for k, v in mlp.items()})


def large_sr_case():
    """SuperresolutionHybrid8XDC(large_sr=True) with hparams['resblocks_in_large_sr'] = 2 (superresolution.py:263-345) on the rendered
    feature image of render_full48."""
    hparams.update({'resblocks_in_large_sr': 2})
    import modules.eg3ds.models.superresolution as sr_mod
    sr_mod.hparams['resblocks_in_large_sr'] = 2
    sr = SuperresolutionHybrid8XDC(channels=32, img_resolution=512, sr_num_fp16_res=0, sr_antialias=True, large_sr=True, channel_base=32768,
                                   channel_max=512, fused_modconv_default='inference_only').eval()
    sr.load_state_dict(syn.make_sr_large_params(seed=8, n_res=2), strict=True)
    g = load('render_full48')
    fimg = torch.from_numpy(g['rgb']).permute(0, 2, 1).reshape(1, 32, 64, 64).contiguous()
    img = sr(fimg[:, :3], fimg, torch.ones(1, 14, 512), noise_mode='none')
    save('sr_large', image=img, seeds=np.array([8]), n_res=2)


def ref_small_case():
    """The reference's renderer wired as oracle/ref_runner.py runs it for the CPU baseline: N=1, 3x32x32x32 planes, 16^2 rays, 12 (+12)
    samples; inputs come from seeds."""
    N, res, S = 1, 16, 12
    planes, cam = syn.make_planes(N, h=32, w=32, seed=0), syn.make_cameras(N, seed=1)
    dec = ref_decoder(syn.make_decoder_params(seed=4))
    out = {}
    for S_imp in (0, 12):
        u_c, u_f = syn.make_jitter(N, res * res, S, S_imp, seed=2)
        _, _, rgb, depth, wsum, valid = ref_render(planes, dec, cam, res, S, S_imp, u_c, u_f)
        out.update({f'imp{S_imp}.rgb': rgb, f'imp{S_imp}.depth': depth, f'imp{S_imp}.wsum': wsum, f'imp{S_imp}.valid': valid})
    save('render_ref_small', res=res, S=S, seeds=np.array([0, 1, 2, 4]), **out)


def load(name):
    return np.load(os.path.join(HERE, name + '.npz'))


if __name__ == '__main__':
    torch.manual_seed(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'warp':
        warp_case()
        warp_case('v1'); warp_case('v3')
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'large_sr':
        large_sr_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'trigrid':
        trigrid_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'ref_small':
        ref_small_case()
        sys.exit(0)
    small_cases()
    layer_cases()
    full_cases()
    warp_case()
    warp_case('v1'); warp_case('v3')
    trigrid_case()
    large_sr_case()
    ref_small_case()
