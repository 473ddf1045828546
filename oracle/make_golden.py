"""Pins oracle/pf_oracle.py against the real reference and writes tests/golden/*.npz.

Run in the build container only (needs /root/reference):   python -m oracle.make_golden
The reference is imported unmodified through oracle/shims (stand-ins for mmengine/timm/... that are not installed
offline), loaded with `synthetic_state_dict(cfg, seed)` and executed on CPU fp32.  Every stage is compared with the
restatement (assert), and strided samples of the reference outputs are stored as fixtures so the same check can be
repeated where the reference tree does not exist (GPU box, CI): tests/test_oracle_golden.py.
"""
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import pf_oracle as po          # noqa: E402
from oracle import ref_harness as rh        # noqa: E402
from patchfusion_b200.configs import depth_anything_patchfusion      # noqa: E402
from patchfusion_b200.params import synthetic_state_dict             # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
CASE = dict(encoder='vits', seed=0, image_raw_shape=(1080, 1920), patch_split_num=(2, 2), process_num=2,
            input_seed=0, sample_stride=8)        # stride 8 keeps tests/golden/vits_case0.npz under 1 MB


def sample(t, stride):
    return t[..., ::stride, ::stride].contiguous().numpy()


def stats(t):
    t = t.double()
    return np.array([t.mean().item(), t.std().item(), t.abs().max().item()], dtype=np.float64)


def case_inputs(case):
    cfg = depth_anything_patchfusion(case['encoder'], image_raw_shape=case['image_raw_shape'],
                                     patch_split_num=case['patch_split_num'])
    sd = synthetic_state_dict(cfg, seed=case['seed'])
    g = torch.Generator().manual_seed(case['input_seed'])
    img = torch.rand(1, 3, *case['image_raw_shape'], generator=g)
    return cfg, sd, img


def main():
    torch.set_num_threads(os.cpu_count())
    case = CASE
    cfg, sd, img = case_inputs(case)
    ref = rh.build_reference(case['encoder'], cfg)
    print(ref.load_state_dict(sd, strict=True))
    orc = po.Oracle(sd, cfg)
    lr = ref.resizer(img)
    assert torch.equal(lr, orc.resizer(img))
    out, st = {}, case['sample_stride']
    with torch.no_grad():
        # ---- coarse branch + taps
        d_ref, f_ref = ref.coarse_forward(lr)
        d_o, f_o = orc.coarse(lr)
        assert (d_ref - d_o).abs().max() < 1e-5
        out['coarse_depth'] = sample(d_ref, st)
        for i, (a, b) in enumerate(zip(f_ref, f_o)):
            assert (a - b).abs().max() < 1e-4 * a.abs().max()
            out['coarse_feat%d_stats' % i] = stats(a)
            out['coarse_feat%d' % i] = sample(a, st if a.shape[-1] > 100 else 1)[:, :8]
        # ---- ROI crop-zoom (torchvision roi_align inside the reference)
        h, w = case['image_raw_shape'][0] // 2, case['image_raw_shape'][1] // 2
        raw = [(0, 0), (h // 2, w // 2)]
        P = cfg['patch_process_shape']
        fx, fy = 1 / case['image_raw_shape'][1] * P[1], 1 / case['image_raw_shape'][0] * P[0]
        boxes = torch.tensor([[x, y, x + w, y + h] for (y, x) in raw]).int() * torch.tensor([[fx, fy, fx, fy]])
        bf = torch.cat([torch.arange(2).unsqueeze(1).float(), boxes], 1)
        post = ref.coarse_postprocess_test(bboxs=None, bboxs_feat=bf, coarse_prediction=d_ref, coarse_features=f_ref)
        rois_o = [po.roi_crop_zoom(f, boxes, f.shape[-2] / P[0]) for f in f_o]
        for i, (a, b) in enumerate(zip(post['coarse_feats_roi'], rois_o)):
            print('roi', i, (a - b).abs().max().item(), a.abs().max().item())
            assert (a - b).abs().max() < 2e-5 * max(1.0, a.abs().max().item())
        out['roi_feat4'] = sample(post['coarse_feats_roi'][4], st)[:, :8]
        # ---- fine branch + fusion on the two tiles
        crops = torch.cat([ref.resizer(img[:, :, y:y + h, x:x + w]) for (y, x) in raw])
        fd_ref, ff_ref = ref.fine_forward(crops)
        fd_o, ff_o = po.branch_forward(sd, 'fine_branch.', crops, cfg['fine_branch'])
        assert (fd_ref - fd_o).abs().max() < 1e-5
        out['fine_depth'] = sample(fd_ref, st)
        bff = bf.clone()
        bff[:, 0] = 0
        fu_ref, _ = ref.fusion_forward(fd_ref, crops, f_ref, ff_ref, bff, **post)
        g2l = po.g2l_all(sd, f_o, cfg['guided_fusion'])
        for i in range(6):
            g_ref = ref.guided_fusion.g2l_list[i](f_ref[i], None)
            print('g2l', i, (g_ref - g2l[i]).abs().max().item(), g_ref.abs().max().item())
            assert (g_ref - g2l[i]).abs().max() < 1e-4
            out['g2l%d_stats' % i] = stats(g_ref)
        out['g2l4'] = sample(g_ref if False else ref.guided_fusion.g2l_list[4](f_ref[4], None), st)[:, :8]
        fu_o = po.fusion_forward(sd, cfg, fd_o, crops, ff_o, boxes, rois_o and po.roi_crop_zoom(d_o, boxes, 1.0),
                                 rois_o, g2l)
        print('fusion', (fu_ref - fu_o).abs().max().item(), fu_ref.min().item(), fu_ref.max().item())
        assert (fu_ref - fu_o).abs().max() < 1e-3 * fu_ref.abs().max()
        out['fusion_depth'] = sample(fu_ref, st)
        # ---- whole forward(mode='infer')
        for mode in ('m1', 'm2', 'r4'):
            random.seed(0)
            y_ref, _ = ref(mode='infer', image_lr=lr, image_hr=img, cai_mode=mode, process_num=case['process_num'])
            random.seed(0)
            y_o = orc.infer(lr, img, cai_mode=mode, process_num=case['process_num'])
            err = (y_ref - y_o).abs().max().item()
            print(mode, tuple(y_ref.shape), 'max|ref-oracle| =', err)
            assert err < 1e-3 * y_ref.abs().max()
            out['infer_' + mode] = sample(y_ref, st)
    os.makedirs(GOLD, exist_ok=True)
    np.savez_compressed(os.path.join(GOLD, 'vits_case0.npz'), **out)
    json.dump({k: (list(v) if isinstance(v, tuple) else v) for k, v in case.items()},
              open(os.path.join(GOLD, 'vits_case0.json'), 'w'))
    print('wrote', os.path.join(GOLD, 'vits_case0.npz'))


def main_default_init():
    """Second reference-pinned fixture: weights drawn from the reference constructor's own distributions
    (params.default_init_state_dict; per-tensor statistics checked against a freshly constructed reference model), the
    reference's outputs for coarse / fine+fusion / m1 stored as strided samples (tests/golden/vits_default0.*)."""
    from patchfusion_b200.params import default_init_state_dict
    torch.set_num_threads(os.cpu_count())
    case = dict(encoder='vits', seed=7, image_raw_shape=(1080, 1920), patch_split_num=(2, 2), process_num=2,
                input_seed=1, sample_stride=4, init='default')
    cfg = depth_anything_patchfusion(case['encoder'], image_raw_shape=case['image_raw_shape'],
                                     patch_split_num=case['patch_split_num'])
    ref = rh.build_reference(case['encoder'], cfg)
    ref_sd = {k: v.clone() for k, v in ref.state_dict().items()}        # the reference's OWN default construction
    sd = default_init_state_dict(cfg, seed=case['seed'])
    assert list(sd) == list(ref_sd)
    bad = []
    for k, v in ref_sd.items():
        if v.dtype != torch.float32 or v.numel() < 4096:
            continue
        a, b = v.double().std().item(), sd[k].double().std().item()
        if abs(a - b) > 0.1 * max(a, 1e-12) + 1e-9:
            bad.append((k, a, b))
    assert not bad, bad[:5]
    for k, v in ref_sd.items():                                           # small tensors: same constants / scale
        if v.dtype == torch.float32 and v.numel() < 4096 and v.numel() > 1 and v.std() == 0:
            assert torch.equal(v, sd[k]), k
    print('default-init statistics match the reference constructor on', len(ref_sd), 'tensors')
    print(ref.load_state_dict(sd, strict=True))
    g = torch.Generator().manual_seed(case['input_seed'])
    img = torch.rand(1, 3, *case['image_raw_shape'], generator=g)
    orc = po.Oracle(sd, cfg)
    lr = ref.resizer(img)
    out, st = {}, case['sample_stride']
    with torch.no_grad():
        d_ref, f_ref = ref.coarse_forward(lr)
        d_o, f_o = orc.coarse(lr)
        assert (d_ref - d_o).abs().max() < 1e-5
        out['coarse_depth'] = sample(d_ref, st)
        for i, a in enumerate(f_ref):
            out['coarse_feat%d_stats' % i] = stats(a)
        random.seed(0)
        y_ref, _ = ref(mode='infer', image_lr=lr, image_hr=img, cai_mode='m1', process_num=case['process_num'])
        y_o = orc.infer(lr, img, cai_mode='m1', process_num=case['process_num'])
        err = (y_ref - y_o).abs().max().item()
        print('m1', tuple(y_ref.shape), 'max|ref-oracle| =', err, 'range', y_ref.min().item(), y_ref.max().item())
        assert err < 1e-4
        out['infer_m1'] = sample(y_ref, st)
    np.savez_compressed(os.path.join(GOLD, 'vits_default0.npz'), **out)
    json.dump({k: (list(v) if isinstance(v, tuple) else v) for k, v in case.items()},
              open(os.path.join(GOLD, 'vits_default0.json'), 'w'))
    print('wrote vits_default0')


def main_vitl_tile():
    """vitl-size fixture (SURVEY build-plan step 1): the reference's coarse depth and ONE fused 4K tile."""
    torch.set_num_threads(os.cpu_count())
    case = dict(encoder='vitl', seed=0, image_raw_shape=(2160, 3840), patch_split_num=(4, 4), input_seed=3,
                sample_stride=4, tile=(540, 960))
    cfg, sd, img = case_inputs(case)
    ref = rh.build_reference(case['encoder'], cfg)
    print(ref.load_state_dict(sd, strict=True))
    orc = po.Oracle(sd, cfg)
    lr = ref.resizer(img)
    out, st = {}, case['sample_stride']
    H, W = case['image_raw_shape']
    h, w = H // 4, W // 4
    y, x = case['tile']
    P = cfg['patch_process_shape']
    with torch.no_grad():
        d_ref, f_ref = ref.coarse_forward(lr)
        d_o, f_o = orc.coarse(lr)
        print('coarse', (d_ref - d_o).abs().max().item())
        assert (d_ref - d_o).abs().max() < 1e-4
        out['coarse_depth'] = sample(d_ref, st)
        fx, fy = 1 / W * P[1], 1 / H * P[0]
        boxes = torch.tensor([[x, y, x + w, y + h]]).int() * torch.tensor([[fx, fy, fx, fy]])
        bf = torch.cat([torch.zeros(1, 1), boxes], 1)
        post = ref.coarse_postprocess_test(bboxs=None, bboxs_feat=bf, coarse_prediction=d_ref, coarse_features=f_ref)
        crop = ref.resizer(img[:, :, y:y + h, x:x + w])
        fd_ref, ff_ref = ref.fine_forward(crop)
        fu_ref, _ = ref.fusion_forward(fd_ref, crop, f_ref, ff_ref, bf, **post)
        g2l = po.g2l_all(sd, f_o, cfg['guided_fusion'])
        tc = po.prepare_tile_cfg((H, W), (4, 4), P)
        fu_o = orc.tiles(img, [(y, x)], d_o, f_o, g2l, 1, tc)
        print('fusion', (fu_ref - fu_o).abs().max().item(), fu_ref.min().item(), fu_ref.max().item())
        assert (fu_ref - fu_o).abs().max() < 1e-3 * fu_ref.abs().max()
        out['fine_depth'] = sample(fd_ref, st)
        out['fusion_depth'] = sample(fu_ref, st)
    np.savez_compressed(os.path.join(GOLD, 'vitl_tile0.npz'), **out)
    json.dump({k: (list(v) if isinstance(v, tuple) else v) for k, v in case.items()},
              open(os.path.join(GOLD, 'vitl_tile0.json'), 'w'))
    print('wrote vitl_tile0')


if __name__ == '__main__':
    which = sys.argv[1] if len(sys.argv) > 1 else 'vits'
    {'vits': main, 'default': main_default_init, 'vitl': main_vitl_tile}[which]()
