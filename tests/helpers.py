"""Shared helpers for the GPU parity tests: seeded synthetic inputs (SURVEY.md section 8d)."""
import numpy as np
import torch
import torch.nn.functional as F

MEAN = [123.675, 116.28, 103.53]
STD = [58.395, 57.12, 57.375]


def synth_image(gen, h, w, lowres=32, noise=8.0):
    """uint8-valued RGB [3,h,w] float32: low-frequency field + N(0,noise) noise."""
    coarse = torch.rand(1, 3, max(h // lowres, 2), max(w // lowres, 2), generator=gen) * 255
    img = F.interpolate(coarse, size=(h, w), mode='bilinear', align_corners=False)[0]
    return (img + torch.randn(3, h, w, generator=gen) * noise).clamp(0, 255).floor()


def normalise(raw):
    return (raw - torch.tensor(MEAN).view(3, 1, 1)) / torch.tensor(STD).view(3, 1, 1)


def make_meta(ih, iw, ori_scale=1.0):
    return dict(img_shape=(ih, iw, 3), ori_shape=(int(ih * ori_scale), int(iw * ori_scale), 3),
                img_norm_cfg=dict(mean=np.array(MEAN, dtype=np.float32), std=np.array(STD, dtype=np.float32),
                                  to_rgb=True))


def synth_boxes(gen, num, hp, wp, lo=48, hi=400):
    hi_w, hi_h = min(hi, wp - 1), min(hi, hp - 1)
    w = torch.rand(num, generator=gen) * (hi_w - min(lo, hi_w)) + min(lo, hi_w)
    h = torch.rand(num, generator=gen) * (hi_h - min(lo, hi_h)) + min(lo, hi_h)
    x1 = torch.rand(num, generator=gen) * (wp - w)
    y1 = torch.rand(num, generator=gen) * (hp - h)
    return torch.stack([x1, y1, x1 + w, y1 + h], 1).float()


def boxinst_case(seed, B, hp, wp, gts_per_img, inst_per_gt, logit_std=2.0, ragged=False, lowres=32, noise=8.0):
    """Inputs of one BoxInst mask-loss step (config A when B=2, 800x1024, 8 GT, 8 inst/GT)."""
    gen = torch.Generator().manual_seed(seed)
    imgs, metas = [], []
    for b in range(B):
        ih, iw = (hp, wp) if not (ragged and b % 2) else (hp - 8 * (b % 3 + 1), wp - 12)
        raw = synth_image(gen, ih, iw, lowres, noise)
        imgs.append(F.pad(normalise(raw), (0, wp - iw, 0, hp - ih)))
        metas.append(make_meta(ih, iw, ori_scale=1.0 if not ragged else 1.7))
    img = torch.stack(imgs)
    gt_bboxes = [synth_boxes(gen, gts_per_img, hp, wp, hi=min(400, hp // 2)) for _ in range(B)]
    gt_inds = torch.arange(B * gts_per_img).repeat_interleave(inst_per_gt)
    img_inds = gt_inds // gts_per_img
    n = gt_inds.numel()
    logits = torch.randn(n, 1, hp // 4, wp // 4, generator=gen) * logit_std
    return dict(img=img, metas=metas, gt_bboxes=gt_bboxes, gt_inds=gt_inds, img_inds=img_inds, logits=logits)


def rel_err(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


GOLDEN_FULL = 4096      # a stored reference output with more elements is kept as a seeded sample + projections


def projections(t, k=16):
    """k random projections of the flattened tensor, one per contiguous block of its elements (float64, seeded)."""
    v = t.detach().double().flatten().cpu()
    m = -(-v.numel() // k)
    v = F.pad(v, (0, k * m - v.numel()))
    r = torch.randn(m, generator=torch.Generator().manual_seed(m), dtype=torch.float64)
    return (v.view(k, m) @ r).numpy()


def check_golden(g, key, t, rtol=None, atol=0.0, rel=None):
    """``t`` against the reference output stored under ``key`` of the golden file ``g``: allclose(rtol, atol) element-wise on
    what is stored, and rel_err <= rel on what is stored and, for an output stored as a sample (``key.idx`` / ``key.val``),
    on the projections of the whole tensor (``key.proj``), so that every element takes part."""
    t = t.detach().cpu()
    if key in g:
        ref, ours = torch.from_numpy(g[key]), t
        assert ours.shape == ref.shape, (key, ours.shape, ref.shape)
    else:
        assert list(t.shape) == g[key + '.shape'].tolist(), (key, t.shape)
        ref, ours = torch.from_numpy(g[key + '.val']), t.flatten()[torch.from_numpy(g[key + '.idx']).long()]
    if rtol is not None:
        assert torch.allclose(ours.to(ref.dtype), ref, rtol=rtol, atol=atol), key
    if rel is not None:
        assert rel_err(ours, ref) <= rel, (key, rel_err(ours, ref))
        if key not in g:
            err = rel_err(torch.from_numpy(projections(t)), torch.from_numpy(g[key + '.proj']))
            assert err <= rel, (key, 'projections', err)


def host_twin(name):
    """Compiles tests/host_harness/<name>.cpp -- the HOST build of the very header a kernel is made of -- with g++ and
    returns the ctypes handle (test infrastructure: lets the CPU suite check a kernel's arithmetic and indexing bit for bit
    against the oracle on a box without a GPU; the product library exports only the CUDA path)."""
    import ctypes
    import os
    import subprocess
    import tempfile
    here = os.path.dirname(os.path.abspath(__file__))
    src = os.path.join(here, 'host_harness', name + '.cpp')
    out = os.path.join(tempfile.gettempdir(), f'bxs_{name}_{os.getuid()}_{int(os.path.getmtime(src))}.so')
    core = os.path.join(here, '..', 'boxinstseg_b200', 'csrc')
    newest = max(os.path.getmtime(os.path.join(core, f)) for f in os.listdir(core) if f.endswith('.cuh'))
    if not os.path.exists(out) or os.path.getmtime(out) < max(newest, os.path.getmtime(src)):
        subprocess.run(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-x', 'c++', src, '-o', out],
                       check=True)
    return ctypes.CDLL(out)
