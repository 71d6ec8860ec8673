"""Golden vectors from the reference's own CUDA extensions (GPU only): runs ``oracle/_ref/pairwise_ext_ref*.so`` and
``oracle/_ref/tree_filter_cuda_ref*.so`` (mmdet/ops/pairwise/csrc and mmdet/ops/tree_filter/src compiled unmodified by
oracle/Makefile) on the inputs the GPU tests build, and writes

  * tests/golden/reference_ext.npz      -- tests/test_reference_ext_gpu.py (rows a7, a12, a13, a15)
  * tests/golden/config_a_reference.npz -- tests/test_config_a_gpu.py (config A at full size: the reference's pairwise op
                                           inside a restatement of CondInstMaskHead.loss, condinst_head.py:1288-1343)

An output of more than tests.helpers.GOLDEN_FULL elements is stored as a seeded sample of its elements (``key.idx`` /
``key.val``, half of the sample drawn among the non-zero elements) and as ``tests.helpers.projections`` of the whole tensor.

      python -m oracle.make_golden_ref_ext [OUT_DIR]"""
import glob
import importlib.util
import os
import sys

import numpy as np
import torch

from oracle.make_golden import OUT
from tests import test_reference_ext_gpu as T
from tests.helpers import GOLDEN_FULL, projections

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMPLE = 2048


def load_ref(name):
    hits = glob.glob(os.path.join(ROOT, 'oracle', '_ref', name + '*.so'))
    assert hits, f'oracle/_ref/{name}*.so is missing: build it with `make -C oracle` next to the reference checkout'
    spec = importlib.util.spec_from_file_location(name, hits[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def store(out, key, t):
    a = t.detach().cpu().numpy()
    if a.size <= GOLDEN_FULL:
        out[key] = a
        return
    flat = a.reshape(-1)
    rng = np.random.default_rng(a.size)
    nz = np.flatnonzero(flat)
    pick = rng.choice(nz, min(SAMPLE // 2, nz.size), replace=False) if nz.size else np.zeros(0, np.int64)
    idx = np.unique(np.concatenate([pick, rng.choice(flat.size, SAMPLE - pick.size, replace=False)]))
    out[key + '.shape'] = np.array(a.shape, np.int64)
    out[key + '.idx'] = idx.astype(np.int32)
    out[key + '.val'] = flat[idx]
    out[key + '.proj'] = projections(t)


def reference_ext(out):
    pw_ext, tf_ext = load_ref('pairwise_ext_ref'), load_ref('tree_filter_cuda_ref')
    for shape, k, d in T.PAIRWISE_CASES:
        x, g = T.pairwise_inputs(shape, k)
        key = T.pairwise_key(shape, k, d)
        pw = pw_ext.pairwise_nlog_forward(k, d, x)
        store(out, key + '.pw', pw)
        store(out, key + '.gx', pw_ext.pairwise_nlog_backward(k, d, x, pw, g))
    for B, C, h, w in T.MST_CASES:
        index, weight = T.mst_problem(B, C, h, w)
        out[f'mst_{B}_{C}_{h}_{w}'] = T.edge_set(tf_ext.mst_forward(index.clone(), weight.clone(), h * w)).astype(np.int32)
    for B, C, h, w in T.REFINE_CASES:
        key = f'refine_{B}_{C}_{h}_{w}'
        idx, par, chd = T.refine_order(B, h, w)
        for n, t in (('idx', idx), ('par', par), ('chd', chd)):
            out[f'{key}.{n}'] = t.cpu().numpy()
        feat, ew, gout = T.refine_inputs(B, C, h * w)
        r = tf_ext.refine_forward(feat, ew.clone(), idx.clone(), par.clone(), chd.clone())    # theirs writes entry 0 in place
        ew0 = ew.clone(); ew0[:, 0] = 0
        par0 = par.clone(); par0[:, 0] = 0
        store(out, key + '.out', r[0])
        store(out, key + '.gf', tf_ext.refine_backward_feature(feat, ew0, idx, par0, chd, *r[:5], gout))
        store(out, key + '.gw', tf_ext.refine_backward_weight(feat, ew0, idx, par0, chd, *r[:5], gout)[:, 1:])
    tree, feat, ew, gout = T.bfs_problem()
    ridx, rpar, rchd = tf_ext.bfs_forward(tree.clone(), 4)
    for n, t in (('idx', ridx), ('par', rpar), ('chd', rchd)):
        out['bfs.' + n] = t.cpu().numpy()
    r = tf_ext.refine_forward(feat, ew.clone(), ridx.clone(), rpar.clone(), rchd.clone())
    for i, t in enumerate(r):
        store(out, f'bfs.out{i}', t)
    ew0 = ew.clone(); ew0[:, 0] = 0
    par0 = rpar.clone(); par0[:, 0] = 0
    store(out, 'bfs.gf', tf_ext.refine_backward_feature(feat, ew0, ridx, par0, rchd, *r[:5], gout))
    store(out, 'bfs.gw', tf_ext.refine_backward_weight(feat, ew0, ridx, par0, rchd, *r[:5], gout)[:, 1:])


def config_a(out):
    import bench
    from boxinstseg_b200.ops.boxinst import boxinst_targets
    ext = load_ref('pairwise_ext_ref')
    dev = torch.device('cuda:0')
    case = bench.synthetic_case(1234)

    class RefPairwise(torch.autograd.Function):            # mmdet/ops/pairwise/pairwise.py:6-26
        @staticmethod
        def forward(ctx, logits, size, dilation):
            pw = ext.pairwise_nlog_forward(size, dilation, logits)
            ctx.save_for_backward(logits, pw)
            ctx.cfg = (size, dilation)
            return pw

        @staticmethod
        def backward(ctx, g):
            logits, pw = ctx.saved_tensors
            return ext.pairwise_nlog_backward(ctx.cfg[0], ctx.cfg[1], logits, pw, g.contiguous()), None, None

    t = boxinst_targets(case['img'].to(dev), case['metas'], [b.to(dev) for b in case['gt_bboxes']], want_similarity=True)
    gi = case['gt_inds'].to(dev)
    sim = t.similarity[case['img_inds'].to(dev)]                       # the G-fold gather of condinst_head.py:1316
    bm = torch.cat(t.bitmasks())[gi][:, None]
    x = case['logits'].to(dev).requires_grad_(True)

    def dice(a, b):                                                    # condinst_head.py:117-131
        a, b = a.flatten(1), b.flatten(1)
        return 1.0 - 2.0 * (a * b).sum(1) / ((a * a).sum(1) + (b * b).sum(1) + 1e-5)

    scores = x.sigmoid()
    prj = (dice(scores.max(dim=2, keepdim=True)[0], bm.max(dim=2, keepdim=True)[0]) +
           dice(scores.max(dim=3, keepdim=True)[0], bm.max(dim=3, keepdim=True)[0])).mean()      # :134-143
    w = (sim >= 0.3).float() * bm
    pair = (RefPairwise.apply(x, 3, 2) * w).sum() / w.sum().clamp(min=1.0)                        # :1318-1332
    (g,) = torch.autograd.grad(prj + pair, x)
    out['loss_prj'] = np.float64(prj.item())
    out['loss_pairwise'] = np.float64(pair.item())
    store(out, 'grad', g)


def main():
    dst = sys.argv[1] if len(sys.argv) > 1 else OUT
    os.makedirs(dst, exist_ok=True)
    for name, fill in (('reference_ext', reference_ext), ('config_a_reference', config_a)):
        out = {}
        fill(out)
        torch.cuda.synchronize()
        np.savez_compressed(os.path.join(dst, name + '.npz'), **out)
        print(name, sorted(out))


if __name__ == '__main__':
    main()
