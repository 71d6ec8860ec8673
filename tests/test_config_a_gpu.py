"""Config A of BASELINE.json at FULL size (B=2 images of 3x800x1024, 8 GT each, N=128 instances, loss grid 200x256,
seed 1234 = the bench inputs): the fused BoxInst mask loss and its gradient against

  * the CPU oracle (oracle/boxinst.py: restated CondInstMaskHead.loss, float64), and
  * the REFERENCE'S OWN compiled CUDA pairwise op (mmdet/ops/pairwise/csrc, compiled unmodified by oracle/Makefile) inside
    a restatement of condinst_head.py:1288-1343 that materialises what the reference materialises, through the golden
    vectors oracle/make_golden_ref_ext.py stored from it (tests/golden/config_a_reference.npz: both losses, and the
    gradient as a seeded sample of its elements plus random projections of the whole tensor).

Tolerance: 1e-3 relative on loss and gradient (BASELINE.json north_star); observed ~1e-6."""
import os

import pytest
import torch

from tests.helpers import check_golden, rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-3


@pytest.fixture(scope='module')
def case():
    import bench
    return bench.synthetic_case(1234)


@pytest.fixture(scope='module')
def ours(case):
    """(loss_prj, loss_pairwise, gradient) of the CUDA path for upstream gradients (1, 1), with and without a plan."""
    from boxinstseg_b200.ops.boxinst import boxinst_loss_plan, boxinst_mask_loss, boxinst_targets
    dev = torch.device(DEV)
    t = boxinst_targets(case['img'].to(dev), case['metas'], [b.to(dev) for b in case['gt_bboxes']], want_similarity=True)
    it = torch.tensor([10000.0], device=dev)
    gi = case['gt_inds'].to(dev)
    res = []
    for planned in (True, False):
        x = case['logits'].to(dev).requires_grad_(True)
        plan = boxinst_loss_plan(t, gi, x.shape[2], x.shape[3], 2) if planned else None
        prj, pair = boxinst_mask_loss(x, t, gi, it, plan=plan)
        (gx,) = torch.autograd.grad(prj + pair, x)
        res.append((prj.detach(), pair.detach(), gx))
    # the plan is only a precomputed work list: same bits with and without it
    assert torch.equal(res[0][2], res[1][2]) and res[0][0].item() == res[1][0].item() and res[0][1].item() == res[1][1].item()
    return t, res[0]


def test_full_size_against_cpu_oracle(case, ours):
    from oracle import boxinst as ob
    _, (prj, pair, gx) = ours
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    sim, bms = ob.boxinst_targets(case['img'], case['metas'], case['gt_bboxes'])
    x = case['logits'].double().requires_grad_(True)
    bm = torch.cat(bms)[case['gt_inds']][:, None].double()
    p64, q64 = ob.boxinst_mask_loss(x, sim[case['img_inds']].double(), bm, warmup_factor=1.0)
    (g64,) = torch.autograd.grad(p64 + q64, x)
    assert abs(prj.item() - p64.item()) <= TOL * abs(p64.item()), (prj.item(), p64.item())
    assert abs(pair.item() - q64.item()) <= TOL * abs(q64.item()), (pair.item(), q64.item())
    assert rel_err(gx.cpu(), g64) <= TOL
    # element-wise as well: arg-max ties do not occur on continuous random logits
    assert torch.allclose(gx.cpu().double(), g64, rtol=TOL, atol=1e-9)


def test_full_size_against_reference_cuda_extension(golden, ours):
    ref = golden('config_a_reference')
    _, (prj, pair, gx) = ours
    assert abs(prj.item() - ref['loss_prj']) <= TOL * abs(ref['loss_prj'])
    assert abs(pair.item() - ref['loss_pairwise']) <= TOL * abs(ref['loss_pairwise'])
    check_golden(ref, 'grad', gx, rel=TOL)
