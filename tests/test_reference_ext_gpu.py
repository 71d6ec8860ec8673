"""GPU parity against the REFERENCE'S OWN CUDA kernels (mmdet/ops/pairwise/csrc/pairwise, mmdet/ops/tree_filter/src),
through golden vectors: oracle/make_golden_ref_ext.py runs the reference's extensions, compiled unmodified by oracle/Makefile,
on the inputs built here and stores their outputs in tests/golden/reference_ext.npz.  These tests pin rows a7, a12, a13, a15
on the reference itself rather than on restatements.  Large outputs are stored as a seeded sample plus random projections
(tests/helpers.py, check_golden)."""
import numpy as np
import pytest
import torch

from tests.helpers import check_golden, rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
PAIRWISE_CASES = [((3, 1, 37, 53), 3, 2), ((2, 1, 16, 64), 3, 1), ((2, 1, 40, 70), 5, 2), ((4, 1, 200, 256), 3, 2)]
MST_CASES = [(2, 3, 24, 40), (1, 5, 50, 64)]
REFINE_CASES = [(2, 4, 24, 40), (1, 1, 50, 64)]


@pytest.fixture(scope='module')
def ref(golden):
    return golden('reference_ext')


# ------------------------------------------------------------------ a7: pairwise_nlog (pairwise.cu:68-149)
def pairwise_inputs(shape, k):
    gen = torch.Generator().manual_seed(3)
    x = (torch.randn(shape, generator=gen) * 3).to(DEV)
    x.view(-1)[:4] = torch.tensor([45.0, -45.0, 30.0, -60.0], device=DEV)[: min(4, x.numel())]
    g = torch.rand(shape[0], k * k - 1, *shape[2:], generator=gen).to(DEV)
    return x, g


def pairwise_key(shape, k, d):
    return 'pairwise_' + '_'.join(map(str, (*shape, k, d)))


@pytest.mark.parametrize('shape,k,d', PAIRWISE_CASES)
def test_pairwise_matches_reference_cuda(ref, shape, k, d):
    from boxinstseg_b200.ops.pairwise import pairwise_ext as ours
    x, g = pairwise_inputs(shape, k)
    key = pairwise_key(shape, k, d)
    pw = ours.pairwise_nlog_forward(k, d, x)
    check_golden(ref, key + '.pw', pw, rtol=1e-4, atol=1e-5, rel=1e-4)
    gx = ours.pairwise_nlog_backward(k, d, x, pw, g)
    check_golden(ref, key + '.gx', gx, rtol=1e-3, atol=1e-5, rel=1e-4)     # theirs: float atomics


# ------------------------------------------------------------------ a12 / a13 / a15: tree filter (src/mst, src/bfs, src/refine)
def _grid_problem(B, C, h, w, seed):
    from boxinstseg_b200.ops.tree_filter import MinimumSpanningTree, TreeFilter2D
    gen = torch.Generator().manual_seed(seed)
    guide = torch.randn(B, C, h, w, generator=gen).to(DEV)
    mst = MinimumSpanningTree(TreeFilter2D.norm2_distance)
    index = mst._build_matrix_index(guide).contiguous()
    weight = mst._build_feature_weight(guide)
    return guide, index, weight


def edge_set(tree):
    """[B, V-1, 2] tree edges -> per batch, the (min, max) vertex pairs in lexicographic order."""
    e = np.sort(tree.cpu().numpy().astype(np.int64), axis=-1)
    return np.stack([eb[np.lexsort((eb[:, 1], eb[:, 0]))] for eb in e])


def mst_problem(B, C, h, w):
    _, index, weight = _grid_problem(B, C, h, w, seed=h)
    return index, weight


@pytest.mark.parametrize('B,C,h,w', MST_CASES)
def test_mst_edge_set_matches_reference(ref, B, C, h, w):
    from boxinstseg_b200.ops.tree_filter import tree_filter_cuda as ours
    index, weight = mst_problem(B, C, h, w)
    t = ours.mst_forward(index, weight, h * w)
    assert np.array_equal(edge_set(t), ref[f'mst_{B}_{C}_{h}_{w}'])


def refine_order(B, h, w):
    """(sorted_index, sorted_parent, sorted_child) of a random grid tree: the BFS order both implementations are fed (stored
    with the golden outputs, so that the check does not depend on how our own MST / BFS order a tree)."""
    from boxinstseg_b200.ops.tree_filter import tree_filter_cuda as ours
    _, index, weight = _grid_problem(B, 3, h, w, seed=7 * h)
    return ours.bfs_forward(ours.mst_forward(index, weight, h * w), 4)


def refine_inputs(B, C, V):
    gen = torch.Generator().manual_seed(1)
    feat = torch.rand(B, C, V, generator=gen).to(DEV)
    ew = torch.rand(B, V, generator=gen).to(DEV) * 0.9 + 0.05     # edge weights in (0, 1), entry 0 ignored
    gout = torch.randn(B, C, V, generator=gen).to(DEV)
    return feat, ew, gout


@pytest.mark.parametrize('B,C,h,w', REFINE_CASES)
def test_refine_matches_reference_cuda(ref, B, C, h, w):
    from boxinstseg_b200.ops.tree_filter import tree_filter_cuda as ours
    key = f'refine_{B}_{C}_{h}_{w}'
    idx, par, chd = (torch.from_numpy(ref[f'{key}.{n}']).to(DEV) for n in ('idx', 'par', 'chd'))
    feat, ew, gout = refine_inputs(B, C, h * w)
    o = ours.refine_forward(feat, ew, idx, par, chd)
    check_golden(ref, key + '.out', o[0], rtol=1e-3, atol=1e-5, rel=1e-5)
    gf = ours.refine_backward_feature(feat, ew, idx, par, chd, o[0], o[1], o[2], o[3], o[4], gout)
    check_golden(ref, key + '.gf', gf, rel=1e-5)
    gw = ours.refine_backward_weight(feat, ew, idx, par, chd, o[0], o[1], o[2], o[3], o[4], gout)
    check_golden(ref, key + '.gw', gw[:, 1:], rel=1e-4)            # entry 0 is the root (no edge)


def bfs_problem():
    from boxinstseg_b200.ops.tree_filter import tree_filter_cuda as ours
    B, C, h, w = 2, 2, 20, 28
    _, index, weight = _grid_problem(B, 3, h, w, seed=11)
    V = h * w
    tree = ours.mst_forward(index, weight, V)
    gen = torch.Generator().manual_seed(2)
    feat = torch.rand(B, C, V, generator=gen).to(DEV)
    gout = torch.randn(B, C, V, generator=gen).to(DEV)
    ew = torch.rand(B, V, generator=gen).to(DEV) * 0.9 + 0.05          # per position of the REFERENCE order
    return tree, feat, ew, gout


def test_reference_bfs_order_is_accepted(ref):
    """The reference's own (racy, any parent-before-child) BFS order, fed to OUR refine entry points, gives the
    reference's results: the shim adopts foreign orders (tree_filter_cuda._adopt) instead of assuming its own."""
    from boxinstseg_b200.ops.tree_filter import tree_filter_cuda as ours
    tree, feat, ew, gout = bfs_problem()
    B, V = ew.shape
    ridx, rpar, rchd = (torch.from_numpy(ref['bfs.' + n]).to(DEV) for n in ('idx', 'par', 'chd'))
    o = ours.refine_forward(feat, ew, ridx, rpar, rchd)
    for i, a in enumerate(o):
        check_golden(ref, f'bfs.out{i}', a, rel=1e-5)
    gf = ours.refine_backward_feature(feat, ew, ridx, rpar, rchd, o[0], o[1], o[2], o[3], o[4], gout)
    check_golden(ref, 'bfs.gf', gf, rel=1e-5)
    gw = ours.refine_backward_weight(feat, ew, ridx, rpar, rchd, o[0], o[1], o[2], o[3], o[4], gout)
    check_golden(ref, 'bfs.gw', gw[:, 1:], rel=1e-4)
    # and the same tree through our own deterministic order gives the same filter output
    idx, par, chd = ours.bfs_forward(tree, 4)
    wv = torch.zeros(B, V, device=DEV).scatter_(1, ridx.long(), ew)   # weight of the edge (vertex -> parent), by vertex id
    o2 = ours.refine_forward(feat, torch.gather(wv, 1, idx.long()), idx, par, chd)[0]
    assert rel_err(o2, o[0]) <= 1e-5
