#!/usr/bin/env python
"""bench.py -- mask-loss fwd+bwd ms/img (BoxInst R-50, 800x1024, batch 2/GPU) on N B200s.

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` prints ONE JSON line on
rank 0.  N > 1 is launched by torchrun, one rank per GPU; the loss is per image so ranks are
replicas (weak scaling, no data-path collective); rank times are combined with MAX.

What one "step" is (config A of BASELINE.json, synthetic, SURVEY.md section 8d): the BoxInst mask
loss of ONE batch -- 2 images of 3x800x1024, 8 GT boxes each, N=128 sampled instances, loss grid
200x256 -- forward (projection + colour-pairwise terms) and backward (d/d mask_logits).
  value : inputs and targets resident in HBM; timed = the public autograd op, forward + backward (single-pass
          schedule: onepass_main + onepass_finalize + onepass_backward kernels), replayed as a CUDA graph.
  e2e   : through the public head API with HOST (pinned) buffers: H2D of image, logits, boxes ->
          target building (LAB, similarity, rects) -> loss fwd+bwd -> D2H of the gradient + losses.
L2 hygiene: the timed loop rotates over R input/gradient sets whose footprint (R x 52 MB) exceeds
the 126 MB L2, so every step streams its logits from HBM.

``--impl reference`` times the reference's own CPU path (the oracle port, torch-on-CPU with all
host threads) on a bounded sample: ONE image (64 instances) of the same workload per step.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = 'mask_loss_fwd_bwd_ms_per_img'
# the workload both arms name (the reference arm times a bounded per-image sample of it: `cpu_baseline.sample`)
WORKLOAD = ('BoxInst R-50 mask loss fwd+bwd (config A): batch 2/GPU x (3,800,1024), 8 GT/img, '
            'N=128 instances, loss grid 200x256, pairwise 3x3 dil 2')
HP, WP, B_IMG, GTS, INST_PER_GT = 800, 1024, 2, 8, 8
H, W, K_NEIGH = HP // 4, WP // 4, 8
N_INST = B_IMG * GTS * INST_PER_GT
ALGO_BYTES = 3 * N_INST * H * W * 4 + 2 * B_IMG * K_NEIGH * H * W * 4     # SURVEY section 8d: 85.2 MB / step
ROTATE = 8
DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs: the most it writes


def ncu_traffic_bytes():
    """DRAM bytes per step from the committed ncu --set full capture (None when the summary is absent)."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'r2_traffic.json')
    try:
        with open(path) as f:
            return float(json.load(f)['step_dram_bytes'])
    except (OSError, KeyError, ValueError):
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap'}
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.005)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f'nvml_unavailable:{type(e).__name__}')

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def pin_to_numa_node(local_rank, world=1):
    """Keep this rank's host threads (launch loop, pinned-memory staging) on the CPU socket its GPU hangs off: the e2e
    path moves 72 MB / step / rank over PCIe, and round 1's 8-rank e2e lost ~35 % to cross-socket traffic and launch
    contention.  Topology of the 8 x B200 boxes of this pool (SCALE_r01.json): GPUs 0-3 <-> CPUs 0-31,64-95; GPUs 4-7 <->
    CPUs 32-63,96-127.  Best effort: any failure leaves the affinity alone."""
    try:
        ncpu = os.cpu_count() or 0
        if ncpu < 128 or not hasattr(os, 'sched_setaffinity'):
            return None
        half = ncpu // 4
        node = 0 if local_rank < 4 else 1
        cpus = set(range(node * half, (node + 1) * half)) | set(range(2 * half + node * half, 2 * half + (node + 1) * half))
        # one slice of the node per rank so that the ranks of a socket do not fight for the same cores
        per = min(4, max(1, (world + 1) // 2))          # ranks sharing this socket
        mine = sorted(cpus)[(local_rank % 4 % per) * (len(cpus) // per):(local_rank % 4 % per + 1) * (len(cpus) // per)]
        os.sched_setaffinity(0, mine)
        if world > 1:
            torch.set_num_threads(max(1, min(8, len(mine))))
        return f'{mine[0]}-{mine[-1]} ({len(mine)} cpus, numa node {node})'
    except Exception:  # noqa: BLE001
        return None


def ddp_allreduce_leg(dist, dev, world, loss_step, steps):
    """The one exchange step of a data-parallel iteration (SURVEY 8e): the DDP gradient all-reduce of BoxInst R-50,
    ~136 MB fp32 in 25 MB buckets (mmdet/apis/train.py:153-161 wraps the model in MMDistributedDataParallel), NCCL over
    NVLink, issued asynchronously so that it overlaps the mask-loss step.  Returns busbw and the exposed time."""
    total_bytes, bucket_bytes = 136 * 2 ** 20, 25 * 2 ** 20
    sizes = [bucket_bytes] * (total_bytes // bucket_bytes) + ([total_bytes % bucket_bytes] if total_bytes % bucket_bytes else [])
    buckets = [torch.zeros(b // 4, device=dev) for b in sizes]          # zeros: repeated sums stay finite

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier(); torch.cuda.synchronize()
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        dist.barrier(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    def comm_only(i):
        for w_ in [dist.all_reduce(b, async_op=True) for b in buckets]:
            w_.wait()

    def loss_and_comm(i):
        works = [dist.all_reduce(b, async_op=True) for b in buckets]     # NCCL's stream: overlaps the loss kernels
        loss_step(i)
        for w_ in works:
            w_.wait()

    for i in range(3):
        loss_and_comm(i)
    k = max(10, min(steps, 50))
    ms_comm, ms_loss, ms_both = timed(comm_only, k), timed(loss_step, k), timed(loss_and_comm, k)
    t = torch.tensor([ms_comm, ms_loss, ms_both], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_comm, ms_loss, ms_both = t.tolist()
    busbw = 2.0 * (world - 1) / world * total_bytes / (ms_comm * 1e-3) / 1e9
    return {'bytes': total_bytes, 'buckets': len(sizes), 'allreduce_ms': ms_comm, 'allreduce_busbw_gbs': busbw,
            'loss_step_eager_ms': ms_loss, 'loss_step_plus_allreduce_ms': ms_both,
            'exposed_comm_us': max(ms_both - ms_loss, 0.0) * 1e3,
            'what': 'fp32 gradient all-reduce of BoxInst R-50 (136 MB, 25 MB buckets, NCCL, async) overlapped with the eager '
                    'mask-loss step; reported next to the replica metric, not folded into it (the loss itself has no collective)'}


def dump_outputs(out_dir, arrays):
    """Writes what the timed path returned in its last step as <out_dir>/<name>.npy (float64 stays float64, every other dtype
    becomes float32), so that two builds can be compared output for output on the same seeded inputs.  When the arrays exceed
    DUMP_BYTES together, each one larger than an equal share of it is replaced by the same seeded sample of its flattened
    elements on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().cpu().numpy().astype(np.float64 if v.dtype == torch.float64 else np.float32)
              for k, v in arrays.items()}
    share = DUMP_BYTES // len(arrays) - 4096          # room for the .npy header
    over = sum(a.nbytes for a in arrays.values()) > DUMP_BYTES - 4096 * len(arrays)
    for name, a in arrays.items():
        if over and a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def reduce_max_over_ranks(values, dist, device):
    """Per-rank timings -> MAX over ranks (the N>1 contract); identity without a process group."""
    t = torch.tensor(values, device=device, dtype=torch.float64)
    if dist is not None and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def synthetic_case(seed, b_img=B_IMG):
    from tests.helpers import boxinst_case
    # smooth image statistics: about one third of the colour-similarity edges pass the 0.3 threshold (a white-noise
    # image passes ~1 %, which would let the pair kernels skip almost all of their arithmetic)
    return boxinst_case(seed, B=b_img, hp=HP, wp=WP, gts_per_img=GTS, inst_per_gt=INST_PER_GT, lowres=160, noise=3.0)


# ------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline (oracle port, all host threads)
# ------------------------------------------------------------------------------------------
def cpu_step(case):
    from oracle import boxinst as ob
    sim, bms = ob.boxinst_targets(case['img'], case['metas'], case['gt_bboxes'])
    x = case['logits'].clone().requires_grad_(True)
    bm = torch.cat(bms)[case['gt_inds']][:, None]
    prj, pair = ob.boxinst_mask_loss(x, sim[case['img_inds']], bm)
    (prj + pair).backward()
    return float(prj), float(pair)


def run_cpu(steps, warmup):
    cores = min(os.cpu_count() or 1, 32)      # torch CPU ops stop scaling (and oversubscribe) beyond this
    torch.set_num_threads(cores)
    case = synthetic_case(1234, b_img=1)          # bounded sample: ONE image, 64 instances
    for _ in range(warmup):
        cpu_step(case)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cpu_step(case)
        ts.append(time.perf_counter() - t0)
    ms_img = 1e3 * sum(ts) / len(ts)              # one image per step
    return ms_img, cores, '1 image (3x800x1024, 8 GT, 64 instances, loss grid 200x256) per step: targets + loss fwd + bwd, torch CPU'


def main_reference(args, rank, world):
    if rank != 0:
        return
    ms_img, cores, sample = run_cpu(max(args.steps, 1), args.warmup)
    line = {'impl': 'reference', 'metric': METRIC, 'value': ms_img, 'unit': 'ms/img', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_img, 'higher_is_better': False,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'sample': 'one image of the workload per step (the metric is per image): ' + sample},
            'cpu_baseline': {'value': ms_img, 'unit': 'ms/img', 'cores': cores, 'cores_available': os.cpu_count(),
                             'cores_note': 'torch intra-op threads capped at 32: the oracle port (elementwise torch ops on '
                                           '[64,8,200,256] tensors) does not scale beyond that', 'kind': 'port', 'sample': sample},
            'e2e': {'value': ms_img, 'unit': 'ms/img', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# The reference's own GPU path for the same loss (baseline only): its unmodified CUDA pairwise op, compiled by
# oracle/Makefile into oracle/_ref/, inside a restatement of CondInstMaskHead.loss (condinst_head.py:1288-1343) that
# materialises what the reference materialises (per-instance similarity [N,8,H,W], bitmask [N,1,H,W], pairwise [N,8,H,W]).
# ------------------------------------------------------------------------------------------
def run_gpu_reference(case, dev, iters=10, ours_grad=None):
    import glob
    import importlib.util
    hits = glob.glob(os.path.join(ROOT, 'oracle', '_ref', 'pairwise_ext_ref*.so'))
    if not hits:
        return None
    from boxinstseg_b200.ops.boxinst import boxinst_targets
    spec = importlib.util.spec_from_file_location('pairwise_ext_ref', hits[0])
    ext = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ext)

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
    sim = t.similarity[case['img_inds'].to(dev)]                       # [N,8,H,W]: the G-fold gather of condinst_head.py:1316
    bm = torch.cat(t.bitmasks())[gi][:, None]                          # [N,1,H,W]
    x = case['logits'].to(dev).requires_grad_(True)

    def dice(a, b):                                                    # condinst_head.py:117-131
        a, b = a.flatten(1), b.flatten(1)
        return 1.0 - 2.0 * (a * b).sum(1) / ((a * a).sum(1) + (b * b).sum(1) + 1e-5)

    def step():
        scores = x.sigmoid()
        prj = (dice(scores.max(dim=2, keepdim=True)[0], bm.max(dim=2, keepdim=True)[0]) +
               dice(scores.max(dim=3, keepdim=True)[0], bm.max(dim=3, keepdim=True)[0])).mean()     # :134-143
        pw = RefPairwise.apply(x, 3, 2)
        w = (sim >= 0.3).float() * bm
        pair = (pw * w).sum() / w.sum().clamp(min=1.0)                                              # :1318-1332
        x.grad = None
        (prj + pair).backward()
        return prj, pair

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        prj, pair = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    grad_err = None
    if ours_grad is not None:
        grad_err = float((ours_grad.double() - x.grad.double()).norm() / x.grad.double().norm())
    return {'value': ms / B_IMG, 'unit': 'ms/img', 'ms_per_step': ms, 'iters': iters, '_grad_rel_err': grad_err,
            'what': "restated CondInstMaskHead.loss (condinst_head.py:1288-1343) on this GPU around the reference's own "
                    'unmodified CUDA pairwise op (oracle/_ref/pairwise_ext_ref, built by oracle/Makefile); targets precomputed, '
                    'eager PyTorch as in the reference',
            'loss_prj': float(prj.detach()), 'loss_pairwise': float(pair.detach())}


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
FWD_BYTES = N_INST * H * W * 4 + B_IMG * K_NEIGH * H * W * 4            # read logits + similarity      (29.5 MB)
BWD_BYTES = 2 * N_INST * H * W * 4 + B_IMG * K_NEIGH * H * W * 4        # re-read logits, write gradient (55.7 MB)
ONEPASS_BYTES = 2 * N_INST * H * W * 4 + B_IMG * H * W                  # logits once + gradient once + edge bytes (52.5 MB)


def main_cuda(args, rank, world, local_rank):
    from boxinstseg_b200 import _lib as L
    from boxinstseg_b200.models.dense_heads import CondInstMaskHead
    from boxinstseg_b200.ops.boxinst import boxinst_loss_plan, boxinst_mask_loss, boxinst_targets
    lib = L.lib()                                # fail loudly if the CUDA extension is missing
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    pinned_cpus = pin_to_numa_node(local_rank, world)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL announces its version on stdout at communicator creation; the contract is ONE JSON line there
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    sampler = ClockSampler(local_rank)
    sampler.start()                              # NVML initialisation happens long before the timed regions

    case = synthetic_case(1234 + rank)
    img = case['img'].to(dev)
    boxes = [b.to(dev) for b in case['gt_bboxes']]
    gt_inds = case['gt_inds'].to(dev)
    gt_inds32 = gt_inds.to(torch.int32)       # instance -> GT indices are part of the (precomputed) targets
    it = torch.tensor([10000.0], device=dev)
    targets = boxinst_targets(img, case['metas'], boxes)
    # the work plan of the single-pass kernel is index work on the targets (item list + weight total): built with them
    plan = None if os.environ.get('BXS_ONEPASS_CTA') == '1' else boxinst_loss_plan(targets, gt_inds32, H, W, 2)
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    logit_sets = [case['logits'].to(dev)] + [torch.randn(N_INST, 1, H, W, device=dev, generator=gen) * 2
                                             for _ in range(ROTATE - 1)]
    logit_sets = [t.requires_grad_(True) for t in logit_sets]
    ones = torch.ones((), device=dev)
    out_ring = [None] * ROTATE        # keeps the last R outputs alive so every step writes a fresh 26 MB gradient

    def step(i):
        x = logit_sets[i % ROTATE]
        prj, pair = boxinst_mask_loss(x, targets, gt_inds32, it, plan=plan)
        torch.autograd.backward([prj, pair], [ones, ones])
        out_ring[i % ROTATE], x.grad = (prj.detach(), pair.detach(), x.grad), None
        return prj, pair

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / steps

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    ms_eager = timed(step, args.steps)
    last = out_ring[(args.steps - 1) % ROTATE]      # (loss_prj, loss_pairwise, d/d mask logits) of the last timed step

    # ---- the same step (public autograd op, forward + backward) captured once per rotating input set
    #      into CUDA graphs: removes the ~0.2 ms/step of Python/autograd launch overhead ----
    graphs, mode, steps_timed, ms_step_spread = [], 'cuda_graph', args.steps, None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(ROTATE):
                logit_sets[i].grad = None
                step(i)
                logit_sets[i].grad = None
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        # one graph = ROTATE consecutive steps over the rotating input sets (a training loop captures whole
        # iterations the same way); the graph launch latency is amortised over its steps
        def capture(n_steps, first):
            gr = torch.cuda.CUDAGraph()
            for x in logit_sets:
                x.grad = None
            with torch.cuda.graph(gr):
                for i in range(first, first + n_steps):
                    x = logit_sets[i % ROTATE]
                    prj, pair = boxinst_mask_loss(x, targets, gt_inds32, it, plan=plan)
                    torch.autograd.backward([prj, pair], [ones, ones])
                    graphs.append((prj, pair, x.grad))
            return gr
        # EXACTLY args.steps steps per timed region: full graphs of ROTATE steps + one tail graph of steps % ROTATE
        full, tail = args.steps // ROTATE, args.steps % ROTATE
        g = capture(ROTATE, 0)
        g_tail = capture(tail, 0) if tail else None
        for i in range(max(warm // ROTATE, 1)):
            g.replay()

        def region(_i):
            for _ in range(full):
                g.replay()
            if g_tail is not None:
                g_tail.replay()
        # a region of K steps is ~25 us x K: one hiccup would move the headline, so the region is timed REGIONS times
        # (each bracketed by barrier + synchronize, device events) and the median region is reported
        REGIONS = 15
        samples = sorted(timed(region, 1) for _ in range(REGIONS))
        ms_step = samples[REGIONS // 2] / args.steps
        last = graphs[-1]                       # the last step of the last graph a region replays
        ms_step_spread = (samples[0] / args.steps, samples[-1] / args.steps)
        steps_timed = args.steps
        mode = f'cuda_graph ({ROTATE} steps per graph' + (f' + one tail graph of {tail}' if tail else '') + \
            f'); median of {REGIONS} timed regions of {args.steps} steps'
    except Exception as e:  # noqa: BLE001
        mode = f'eager (graph capture failed: {type(e).__name__})'
        ms_step = ms_eager

    # ---- per-call timing through the C ABI (same rotation): the single-pass schedule the step uses, and the
    #      two-call kernels (forward-only / fallback path) for comparison ----
    inst_gt = gt_inds32
    ws = torch.empty(lib.bxs_boxinst_loss_workspace_bytes(N_INST, H, W), dtype=torch.uint8, device=dev)
    ws1 = torch.empty(lib.bxs_boxinst_loss_fused_workspace_bytes(N_INST, H, W), dtype=torch.uint8, device=dev)
    sched = torch.zeros(int(lib.bxs_boxinst_loss_fused_sched_bytes()), dtype=torch.uint8, device=dev)
    out4 = torch.empty(4, device=dev)
    g2 = torch.ones(2, device=dev)
    raw_x = [t.detach() for t in logit_sets]
    raw_g = [torch.empty_like(raw_x[0]) for _ in range(ROTATE)]
    st = L.stream()

    def raw_fwd(i, s_=None):
        L.check(lib.bxs_boxinst_loss_forward(L.ptr(raw_x[i % ROTATE]), L.ptr(targets.edge_bits), L.ptr(targets.rects),
                                             L.ptr(inst_gt), L.ptr(targets.gt_img), L.ptr(it), 10000.0, L.ptr(ws),
                                             L.ptr(out4), N_INST, H, W, 2, s_ or st), 'fwd')

    def raw_bwd(i, s_=None):
        L.check(lib.bxs_boxinst_loss_backward(L.ptr(raw_x[i % ROTATE]), L.ptr(targets.edge_bits), L.ptr(targets.rects),
                                              L.ptr(inst_gt), L.ptr(targets.gt_img), L.ptr(ws), L.ptr(g2),
                                              L.ptr(raw_g[i % ROTATE]), N_INST, H, W, 2, s_ or st), 'bwd')

    def raw_one_fwd(i, s_=None):
        if plan is not None:
            L.check(lib.bxs_boxinst_loss_fused_forward_planned(L.ptr(raw_x[i % ROTATE]), L.ptr(targets.edge_bits), L.ptr(plan),
                                                               L.ptr(it), 10000.0, L.ptr(ws1), L.ptr(sched), L.ptr(out4),
                                                               L.ptr(raw_g[i % ROTATE]), N_INST, H, W, 2, s_ or st), 'fused fwd')
            return
        L.check(lib.bxs_boxinst_loss_fused_forward(L.ptr(raw_x[i % ROTATE]), L.ptr(targets.edge_bits), L.ptr(targets.rects),
                                                   L.ptr(inst_gt), L.ptr(targets.gt_img), L.ptr(it), 10000.0, L.ptr(ws1),
                                                   L.ptr(sched), L.ptr(out4), L.ptr(raw_g[i % ROTATE]), N_INST, H, W, 2, s_ or st),
                'fused fwd')

    def raw_one_bwd(i, s_=None):
        L.check(lib.bxs_boxinst_loss_fused_backward(L.ptr(ws1), L.ptr(g2[0:1]), L.ptr(g2[1:2]), L.ptr(raw_g[i % ROTATE]),
                                                    N_INST, H, W, s_ or st), 'fused bwd')
    def graph_us(fn):
        """device time per call: ROTATE calls captured in one CUDA graph (no host launch overhead), replayed"""
        for i in range(ROTATE):
            fn(i)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cur = L.stream()
            for i in range(ROTATE):
                fn(i, cur)
        g.replay()
        reps = max(args.steps // ROTATE, 1)
        return timed(lambda i: g.replay(), reps) * 1e3 / ROTATE

    us_fwd = graph_us(raw_fwd)
    us_bwd = graph_us(raw_bwd)
    us_one_fwd = graph_us(raw_one_fwd)

    def raw_one_both(i, s_=None):
        raw_one_fwd(i, s_)
        raw_one_bwd(i, s_)
    us_one_step = graph_us(raw_one_both)
    us_one_bwd = us_one_step - us_one_fwd

    # ---- e2e through the public head API with host buffers ----
    head = CondInstMaskHead(in_channels=16, in_stride=8, out_stride=4, topk_per_img=64, max_proposals=-1,
                            boxinst_enabled=True, pairwise_warmup=10000).to(dev)
    h_img = case['img'].pin_memory()
    h_logits = case['logits'].pin_memory()
    h_boxes = [b.pin_memory() for b in case['gt_bboxes']]
    # two steps in flight on two streams: the H2D of step i+1 overlaps the kernels and the D2H of step i
    # (separate copy engines, full-duplex link); every step still moves all of its inputs and results
    SLOTS = 2
    h_grad = [torch.empty_like(case['logits']).pin_memory() for _ in range(SLOTS)]
    h_loss = [torch.empty(2).pin_memory() for _ in range(SLOTS)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(SLOTS)]
    h2d = h_img.numel() * 4 + h_logits.numel() * 4 + sum(b.numel() * 4 for b in h_boxes)
    d2h = h_grad[0].numel() * 4 + 8

    def e2e_step(i):
        slot = i % SLOTS
        with torch.cuda.stream(streams[slot]):
            d_img = h_img.to(dev, non_blocking=True)
            d_logits = h_logits.to(dev, non_blocking=True).requires_grad_(True)
            d_boxes = [b.to(dev, non_blocking=True) for b in h_boxes]
            losses = head.loss(d_img, case['metas'], d_logits, gt_inds, d_boxes, None, None)
            torch.autograd.backward([losses['loss_prj'], losses['loss_pairwise']], [ones, ones])
            h_grad[slot].copy_(d_logits.grad, non_blocking=True)
            h_loss[slot].copy_(torch.stack([losses['loss_prj'].detach(), losses['loss_pairwise'].detach()]),
                               non_blocking=True)

    def timed_streams(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        cur = torch.cuda.current_stream()
        e0.record()
        for s_ in streams:
            s_.wait_stream(cur)
        for i in range(steps):
            fn(i)
        for s_ in streams:
            cur.wait_stream(s_)
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / steps

    head._iter.fill_(9999)
    for i in range(4):
        e2e_step(i)
    ms_e2e = timed_streams(e2e_step, args.steps)
    ddp = ddp_allreduce_leg(dist, dev, world, step, args.steps) if dist is not None else None
    clocks = sampler.stop()

    ms_step, ms_e2e, ms_eager, us_fwd, us_bwd, us_one_fwd, us_one_bwd, us_one_step = reduce_max_over_ranks(
        [ms_step, ms_e2e, ms_eager, us_fwd, us_bwd, us_one_fwd, us_one_bwd, us_one_step], dist, dev)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(('loss_prj', 'loss_pairwise', 'grad_mask_logits'), last)))

    peak, peak_src = measured_peak_gbs()
    achieved = ALGO_BYTES / (ms_step * 1e-3) / 1e9
    ach_f, ach_b = FWD_BYTES / (us_fwd * 1e-6) / 1e9, BWD_BYTES / (us_bwd * 1e-6) / 1e9
    cpu_ms, cores, sample = (None, None, None)
    if world == 1 and not args.no_cpu_baseline:
        cpu_ms, cores, sample = run_cpu(2, 1)
    line = {
        'metric': METRIC, 'value': ms_step / (B_IMG * world),   # whole job: step time / images of all ranks
        'unit': 'ms/img', 'n_gpus': world,
        'steps': steps_timed, 'warmup': warm, 'ms_per_step': ms_step, 'higher_is_better': False, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD,
                   'l2': f'inputs rotate over {ROTATE} logit/grad sets ({ROTATE * 52} MB > 126 MB L2)',
                   'launch': mode, 'eager_ms_per_step': ms_eager,
                   'e2e_mode': 'CondInstMaskHead.loss + backward from pinned host buffers, 2 steps in flight on 2 streams',
                   'parallelism': f'replicas x{world} (loss is per image; no data-path collective)',
                   'aggregate_img_per_s': world * B_IMG / (ms_step * 1e-3)},
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': ncu_traffic_bytes(),
                     'traffic_source': 'profiles/r2_traffic.json (ncu --set full, dram read+write per launch, summed over the '
                                       'kernels of one step)',
                     'peak_source': peak_src,
                     'note': 'headline = the WHOLE step (wq_main + wq_finalize + onepass_backward kernels, CUDA-graph replay '
                             'through the public autograd op) against the 85.2 MB/step ALGORITHMIC figure of SURVEY 8d '
                             '(logits read in fwd and in bwd + gradient written + similarity read twice).  The single-pass '
                             'schedule moves 52.5 MB (logits once, gradient once, edge bytes): see kernels.*; the dominant '
                             'kernel is wq_main_kernel (its share of the step: profiles/r2_launches_bench.csv)',
                     'kernels': {'single_pass_forward(wq_main+wq_finalize)': {
                                     'us': us_one_fwd, 'moved_mb': ONEPASS_BYTES / 1e6,
                                     'achieved_moved': ONEPASS_BYTES / (us_one_fwd * 1e-6) / 1e9,
                                     'frac_moved': ONEPASS_BYTES / (us_one_fwd * 1e-6) / 1e9 / peak,
                                     'achieved_algorithmic': ALGO_BYTES / (us_one_fwd * 1e-6) / 1e9,
                                     'frac_algorithmic': ALGO_BYTES / (us_one_fwd * 1e-6) / 1e9 / peak},
                                 'single_pass_backward(onepass_backward, in place)': {'us': us_one_bwd},
                                 'single_pass_step_c_abi': {'us': us_one_step, 'achieved_algorithmic': ALGO_BYTES / (us_one_step * 1e-6) / 1e9,
                                                            'frac_algorithmic': ALGO_BYTES / (us_one_step * 1e-6) / 1e9 / peak},
                                 'two_call_forward(fwd_fused+finalize)': {'us': us_fwd, 'algo_mb': FWD_BYTES / 1e6, 'achieved': ach_f,
                                                                          'frac': ach_f / peak},
                                 'two_call_backward(bwd_rows)': {'us': us_bwd, 'algo_mb': BWD_BYTES / 1e6, 'achieved': ach_b,
                                                                 'frac': ach_b / peak}},
                     'timing': 'per-call numbers: 8 rotating calls captured in one CUDA graph, CUDA events around replays'},
        'e2e': {'value': ms_e2e / (B_IMG * world), 'unit': 'ms/img', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
        'gpu_launches': 3 * steps_timed,        # wq_main + wq_finalize + onepass_backward kernels per step
        'clocks': clocks,
    }
    if ddp is not None:
        line['ddp_allreduce'] = ddp
    if pinned_cpus:
        line['config']['cpu_affinity_rank0'] = pinned_cpus
    # the B200 arm's own results on logit set 0 (the set the gpu_reference leg uses)
    x0 = logit_sets[0].detach().clone().requires_grad_(True)
    p0, q0 = boxinst_mask_loss(x0, targets, gt_inds32, it, plan=plan)
    (g0,) = torch.autograd.grad(p0 + q0, x0)
    line['losses'] = {'loss_prj': float(p0.detach()), 'loss_pairwise': float(q0.detach()), 'logit_set': 0}
    if ms_step_spread is not None:
        line['config']['region_ms_per_step_min_max'] = list(ms_step_spread)
    if cpu_ms is not None:
        line['cpu_baseline'] = {'value': cpu_ms, 'unit': 'ms/img', 'cores': f'{cores} of {os.cpu_count()}', 'kind': 'port',
                                'sample': sample}
    if world == 1 and not args.no_cpu_baseline:
        try:
            ref_gpu = run_gpu_reference(case, dev, ours_grad=g0)
        except Exception as e:  # noqa: BLE001  (baseline only: never let it take the bench line down)
            ref_gpu = {'unavailable': f'{type(e).__name__}: {e}'[:200]}
        if ref_gpu is not None:
            line['gpu_reference'] = ref_gpu
            if 'loss_prj' in ref_gpu and 'losses' in line:
                rp, rq = ref_gpu['loss_prj'], ref_gpu['loss_pairwise']
                line['parity_vs_gpu_reference'] = {
                    'rel_err_loss_prj': abs(line['losses']['loss_prj'] - rp) / abs(rp),
                    'rel_err_loss_pairwise': abs(line['losses']['loss_pairwise'] - rq) / abs(rq),
                    'rel_err_grad': ref_gpu.pop('_grad_rel_err', None),
                    'what': 'B200 arm vs the restated reference loss around the reference CUDA pairwise op, same logits (set 0), '
                            'same targets; bar: 1e-3 (BASELINE.json north_star)'}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# configs C / D / E (BASELINE.json configs[2..4]): the mask-loss steps of DiscoBox, BoxLevelset, Box2Mask
# ------------------------------------------------------------------------------------------
def main_config(args, rank, world, local_rank):
    import bench_configs as bc
    from boxinstseg_b200 import _lib as L
    L.lib()                                      # fail loudly if the CUDA extension is missing
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    sampler = ClockSampler(local_rank)
    sampler.start()
    cfg = args.config
    # rotate over R independent input sets so that a step never finds its inputs in the 126 MB L2
    set_mb = dict(C=110, D=30, E=75)[cfg]
    R = max(2, -(-140 // set_mb))
    built = [bc.BUILDERS[cfg](dev, 1234 + rank + 100 * r) for r in range(R)]
    steps_fn = [b[0] for b in built]
    info = built[0][1]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / steps

    warm = max(args.warmup, 3)
    for i in range(max(warm, R)):
        steps_fn[i % R]()
    steps = args.steps
    eager_last = []

    def eager_step(i):
        out = steps_fn[i % R]()
        if i == steps - 1:                        # kept without its autograd graph, which would break the capture below
            losses, grads = out
            eager_last.append(({k: v.detach() for k, v in losses.items()} if isinstance(losses, dict) else losses.detach(),
                               grads))
    ms_eager = timed(eager_step, steps)
    last = eager_last[0]               # (losses, gradients) of the last timed step
    mode, ms_step, steps_timed = 'eager', ms_eager, steps
    try:                                          # the same steps as CUDA graphs of R consecutive steps
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for r in range(R):
                steps_fn[r]()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        keep = []

        def capture(n):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for r in range(n):
                    keep.append(steps_fn[r]())
            return gr
        # EXACTLY `steps` steps in the timed region: full graphs of R steps + one tail graph of steps % R
        full, tail = steps // R, steps % R
        g = capture(R)
        g_tail = capture(tail) if tail else None

        def region(_i):
            for _ in range(full):
                g.replay()
            if g_tail is not None:
                g_tail.replay()
        g.replay()
        if g_tail is not None:
            g_tail.replay()
        ms_step = timed(region, 1) / steps
        last = keep[-1]
        mode = f'cuda_graph ({R} steps per graph' + (f' + one tail graph of {tail}' if tail else '') + ')'
    except Exception as e:  # noqa: BLE001
        mode = f'eager (graph capture failed: {type(e).__name__}: {str(e)[:80]})'
    clocks = sampler.stop()
    ms_step, ms_eager = reduce_max_over_ranks([ms_step, ms_eager], dist, dev)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        losses, grads = last
        arrays = dict(losses) if isinstance(losses, dict) else {'loss': losses}
        arrays.update((f'grad_{i}', t) for i, t in enumerate(grads))
        dump_outputs(args.dump_outputs, arrays)
    peak, peak_src = measured_peak_gbs()
    achieved = info['algo_bytes'] / (ms_step * 1e-3) / 1e9
    imgs = info['images']
    line = {
        'metric': METRIC, 'value': ms_step / (imgs * world), 'unit': 'ms/img', 'n_gpus': world, 'steps': steps_timed,
        'warmup': warm, 'ms_per_step': ms_step, 'higher_is_better': False, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': info['workload'], 'gradients': info['grads'],
                   'l2': f'inputs rotate over {R} independent sets (> 126 MB L2 in total)',
                   'launch': mode, 'eager_ms_per_step': ms_eager,
                   'parallelism': f'replicas x{world} (loss is per image; no data-path collective)'},
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': None, 'peak_source': peak_src, 'algorithmic_bytes_per_step': info['algo_bytes'],
                     'algorithmic_bytes': info['algo'],
                     'note': 'whole step against the HBM lower bound of SURVEY 8d; the tree-filter / mean-field / LCM kernels are '
                             'dependency-latency bound (levels / iterations), see profiles/r2_notes.md for the per-kernel ncu summaries'},
        'e2e': {'value': ms_eager / (imgs * world), 'unit': 'ms/img', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'note': 'eager launch through the public head API (Python + autograd overhead included); inputs are feature maps '
                        'produced on the device by the network, so there is no host copy on this path'},
        'gpu_launches': None,
        'clocks': clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        try:
            ref = bc.REFERENCE[cfg](info)
            if ref is not None:
                for _ in range(2):
                    ref()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                iters = 3
                for _ in range(iters):
                    rl = ref()
                e1.record()
                torch.cuda.synchronize()
                ours = steps_fn[0]()
                ours_loss = ours[0] if torch.is_tensor(ours[0]) else sum(ours[0].values())
                line['gpu_reference'] = {
                    'value': e0.elapsed_time(e1) / iters / imgs, 'unit': 'ms/img', 'iters': iters,
                    'what': "the reference's eager PyTorch path on this GPU around its own compiled tree_filter_cuda (oracle/_ref, "
                            'built by oracle/Makefile from mmdet/ops/tree_filter/src unmodified), restated in bench_configs.py',
                    'loss_reference': float(rl[0].detach()) if hasattr(rl[0], 'detach') else float(rl[0]), 'loss_b200': float(ours_loss.detach()) if hasattr(ours_loss, 'detach') else float(ours_loss)}
        except Exception as e:  # noqa: BLE001
            line['gpu_reference'] = {'unavailable': f'{type(e).__name__}: {e}'[:300]}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f'{v} is not a positive integer')
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=positive_int, default=200, help='timed steps')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--config', default='A', choices=['A', 'C', 'D', 'E'],
                    help='A (default, the headline): BoxInst; C: DiscoBox; D: BoxLevelset; E: Box2Mask (BASELINE.json configs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned (losses, gradients) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the B200 arm computed; --impl reference has no such outputs')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        main_reference(args, rank, world)
    elif args.config != 'A':
        main_config(args, rank, world, local_rank)
    else:
        main_cuda(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
