#!/usr/bin/env python
"""bench.py - poses/sec at 20 diffusion steps (BASELINE.json metric) on synthetic protein-ligand graphs.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W     # the CPU oracle (reference restatement) on the host cores
    python bench.py --steps K --dump-outputs DIR              # also write the last timed step's poses to DIR/ligand_pos.npy

A "step" is one reverse-diffusion step of the hot path for one batch: set_time -> score-model forward (graph build,
embeddings, 6 tensor-product conv layers, tr/rot/tor heads) -> pose update, for POSES poses of one synthetic complex
(1500 residues / 40 ligand atoms; 40 poses = BASELINE config 3, the full sampling loop) per GPU; consecutive steps walk
the 20-step 'expbeta' schedule (t: 1 -> 0.05), so K=20 is exactly one sampling run.  value = total poses / (20 * mean step
time), steps launched as replays of the sampler's CUDA graph (diffdock_b200.sampling.GraphedSteps), inputs resident.
The JSON line also carries: the end-to-end number through diffdock_b200.sampling.sampling() with host inputs (median of 5
calls after one warm call), the same measurement for BASELINE config 2 (batch 32) and for the sh_lmax=1 model (CFG-L1), the
roofline of the fused tensor-product conv kernel on ALGORITHMIC work (SURVEY 8(d) bytes and fp32 FLOPs per edge) next to
the issued tensor-pipe rate, measured live with CUDA events, the parity of the timed workload against the CPU oracle, and
the CPU baseline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from functools import partial

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from diffdock_b200.synthetic import default_model_args, make_pose_list   # noqa: E402
from diffdock_b200.hetero import collate                                  # noqa: E402

TEMPS = dict(temp_sampling=[1.170050527854316, 2.06391612594481, 7.044261621607846],      # default_inference_args.yaml
             temp_psi=[0.727287304570729, 0.9022615585677628, 0.5946212391366862],
             temp_sigma_data=[0.9299802531572672, 0.7464326999906034, 0.6943254174849822])
N_SCHED = 20


def model_kwargs(a):
    return dict(sigma_embed_dim=a.sigma_embed_dim, sh_lmax=a.sh_lmax, ns=a.ns, nv=a.nv, num_conv_layers=a.num_conv_layers,
                lig_max_radius=a.max_radius, rec_max_radius=a.rec_max_radius, cross_max_distance=a.cross_max_distance,
                center_max_distance=a.center_max_distance, distance_embed_dim=a.distance_embed_dim,
                cross_distance_embed_dim=a.cross_distance_embed_dim, dynamic_max_cross=a.dynamic_max_cross,
                lm_embedding_type='precomputed', embed_also_ligand=True, num_prot_emb_layers=a.num_prot_emb_layers)


def randomise_bn(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in model.modules():
            if hasattr(m, 'running_var') and hasattr(m, 'running_mean'):
                m.running_mean.copy_(0.1 * torch.randn(m.running_mean.shape, generator=g))
                m.running_var.copy_(0.5 + torch.rand(m.running_var.shape, generator=g))


def host_threads():
    """Threads for the CPU oracle: every host core up to 32 (beyond that the oracle's many small PyTorch ops lose time
    to oversubscription: 134 s/pose-step with 128 threads vs 17 s with 8 on this workload); override DDB200_CPU_THREADS."""
    return int(os.environ.get('DDB200_CPU_THREADS', min(os.cpu_count() or 1, 32)))


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p)), 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self._halt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.rows)}


# ----------------------------------------------------------------------------------------------------- CPU oracle arm
def oracle_step_fn(args, n_res, n_atoms, seed, want_scores=False):
    """One bounded sample of the workload on the host: ONE pose of the same synthetic complex - score-model forward
    (oracle restatement of the reference's e3nn/torch_scatter op sequence) + the SDE perturbation WITH its noise terms +
    pose update, at schedule point t_idx (utils/sampling.py:96-191).  The pose returns to the prior at t_idx == 0."""
    from oracle.cg_model import CGModel
    from oracle.diffusion import modify_conformer_batch, set_time, t_to_sigma
    from oracle.layers import get_timestep_embedding
    from diffdock_b200.diffusion_utils import get_t_schedule
    from diffdock_b200.sampling import step_coefficients
    torch.manual_seed(0)
    model = CGModel(partial(t_to_sigma, args=args), 'cpu',
                    get_timestep_embedding('sinusoidal', args.sigma_embed_dim, args.embedding_scale), **model_kwargs(args)).eval()
    randomise_bn(model, 1)
    pose = make_pose_list(1, n_res=n_res, n_atoms=n_atoms, seed=seed, tr_sigma_max=args.tr_sigma_max)
    g = collate(pose)
    pos0 = g['ligand'].pos.clone()
    sched = get_t_schedule('expbeta', N_SCHED)
    mask_rotate = torch.from_numpy(pose[0]['ligand'].mask_rotate[0])
    gen = torch.Generator().manual_seed(7)

    def step(t_idx, pos=None):
        t_idx = t_idx % N_SCHED
        if pos is not None:
            g['ligand'].pos = pos.clone()
        elif t_idx == 0:
            g['ligand'].pos = pos0.clone()
        t = sched[t_idx]
        set_time(g, t, t, t, 1, 'cpu')
        with torch.no_grad():
            tr, rot, tor, _ = model(g)
            c = step_coefficients(t_idx, N_SCHED, sched, sched, sched, partial(t_to_sigma, args=args), args, False,
                                  **TEMPS)
            last = t_idx == N_SCHED - 1
            z = (lambda shape: torch.zeros(shape)) if last else (lambda shape: torch.randn(shape, generator=gen))
            g['ligand'].pos = modify_conformer_batch(g['ligand'].pos, g, c[0] * tr + c[1] * z(tr.shape),
                                                     c[2] * rot + c[3] * z(rot.shape), c[4] * tor + c[5] * z(tor.shape),
                                                     mask_rotate)
        return (tr, rot, tor) if want_scores else None
    step.pos0, step.model, step.graph = pos0, model, g
    return step


# schedule points the CPU arm times when the whole 20-step trajectory does not fit its budget: both ends and three interior
# points; the per-step cost falls monotonically with t (the cross graph shrinks with 3 sigma_tr + 20 A), so the trapezoid
# rule over these points estimates the trajectory total without the high-noise bias of "the first few steps".
STRATA = (0, 5, 10, 15, 19)


def trajectory_seconds(costs):
    """costs: {t_idx: seconds}.  Sum over t_idx = 0..19 of the piecewise-linear interpolant through the measured points."""
    pts = sorted(costs)
    if len(pts) == N_SCHED:
        return float(sum(costs.values()))
    if len(pts) == 1:
        return float(N_SCHED * costs[pts[0]])
    xs = np.arange(N_SCHED)
    return float(np.interp(xs, pts, [costs[p] for p in pts]).sum())


def run_reference(cli):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = host_threads()
    torch.set_num_threads(cores)
    args = default_model_args(sh_lmax=cli.sh_lmax)
    step = oracle_step_fn(args, cli.n_res, cli.n_atoms, seed=100)
    budget = float(os.environ.get('DDB200_REF_BUDGET_S', '480'))
    t0 = time.perf_counter()
    step(N_SCHED - 1)             # warm-up at the cheapest schedule point doubles as the cost probe
    probe = time.perf_counter() - t0
    warm = 1
    # cost at t_idx 0 is ~3.5-4x the probe (measured: 46 s vs 11 s); the trajectory averages ~1.6x (349 s / 20 / 10.9 s).
    # With the default budget the whole 20-point schedule of one pose is timed (~6.5 min on the 32 threads of the GPU box,
    # steps = K as requested); a slower host falls back to the stratified points.
    if cli.steps >= N_SCHED and probe * (1.65 * N_SCHED + max(cli.warmup - 1, 0)) <= budget:
        points = list(range(N_SCHED))
        for _ in range(max(cli.warmup - 1, 0)):
            step(N_SCHED - 1)
            warm += 1
    else:
        k = min(len(STRATA), cli.steps)
        points = list(STRATA) if k >= len(STRATA) else ([0, N_SCHED - 1] if k >= 2 else [N_SCHED // 2])
    costs = {}
    for t_idx in points:          # in schedule order (the cost of a step is set by its cut-off 3 sigma_tr(t) + 20 A)
        t0 = time.perf_counter()
        step(t_idx)
        costs[t_idx] = time.perf_counter() - t0
    total = trajectory_seconds(costs)
    steps = len(points)
    value = 1.0 / total           # one pose through the full 20-step schedule
    sample = (f"1 pose of the {cli.n_res}-residue/{cli.n_atoms}-atom complex per step (forward + noise + pose update); "
              f"schedule points {points} timed ({', '.join(f'{costs[p]:.1f}' for p in points)} s), trajectory total "
              f"{'summed' if steps == N_SCHED else 'by trapezoid interpolation over the 20 points'} = {total:.0f} s; "
              f"budget {budget:.0f} s")
    line = {"impl": "reference", "metric": "poses/sec at 20 diffusion steps", "value": value, "unit": "poses/s",
            "n_gpus": cli.gpus, "steps": steps, "warmup": warm, "ms_per_step": total / N_SCHED * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cli, cli.poses),      # same workload as the CUDA arm; the bounded sample is below
            "schedule_points": points, "seconds_per_point": {str(k): v for k, v in costs.items()},
            "cpu_baseline": {"value": value, "unit": "poses/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(cli, poses):
    cfgname = "BASELINE config 3 (full 20-step sampling loop, 40 poses/complex)" if poses == 40 else \
        ("BASELINE config 2 (batch 32)" if poses == 32 else f"{poses} poses")
    return {"workload": f"DiffDock-L-shaped score model (ns=48,nv=10,sh_lmax={cli.sh_lmax},6 conv layers) reverse-diffusion "
                        f"step, synthetic complex {cli.n_res} residues / {cli.n_atoms} ligand atoms, {poses} poses per GPU "
                        f"[{cfgname}], 20-step expbeta schedule",
            "poses_per_gpu": poses, "n_res": cli.n_res, "n_atoms": cli.n_atoms, "sh_lmax": cli.sh_lmax,
            "l2": "per-step working set (edge embeddings ~0.3 GB per receptor edge group and layer, operand images, "
                  "node tensors) exceeds the 126 MB L2; no explicit flush",
            "warmup_executed": cli.warmup if getattr(cli, 'short_warmup', False) else max(cli.warmup, N_SCHED),
            "launch": "one CUDA-graph replay per step (diffdock_b200.sampling.GraphedSteps); the eager op-by-op step is "
                      "reported as eager_ms_per_step",
            "parallelism": f"poses sharded over {cli.gpus} GPU(s), no data-path collective"}


# ----------------------------------------------------------------------------------------------------- CUDA arm
def tpconv_stream_roofline(dev, n_edges=200000):
    """BASELINE metric 'fused TP-conv HBM GB/s vs peak': the streaming tensor-product conv kernel (per-edge weights read
    from HBM, the un-fused formulation of SURVEY 8(d)) timed alone with CUDA events on 200k receptor-like edges of the
    full-width 156->156 layer (5.7 GB of weights >> L2), median of 5 launches."""
    from diffdock_b200 import ops
    from diffdock_b200.tensor_layers import get_irrep_seq
    from diffdock_b200.tp_table import build_table
    seq = get_irrep_seq(48, 10, False, False)
    t = build_table(seq[3], '1x0e+1x1o+1x2e', seq[3], 'fctp')
    h = ops.TpHandle(t)
    g = torch.Generator(device=dev).manual_seed(0)
    n_nodes = 48000
    x = torch.randn(n_nodes, t.d_in, device=dev, generator=g)
    dst = (torch.arange(n_edges, device=dev) // 24).clamp_max(n_nodes - 1).int()
    src = torch.randint(0, n_nodes, (n_edges,), device=dev, generator=g).int()
    vec = torch.randn(n_edges, 3, device=dev, generator=g)
    w = torch.randn(n_edges, t.weight_numel_padded, device=dev, generator=g)
    out, cnt = torch.zeros(n_nodes, t.d_out, device=dev), torch.zeros(n_nodes, device=dev)
    was = ops.PROFILE.enabled
    ops.PROFILE.enabled = False
    times = []
    for i in range(8):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.tpconv_accumulate(h, x, src, dst, vec, w, out, cnt)
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            times.append(e0.elapsed_time(e1))
    ops.PROFILE.enabled = was
    ms = sorted(times)[len(times) // 2]
    nbytes = n_edges * (4 * t.weight_numel + 16) + 4 * (n_nodes + 1) + 4 * n_nodes * t.d_in + 4 * n_nodes * t.d_out
    return {"bound": "hbm", "kernel": "tpconv_accumulate_kernel", "achieved": nbytes / ms / 1e6, "unit": "GB/s",
            "edges": n_edges, "bytes_per_launch": nbytes, "ms_per_launch": ms, "traffic": None,
            "how": "standalone launches, CUDA events, weights (5.7 GB) larger than L2; the model itself runs the fully "
                   "fused kernel (see 'roofline')"}


def _ncu_traffic():
    """DRAM bytes per launch of the fused kernel from the committed ncu capture of this round (None if absent): the run
    itself cannot read dram__bytes without a profiler attached."""
    for name in ('r02m_fused_traffic.json', 'r02_fused_traffic.json'):        # newest capture first
        p = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(p):
            try:
                return json.load(open(p))
            except Exception:
                return None
    return None


class Workload:
    """Model + one batch of POSES poses of the synthetic complex on this rank's GPU, with the three ways of running it:
    graph replays (the timed region), eager steps (per-launch events for the roofline), sampling() from host inputs (e2e)."""

    def __init__(self, cli, n_poses, sh_lmax, dev, rank, seed=None):
        from diffdock_b200.cg_model import CGModel
        from diffdock_b200.diffusion_utils import get_t_schedule, get_timestep_embedding, t_to_sigma
        from diffdock_b200.sampling import GraphedSteps, step_coefficients
        self.cli, self.n_poses, self.dev = cli, n_poses, dev
        self.args = args = default_model_args(sh_lmax=sh_lmax)
        self.t2s = partial(t_to_sigma, args=args)
        torch.manual_seed(0)
        model = CGModel(self.t2s, dev, get_timestep_embedding('sinusoidal', args.sigma_embed_dim, args.embedding_scale),
                        **model_kwargs(args)).eval()
        randomise_bn(model, 1)
        self.model = model.to(dev)
        self.poses = make_pose_list(n_poses, n_res=cli.n_res, n_atoms=cli.n_atoms, seed=(100 + rank) if seed is None else seed,
                                    tr_sigma_max=args.tr_sigma_max)
        self.sched = get_t_schedule('expbeta', N_SCHED)
        lig0 = self.poses[0]['ligand']
        self.mask_u8 = torch.from_numpy(lig0.mask_rotate[0].astype(np.uint8)).to(dev)
        rb = self.poses[0]['ligand', 'ligand'].edge_index.T[lig0.edge_mask]
        self.bu, self.bv = rb[:, 0].int().contiguous().to(dev), rb[:, 1].int().contiguous().to(dev)
        from diffdock_b200.hetero import collate_shared_receptor
        self.g = collate_shared_receptor(self.poses, dev)       # what sampling() does with N poses of one complex
        self.pos0 = self.g['ligand'].pos.clone()
        self.coef_rows, self.t_rows = [], []
        for t_idx in range(N_SCHED):
            c = step_coefficients(t_idx, N_SCHED, self.sched, self.sched, self.sched, self.t2s, args, False, **TEMPS)
            if t_idx == N_SCHED - 1:
                c[1] = c[3] = c[5] = 0.0
            self.coef_rows.append(c)
            self.t_rows.append([float(self.sched[t_idx])] * 3)
        self.graphed = None
        if model.sync_free_capable() and os.environ.get('DDB200_CUDA_GRAPH', '1') != '0':
            self.graphed = GraphedSteps(self.model, self.g, n_poses, self.coef_rows, self.t_rows, self.bu, self.bv, self.mask_u8,
                                        True, dev, draw_noise=True, philox=(1234 + rank, torch.arange(n_poses, device=dev)))
            self.pos0 = self.graphed.pos.clone()
        self.gen = torch.Generator(device=dev).manual_seed(1234 + rank)

    def graph_step(self, i):
        t_idx = i % N_SCHED
        if t_idx == 0:            # a fresh sampling run starts from the prior again
            self.graphed.pos.copy_(self.pos0)
            self.graphed.step.zero_()
        self.graphed.graph.replay()

    def eager_step(self, i):
        from diffdock_b200 import ops
        from diffdock_b200.diffusion_utils import set_time
        g, dev, n = self.g, self.dev, self.n_poses
        t_idx = i % N_SCHED
        if t_idx == 0:
            g['ligand'].pos = self.pos0.clone()
        t = self.sched[t_idx]
        set_time(g, None, t, t, t, n, False, dev)
        g._uniform_t = True                 # like the sampler: one diffusion time for the whole batch
        tr, rot, tor = self.model(g)[:3]
        last = t_idx == N_SCHED - 1
        z = (lambda shape: None) if last else (lambda shape: torch.randn(shape, device=dev, generator=self.gen))
        g['ligand'].pos = ops.pose_update(g['ligand'].pos, n, self.bu, self.bv, self.mask_u8, tr, rot, tor,
                                          self.coef_rows[t_idx], z((n, 3)), z((n, 3)), z(tuple(tor.shape)))

    def step(self, i):
        (self.graph_step if self.graphed is not None else self.eager_step)(i)

    def e2e(self, host_list, repeats=5):
        """sampling() from pinned host inputs to host outputs: median wall time of `repeats` calls after one warm call."""
        from diffdock_b200.sampling import sampling
        times, final = [], None
        for r in range(repeats + 1):
            inp = [p.clone() for p in host_list]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out, _ = sampling(inp, self.model, N_SCHED, self.sched, self.sched, self.sched, self.dev, self.t2s, self.args,
                              batch_size=self.n_poses, no_final_step_noise=True, **TEMPS)
            final = torch.stack([d['ligand'].pos for d in out]).cpu()      # D2H of the result inside the timed region
            torch.cuda.synchronize()
            if r > 0:
                times.append(time.perf_counter() - t0)
        return sorted(times)[len(times) // 2], times, final


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Write each array as DIR/<name>.npy, DUMP_LIMIT_BYTES in all.  An array over its share keeps a fixed, seeded sample of
    its rows, so the same arguments always select the same rows and two builds stay comparable entry by entry."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays)
    for name, a in arrays.items():
        if a.nbytes > share:
            keep = share // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(dirname, name + '.npy'), a)


def timed_steps(w, steps, warmup_steps, sync_all):
    for i in range(warmup_steps):
        w.step(i)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        w.step(warmup_steps + i)
    e1.record()
    sync_all()
    return e0.elapsed_time(e1) / steps


def run_cuda(cli):
    import torch.distributed as dist
    from diffdock_b200 import ops, _lib
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    _lib.lib()          # the library build() made; the benchmark compiles nothing
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
        dist.barrier()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ops.PROFILE.reset(enabled=False)
    w = Workload(cli, cli.poses, cli.sh_lmax, dev, rank)
    launches_per_step = None
    # Warm-up: the W requested steps, extended to one full pass over the 20-point schedule (every point of the schedule
    # has its own neighbour-list sizes; the graph replays have static shapes, the eager path grows the allocator).
    n_warm = cli.warmup if cli.short_warmup else max(cli.warmup, N_SCHED)
    sampler = ClockSampler(local) if rank == 0 else None
    for i in range(n_warm):
        w.step(i + cli.warmup - n_warm)
    sync_all()
    if sampler:
        sampler.start()
    ops.PROFILE.reset(enabled=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(cli.steps):
        w.step(cli.warmup + i)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1) / cli.steps
    clocks = sampler.stop() if sampler else None
    if cli.dump_outputs and rank == 0:
        # the ligand coordinates after the last timed step, per pose: what the sampler hands back to its caller
        pos = w.g['ligand'].pos.detach().float().view(w.n_poses, -1, 3).cpu().numpy()
        dump_outputs(cli.dump_outputs, {'ligand_pos': pos})
    ms_max = max_over_ranks(ms)
    value = world * cli.poses / (N_SCHED * ms_max * 1e-3)

    # Per-kernel durations: K EAGER steps with a CUDA-event pair (launching stream) around every tensor-product conv launch,
    # kept out of the timed region; the same kernels as the graph replays, launched one by one.
    for i in range(3):
        w.eager_step(i)
    torch.cuda.synchronize()
    ops.PROFILE.reset(enabled=False)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for i in range(cli.steps):
        w.eager_step(cli.warmup + i)
    r1.record()
    torch.cuda.synchronize()
    eager_ms = r0.elapsed_time(r1) / cli.steps
    launches_per_step = ops.PROFILE.all_launches / cli.steps
    ops.PROFILE.reset(enabled=True)
    for i in range(cli.steps):
        w.eager_step(cli.warmup + i)
    prof = ops.PROFILE.summary()
    ops.PROFILE.reset(enabled=False)

    if cli.no_e2e:
        if rank == 0:
            print(json.dumps({"profiling_run": True, "ms_per_step": ms_max, "value": value, "eager_ms_per_step": eager_ms,
                              "tpconv": prof}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end to end through the public API with host inputs ---------------------------------------------------
    host_list = [p.clone() for p in w.poses]
    for p in host_list:
        p._apply(lambda t: t.pin_memory() if t.is_floating_point() or t.dtype in (torch.int64, torch.bool) else t)
    h2d_unique = sum(t.numel() * t.element_size() for st in list(host_list[0]._nodes.values()) + list(host_list[0]._edges.values())
                     for t in st.__dict__.values() if torch.is_tensor(t))
    lig_bytes = sum(t.numel() * t.element_size() for k, st in list(host_list[0]._nodes.items()) + list(host_list[0]._edges.items())
                    if 'receptor' not in k for t in st.__dict__.values() if torch.is_tensor(t))
    h2d = h2d_unique + (cli.poses - 1) * lig_bytes          # one receptor copy + every pose's ligand (shared-receptor collate)
    sync_all()
    e2e_s, e2e_all, final = w.e2e(host_list)
    e2e_max = max_over_ranks(e2e_s)
    if world > 1:       # final pose gather over NCCL
        gathered = [torch.empty_like(final, device=dev) for _ in range(world)]
        dist.all_gather(gathered, final.to(dev))
    e2e_val = world * cli.poses / e2e_max
    assert torch.isfinite(final).all()

    extra = {}
    if rank == 0 and world == 1 and not cli.quick:
        # BASELINE config 2 (batch 32) and CFG-L1 (sh_lmax = 1: FasterTensorProduct weight layout) on the same complex
        for key, poses, lmax in (("config2_batch32", 32, cli.sh_lmax), ("cfg_l1_sh_lmax1", cli.poses, 1)):
            if poses == cli.poses and lmax == cli.sh_lmax:
                continue
            w2 = Workload(cli, poses, lmax, dev, rank)
            ms2 = timed_steps(w2, N_SCHED, N_SCHED, sync_all)
            hl = [p.clone() for p in w2.poses]
            s2, _, _ = w2.e2e(hl, repeats=1)
            extra[key] = {"value": poses / (N_SCHED * ms2 * 1e-3), "unit": "poses/s", "ms_per_step": ms2, "poses": poses,
                          "sh_lmax": lmax, "e2e_value": poses / s2, "graphed": w2.graphed is not None}
            del w2
            torch.cuda.empty_cache()

    stream_roof = tpconv_stream_roofline(dev) if rank == 0 else None
    if rank == 0:
        pk, pk_kind = peaks()
        roof = None
        if prof['fused_launches']:
            sec = prof['fused_ms'] * 1e-3
            issued = prof['fused_flops'] / sec / 1e12
            alg = prof['fused_alg_flops'] / sec / 1e12
            eq_gbs = prof['fused_bytes'] / sec / 1e9
            peak_tf = pk.get('bf16_tflops_sustained', pk['bf16_tflops'])
            ncu = _ncu_traffic()
            roof = {"bound": "hbm", "kernel": "fused_conv_kernel",
                    "achieved": eq_gbs, "peak": pk['hbm_gbs'], "unit": "GB/s", "frac": eq_gbs / pk['hbm_gbs'],
                    "peak_kind": pk_kind + " (HBM copy bandwidth, MEASURED_PEAKS.json)",
                    "definition": "SURVEY 8(d): ALGORITHMIC bytes of the tensor-product convolution (E (4 W + 16) + node "
                                  "tensors; the per-edge weights W counted as an HBM stream although the fused kernel keeps "
                                  "them in tensor memory) / fused-kernel time; may exceed 1 because of that",
                    "traffic": (ncu or {}).get('dram_bytes_per_launch'), "traffic_source": (ncu or {}).get('source'),
                    "tensor": {"issued_TFLOPs": issued, "issued_frac_of_bf16_peak": issued / peak_tf, "bf16_peak_TFLOPs": peak_tf,
                               "algorithmic_TFLOPs": alg,
                               "algorithmic_def": "fp32 FLOPs of the reference formulation per edge: radial MLP 2 K H + 2 H W "
                                                  "and the tensor product (SURVEY 8(d)); issued = bf16 tcgen05 FLOPs (split-bf16 "
                                                  "x3 + bias step, 16-column K steps, N tiles trimmed to 32 columns)",
                               "issued_over_algorithmic": issued / alg if alg else None},
                    "launches": prof['fused_launches'],
                    "timing": "CUDA-event pair per launch on the launching stream, over K eager steps after the timed region "
                              "(the timed region replays CUDA graphs and carries no per-launch events)",
                    "kernel_ms_per_step": prof['fused_ms'] / cli.steps, "share_of_step": prof['fused_ms'] / cli.steps / ms}
        if stream_roof:
            stream_roof.update(peak=pk['hbm_gbs'], frac=stream_roof['achieved'] / pk['hbm_gbs'], peak_kind=pk_kind)
        line = {"metric": "poses/sec at 20 diffusion steps", "value": value, "unit": "poses/s", "n_gpus": world,
                "steps": cli.steps, "warmup": cli.warmup, "ms_per_step": ms_max, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(cli, cli.poses), "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": "poses/s", "h2d_bytes_per_step": h2d // N_SCHED,
                        "d2h_bytes_per_step": int(final.numel() * 4 // N_SCHED), "seconds_per_run": e2e_max,
                        "runs_s": e2e_all, "how": "median of 5 sampling() calls after one warm call; each call collates the "
                                                  "host poses, uploads one receptor copy + all ligands, captures the step graph, "
                                                  "replays it 20 times and copies the final coordinates back"},
                "gpu_launches": int(round(launches_per_step * cli.steps)), "launches_per_step": launches_per_step,
                "graphed": w.graphed is not None, "eager_ms_per_step": eager_ms,
                "roofline": roof, "roofline_tpconv_stream": stream_roof}
        line.update(extra)
        if world == 1 and not cli.no_cpu_baseline:
            cores = host_threads()
            torch.set_num_threads(cores)
            ostep = oracle_step_fn(w.args, cli.n_res, cli.n_atoms, seed=100, want_scores=True)
            t_idx = 10          # t = 0.5: mid-schedule edge count
            t0 = time.perf_counter()
            o_tr, o_rot, o_tor = ostep(t_idx, pos=ostep.pos0)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": 1.0 / (N_SCHED * dt), "unit": "poses/s", "cores": cores, "kind": "port",
                                    "sample": f"1 pose-step (forward + noise + pose update) of the same complex at t=0.5, "
                                              f"{dt:.1f} s on {cores} host threads, oracle = reference op sequence restated; "
                                              f"the reference arm (--impl reference) integrates the whole schedule"}
            # parity of the timed workload: the product's scores for the same pose / same weights / same t
            from diffdock_b200.diffusion_utils import set_time
            g1 = collate(make_pose_list(1, n_res=cli.n_res, n_atoms=cli.n_atoms, seed=100, tr_sigma_max=w.args.tr_sigma_max)).to(dev)
            t = w.sched[t_idx]
            set_time(g1, None, t, t, t, 1, False, dev)
            p_tr, p_rot, p_tor = w.model(g1)[:3]
            rel = lambda a, b: float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
            line["parity"] = {"vs": "CPU oracle (reference op sequence), same synthetic complex, 1 pose, t=0.5, same weights",
                              "tr_rel_err": rel(p_tr, o_tr), "rot_rel_err": rel(p_rot, o_rot),
                              "tor_rel_err": rel(p_tor, o_tor) if o_tor.numel() else None, "tolerance": 1e-4}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config5(cli):
    """BASELINE config 5: 64 complexes (N_r ~ U(200,600), N_l ~ U(15,50)) x 40 poses, 20 steps, sharded over the GPUs of the box:
    whole complexes per rank (size-balanced by N_r N_l), every complex sampled as one batch through sampling() with per-(complex,
    pose, step) Philox noise, ONE all_gather of the final coordinates INSIDE the timed region.  Fixed total work: strong scaling."""
    import torch.distributed as dist
    from diffdock_b200.cg_model import CGModel
    from diffdock_b200.diffusion_utils import get_t_schedule, get_timestep_embedding, t_to_sigma
    from diffdock_b200.distributed import assign_balanced, sample_complexes_sharded
    from diffdock_b200.sampling import sampling
    from diffdock_b200.synthetic import config5_sizes
    from diffdock_b200 import _lib
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    _lib.lib()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
        dist.barrier()
    args = default_model_args(sh_lmax=cli.sh_lmax)
    t2s = partial(t_to_sigma, args=args)
    torch.manual_seed(0)
    model = CGModel(t2s, dev, get_timestep_embedding('sinusoidal', args.sigma_embed_dim, args.embedding_scale),
                    **model_kwargs(args)).eval()
    randomise_bn(model, 1)
    model = model.to(dev)
    sched = get_t_schedule('expbeta', N_SCHED)
    n_cx, n_poses = cli.complexes, cli.poses
    sizes = config5_sizes(n_cx, seed=0)
    costs = [r * a * n_poses for r, a in sizes]
    shapes = [(n_poses, a, 3) for _, a in sizes]
    mine = assign_balanced(costs, world)[rank]
    data = {i: make_pose_list(n_poses, n_res=sizes[i][0], n_atoms=sizes[i][1], seed=1000 + i, tr_sigma_max=args.tr_sigma_max,
                              share_receptor=True) for i in mine}

    trace = [] if os.environ.get('DDB200_CONFIG5_TRACE') else None

    def sample_one(i):
        keys = (i << 32) + torch.arange(n_poses, dtype=torch.int64)
        t0 = time.perf_counter()
        out, _ = sampling(data[i], model, N_SCHED, sched, sched, sched, dev, t2s, args, batch_size=n_poses,
                          no_final_step_noise=True, rng='philox', seed=2024, pose_keys=keys, **TEMPS)
        res = torch.stack([d['ligand'].pos for d in out])
        if trace is not None:
            torch.cuda.synchronize()
            trace.append((i, sizes[i][0], sizes[i][1], round(time.perf_counter() - t0, 3)))
        return res

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # warm-up: the smallest complex of this rank once (lazy initialisation, allocator), untimed; its poses are regenerated
    if mine:
        w0 = min(mine, key=lambda i: costs[i])
        sample_one(w0)
        data[w0] = make_pose_list(n_poses, n_res=sizes[w0][0], n_atoms=sizes[w0][1], seed=1000 + w0,
                                  tr_sigma_max=args.tr_sigma_max, share_receptor=True)
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    allpos = sample_complexes_sharded(n_cx, costs, shapes, sample_one, device=dev)        # includes the NCCL all_gather
    e1.record()
    sync_all()
    wall = time.perf_counter() - t0
    dev_s = e0.elapsed_time(e1) * 1e-3
    tt = torch.tensor([dev_s, wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_max, wall_max = float(tt[0]), float(tt[1])
    clocks = sampler.stop() if sampler else None
    checksum = float(sum(float(p.double().sum()) for p in allpos))
    finite = all(bool(torch.isfinite(p).all()) for p in allpos)
    if rank == 0:
        total = n_cx * n_poses
        line = {"metric": "poses/sec at 20 diffusion steps", "value": total / dev_max, "unit": "poses/s", "n_gpus": world,
                "steps": N_SCHED, "warmup": 1, "ms_per_step": dev_max / N_SCHED * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"BASELINE config 5: {n_cx} complexes (N_r~U(200,600), N_l~U(15,50)) x {n_poses} poses, "
                                       f"20 steps, whole complexes sharded over {world} GPU(s) by N_r*N_l, Philox noise per "
                                       f"(complex, pose, step), final all_gather inside the timed region",
                           "complexes": n_cx, "poses_per_complex": n_poses, "sh_lmax": cli.sh_lmax,
                           "timing": "CUDA events on the sampling stream around the whole job incl. collate / H2D / graph "
                                     "capture per complex / gather; max over ranks",
                           "parallelism": f"complex-level sharding over {world} GPU(s), one NCCL all_gather at the end"},
                "clocks": clocks, "e2e": {"value": total / wall_max, "unit": "poses/s", "seconds_per_run": wall_max,
                                          "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                                          "how": "wall clock of the same region (host inputs -> gathered coordinates)"},
                "checksum_sum_of_coordinates": checksum, "finite": finite,
                "complexes_per_rank": [len(p) for p in assign_balanced(costs, world)],
                "load_imbalance": max(sum(costs[i] for i in p) for p in assign_balanced(costs, world)) * world / sum(costs)}
        if trace is not None:
            line["trace_rank0"] = trace
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--poses', type=int, default=40)
    ap.add_argument('--n-res', dest='n_res', type=int, default=1500)
    ap.add_argument('--n-atoms', dest='n_atoms', type=int, default=40)
    ap.add_argument('--sh-lmax', dest='sh_lmax', type=int, default=2)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true', help='skip the end-to-end leg (profiling runs)')
    ap.add_argument('--workload', default='single', choices=['single', 'config5'],
                    help="'config5': 64 complexes x 40 poses sharded over the GPUs (strong scaling)")
    ap.add_argument('--complexes', type=int, default=64)
    ap.add_argument('--quick', action='store_true', help='skip the config-2 / CFG-L1 side measurements')
    ap.add_argument('--short-warmup', dest='short_warmup', action='store_true',
                    help='warm up exactly --warmup steps instead of a full schedule pass (runs under ncu)')
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR',
                    help='write the ligand coordinates after the last timed step to DIR/ligand_pos.npy (float32, '
                         '[poses, atoms, 3]); inputs are seeded, so equal arguments give equal inputs')
    cli = ap.parse_args()
    if cli.steps < 1:
        ap.error('--steps must be at least 1')
    if cli.dump_outputs and (cli.impl != 'cuda' or cli.workload != 'single'):
        ap.error('--dump-outputs applies to the single-complex CUDA workload (--impl cuda --workload single)')
    cli.warmup = max(cli.warmup, 0)
    if cli.impl == 'reference':
        run_reference(cli)
    else:
        if cli.warmup < 3:
            cli.warmup = 3
        if cli.workload == 'config5':
            run_config5(cli)
        else:
            run_cuda(cli)


if __name__ == '__main__':
    main()
