#!/usr/bin/env python
"""bench.py — MPC solves/s of the ADMM hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # own arm (B200 kernels)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm (compiled port of the path)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as DIR/*.npy

Workload ("step" = one batched solve of B instances per GPU, cold warm-start state, inputs resident
in HBM): metric row of SURVEY.md §8d — Ackermann robot 4.6 x 1.6 m, horizon T=30, N=20 static
polygon obstacles (E=4), 50 ADMM iterations with early stop disabled (iter_threshold = 0), seeded
synthetic instances (rda_planner_b200/scenarios.py).  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T, N, E, R, ITERS = 30, 20, 4, 4, 50
METRIC = 'MPC solves/sec (T=30, 20 obs, 50 ADMM iters)'
WORKLOAD = 'metric row: acker, T=30, N=20 static polygons (E=4), 50 ADMM iterations, iter_threshold=0, cold start'
DUMP_LIMIT = 64 << 20          # bytes of all files written by --dump-outputs


def dump_outputs(out, path, seed=0):
    """Write the result dict of one solve (u, s, resi_pri, resi_dual, status, iters) as <path>/<name>.npy: float fields as
    float32, integer fields as float64 (exact).  A batch above DUMP_LIMIT is cut to a fixed, seeded sample of instances
    whose indices are written as instance_index.npy, so that two builds run with the same arguments compare row for row.
    u, s, status and iters repeat bitwise from run to run; resi_pri and resi_dual are float atomic sums over the cells and
    differ in the last bits."""
    arrs = {k: v.cpu().numpy() for k, v in out.items()}
    arrs = {k: a.astype(np.float64 if a.dtype.kind in 'iu' else np.float32) for k, a in arrs.items()}
    B = len(arrs['u'])
    per_instance = sum(a[0].nbytes for a in arrs.values()) + 8
    if B * per_instance > DUMP_LIMIT - 4096:            # 4 KB for the .npy headers
        idx = np.sort(np.random.default_rng(seed).choice(B, (DUMP_LIMIT - 4096) // per_instance, replace=False))
        arrs = {k: a[idx] for k, a in arrs.items()}
        arrs['instance_index'] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(path, f'{k}.npy'), a)


def algorithmic_bytes():
    """SURVEY.md §8d, float32: compulsory HBM bytes per instance-iteration of K2 (cells) and K1 (su)."""
    w = 4
    k2 = w * (N * T * (2 * E + 2 * R + 2 + 4 + 2 + 5) + 3 * N * E * 1 + 4 * T)
    k1 = w * (5 * N * T + 3 * (T + 1) + 2 * (3 * (T + 1) + 3 * T))
    return k2, k1


def _one_instance(job):
    """(config, seed, lateral) -> packed arrays of one seeded instance (worker of build_inputs; numpy only)."""
    from rda_planner_b200.scenarios import config_instance, make_instance, CONFIGS
    from rda_planner_b200.rda_solver import pack_obstacles
    config, seed, lateral = job
    c = CONFIGS[config]
    inst = config_instance(config, seed) if lateral is None else make_instance(seed, T=c['T'], N=c['N'], E=c['E'], lateral=lateral)
    return inst, pack_obstacles(list(inst['obstacles']), c['T'], c['N'], c['E'])


def build_inputs(batch, seed0, config='metric', lateral=None, unique=None):
    """Host arrays of `batch` seeded instances.  The metric row is generated with EVERY instance unique (a process pool over
    the leased host cores: call this before CUDA is initialised); the side configs keep 256 unique instances, tiled.
    lateral: override of the obstacle band of the metric generator (the parity tests use the harsher (0.3, 3.5))."""
    import multiprocessing as mp
    uniq = min(batch, unique if unique is not None else (batch if config == 'metric' else 256))
    jobs = [(config, seed0 + i, lateral) for i in range(uniq)]
    workers = min(32, len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1))
    if uniq >= 512 and workers > 1:
        with mp.get_context('fork').Pool(workers) as pool:
            res = pool.map(_one_instance, jobs, chunksize=max(1, uniq // (8 * workers)))
    else:
        res = [_one_instance(j) for j in jobs]
    insts, packs = [r[0] for r in res], [r[1] for r in res]
    rep = -(-batch // uniq)

    def tile(a):
        return np.concatenate([a] * rep, 0)[:batch]
    return {
        'nom_s': tile(np.stack([i['nom_s'] for i in insts]).astype(np.float32)),
        'nom_u': tile(np.stack([i['nom_u'] for i in insts]).astype(np.float32)),
        'ref_s': tile(np.stack([i['ref'] for i in insts]).astype(np.float32)),
        'ref_speed': tile(np.array([i['ref_speed'] for i in insts], np.float32)),
        'obs_A': tile(np.stack([p[0] for p in packs])),
        'obs_b': tile(np.stack([p[1] for p in packs])),
        'obs_kind': tile(np.stack([p[2] for p in packs])),
        'obs_count': tile(np.array([p[3] for p in packs], np.int32)),
    }


def run_config(args):
    """BASELINE.json configs B-E at their stated global batch (STRONG scaling: the global batch is fixed and split
    over the ranks), 50 ADMM iterations, early stop disabled.  --scatter-from-rank0: rank 0 owns the whole batch; the
    timed region then contains scatter_batch (NCCL) + solve + gather_batch of (u, s) — SURVEY.md §8e "report both".
    Config E additionally runs the float32 su-QP and reports residual / trajectory gaps against float64 by iteration."""
    import torch
    import torch.distributed as dist
    from rda_planner_b200.rda_solver import RDA_solver
    from rda_planner_b200.scenarios import rectangle_robot, CONFIGS
    from rda_planner_b200 import build as rbuild
    from rda_planner_b200.sharding import gather_batch, scatter_batch, shard_bounds
    cfg = CONFIGS[args.config]
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device(f'cuda:{local}')
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')
        dist.init_process_group('nccl', device_id=dev)
    rbuild.build()
    G = args.global_batch or cfg['global_batch']
    lo, hi = shard_bounds(G, world, rank)
    nloc = hi - lo
    car = rectangle_robot(dynamics=cfg['dynamics'])
    Tc, Nc, Ec = cfg['T'], cfg['N'], cfg['E']
    full = build_inputs(G, 1000 * 7, args.config) if (rank == 0 or not args.scatter_from_rank0) else None
    tv = bool(full['obs_A'].shape[2] > 1) if full is not None else False
    if world > 1:
        flag = torch.tensor([int(tv)], device=dev)
        dist.broadcast(flag, 0)
        tv = bool(flag.item())
    full_t = {k: torch.from_numpy(v) for k, v in full.items()} if full is not None else None

    def mk(su_fp64=True):
        return RDA_solver(Tc, car, max_edge_num=Ec, max_obs_num=Nc, iter_num=cfg['iter_num'], iter_threshold=0.0,
                          time_print=False, batch=nloc, device=dev, su_fp64=su_fp64, **cfg['tun'])
    solver = mk()
    if args.scatter_from_rank0:
        src = {k: v.to(dev) for k, v in full_t.items()} if rank == 0 else None      # resident on rank 0's GPU
    else:
        devin = {k: v[lo:hi].to(dev) for k, v in full_t.items()}

    def step():
        if args.scatter_from_rank0:
            inp, n = scatter_batch(src, G, dev)
        else:
            inp = devin
        solver.cold_start()
        out = solver.iterative_solve_batch(inp['nom_s'], inp['nom_u'], inp['ref_s'], inp['ref_speed'], inp['obs_A'],
                                           inp['obs_b'], inp['obs_kind'], inp['obs_count'], tv)
        if args.scatter_from_rank0:
            gu = gather_batch(out['u'], G)
            gs = gather_batch(out['s'], G)
            return out, (gu, gs)
        return out, None

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out, gathered = step()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    st = out['status'].cpu()
    bits = torch.tensor([int(((st & b) != 0).sum()) for b in (1, 2, 4)], device=dev)
    if world > 1:
        dist.all_reduce(bits)
    line = {'metric': f'MPC solves/sec (config {args.config}: {cfg["what"]}, {cfg["iter_num"]} ADMM iterations)',
            'value': G * args.steps / (ms * 1e-3), 'unit': 'solves/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32 state / f64 su-QP interior point', 'data': 'synthetic',
            'config': {'workload': f'BASELINE config {args.config}', 'global_batch': G, 'batch_per_gpu': nloc,
                       'T': Tc, 'N': Nc, 'E': Ec, 'time_varying_obstacles': tv,
                       'inputs': 'scattered from rank 0 over NCCL inside the timed region, (u, s) gathered back'
                       if args.scatter_from_rank0 else 'each rank generates its shard in place',
                       'l2_policy': 'cold start every step; state of one step exceeds L2 only for configs D/E at full batch'},
            'status_bits': {'su_iteration_cap(1)': int(bits[0]), 'su_nonfinite_keep_previous(2)': int(bits[1]),
                            'cell_failed_keep_previous(4)': int(bits[2])},
            'gpu_launches': (solver.launch_count() + 1) * args.steps}
    from rda_planner_b200 import _cabi
    cnt = solver.state_buffer(_cabi.BUF_COUNTERS).cpu().numpy().tolist()
    cells = max(nloc * Nc * Tc * cfg['iter_num'], 1)
    line['counters_rank0_last_step'] = {'cells_closed_form_fraction': cnt[0] / cells, 'cells_interior_point_fraction': cnt[1] / cells,
                                        'cells_failed': cnt[2], 'su_ipm_iterations_per_solve': cnt[3] / max(cnt[4], 1)}
    if args.scatter_from_rank0 and rank == 0:
        line['gathered_shapes'] = [list(gathered[0].shape), list(gathered[1].shape)]
        line['scatter_bytes_per_step'] = int(sum(v.numel() * v.element_size() for v in src.values()))
    if args.config == 'E' or args.precision_sweep:
        # float32 vs float64 su-QP: residuals and trajectory gap by iteration (same inputs, phase API)
        inp = scatter_batch(src, G, dev)[0] if args.scatter_from_rank0 else devin
        s32 = mk(False)
        rows = []
        runs = {}
        for name, sv in (('f64', solver), ('f32', s32)):
            sv.cold_start()
            sv.begin(inp['nom_s'], inp['nom_u'], inp['ref_s'], inp['ref_speed'], inp['obs_A'], inp['obs_b'], inp['obs_kind'],
                     inp['obs_count'], tv, 0.0)
            tr = {}
            for it in range(1, cfg['iter_num'] + 1):
                sv.step_su(); sv.step_lammuz()
                if it in (1, 2, 4, 8, 16, 32, cfg['iter_num']):
                    o = sv.finish()
                    tr[it] = {k: o[k].clone() for k in ('s', 'u', 'resi_pri', 'resi_dual')}
            runs[name] = tr
        for it in sorted(runs['f64']):
            a, b = runs['f64'][it], runs['f32'][it]
            gap = (a['s'] - b['s']).abs().flatten(1).max(1).values
            rows.append({'iteration': it,
                         'resi_pri_f64_median': float(a['resi_pri'].median()), 'resi_pri_f32_median': float(b['resi_pri'].median()),
                         'resi_dual_f64_median': float(a['resi_dual'].median()), 'resi_dual_f32_median': float(b['resi_dual'].median()),
                         'state_gap_median': float(gap.median()), 'state_gap_p95': float(gap.quantile(0.95)), 'state_gap_max': float(gap.max())})
        line['fp32_vs_fp64_su'] = rows
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.idx), '-lms', '100'], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def cpu_port_rate(inputs, sample, threads, iters=ITERS):
    """Compiled CPU port (oracle/cpu_port) on `sample` instances; returns (solves/s, seconds)."""
    from oracle import cpu_port
    from rda_planner_b200.scenarios import rectangle_robot
    sub = {k: v[:sample] for k, v in inputs.items()}
    t0 = time.perf_counter()
    cpu_port.solve_batch(rectangle_robot(), T, N, E, sub['nom_s'], sub['nom_u'], sub['ref_s'], sub['ref_speed'],
                         sub['obs_A'], sub['obs_b'], sub['obs_kind'], sub['obs_count'], iter_num=iters,
                         iter_threshold=0.0, threads=threads)
    dt = time.perf_counter() - t0
    return sample / dt, dt


def closed_loop_probe(dev, B, steps=3):
    """SURVEY.md §8 f1-f3: whole control steps on the device (pre_process -> obstacle conversion ->
    50-iteration solve -> arrive rule -> state advance) for B robots on one 60 m reference line.
    Reported next to the headline metric, not instead of it."""
    import torch
    from rda_planner_b200.frontend import BatchedMPC
    from rda_planner_b200.scenarios import rectangle_robot
    rng = np.random.default_rng(77)
    path = np.stack([np.arange(0, 60, 0.1), np.zeros(600), np.zeros(600)], 1)
    bm = BatchedMPC(rectangle_robot(), path, B, receding=T, sample_time=0.1, iter_num=ITERS, max_edge_num=E,
                    max_obs_num=N, iter_threshold=0.0, device=dev)
    idx = rng.integers(0, 480, B)
    state = torch.as_tensor(path[idx] + rng.normal(0, [0.3, 0.3, 0.1], (B, 3)), dtype=torch.float32, device=dev)
    bm.cur_index[:] = torch.as_tensor(np.maximum(idx - 3, 0), dtype=torch.int32)
    bm.cur_vel[:, 0, :] = 4.0
    # N boxes (2 x 1 m, random yaw) per robot, 2-8 m ahead and 1.5-5 m to either side
    M = N
    ctr = path[idx][:, None, :2] + np.stack([rng.uniform(2, 14, (B, M)), rng.uniform(1.8, 6, (B, M)) * rng.choice([-1, 1], (B, M))], -1)
    yaw = rng.uniform(0, np.pi, (B, M))
    corners = np.array([[-1, -0.5], [1, -0.5], [1, 0.5], [-1, 0.5]])
    rot = np.stack([np.stack([np.cos(yaw), -np.sin(yaw)], -1), np.stack([np.sin(yaw), np.cos(yaw)], -1)], -2)
    xy = np.zeros((B, M, 8, 2), np.float32)
    xy[:, :, :4] = ctr[:, :, None, :] + np.einsum('bmij,kj->bmki', rot, corners)
    shapes = {'kind': np.zeros((B, M), np.int32), 'nv': np.full((B, M), 4, np.int32), 'xy': xy,
              'radius': np.zeros((B, M), np.float32), 'vel': np.zeros((B, M, 2), np.float32),
              'count': np.full(B, M, np.int32)}
    shapes = {k: torch.as_tensor(v, device=dev) for k, v in shapes.items()}
    bm.control(state, 4.0, shapes)
    bm.advance(state)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        u0, info = bm.control(state, 4.0, shapes)
        bm.advance(state)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    ok = bool(torch.isfinite(u0).all()) and int((info['status'] & 6).sum()) == 0
    return {'mpc_steps_per_s': B / (ms * 1e-3), 'ms_per_control_step': ms, 'robots': B, 'finite_and_converged': ok,
            'what': 'BatchedMPC.control + advance: pre_process, obstacle conversion, 50 ADMM iterations (warm-started), '
                    'arrive rule, model step; all on the device'}


def extra_probes(dev, solver, devin, B, host_harsh=None):
    """SURVEY.md §8(d) side measurements (never the headline): the same batch with the reference's
    early-stop rule (iter_threshold 0.2, rda_solver.py:22,594-596) and the latency of ONE instance
    (the reference's own use case)."""
    import torch
    from rda_planner_b200.rda_solver import RDA_solver
    from rda_planner_b200.scenarios import rectangle_robot
    out = {}

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps, r

    def early():
        solver.cold_start()
        return solver.iterative_solve_batch(devin['nom_s'], devin['nom_u'], devin['ref_s'], devin['ref_speed'],
                                            devin['obs_A'], devin['obs_b'], devin['obs_kind'], devin['obs_count'], False,
                                            iter_threshold=0.2)
    ms, r = timed(early, 2)
    out['early_stop'] = {'solves_per_s': B / (ms * 1e-3), 'iter_threshold': 0.2,
                         'mean_iterations': float(r['iters'].float().mean()),
                         'stopped_early_fraction': float((r['iters'] < ITERS).float().mean())}
    one = RDA_solver(T, rectangle_robot(), max_edge_num=E, max_obs_num=N, iter_num=ITERS, iter_threshold=0.0,
                     time_print=False, batch=1, device=dev)
    d1 = {k: v[:1].contiguous() for k, v in devin.items()}

    def single():
        one.cold_start()
        return one.iterative_solve_batch(d1['nom_s'], d1['nom_u'], d1['ref_s'], d1['ref_speed'], d1['obs_A'], d1['obs_b'],
                                         d1['obs_kind'], d1['obs_count'], False)
    ms1, _ = timed(single, 3)
    out['single_instance'] = {'latency_ms': ms1, 'what': 'one instance, 50 iterations, cold start, inputs on the device '
                                                         '(single-launch persistent kernel, SURVEY §8 f4)'}
    # the reference's own use case (example/path_track/path_track.py:22): T=10, N=11, iter_num=2, one robot, warm-started
    # control steps through the numpy-in / numpy-out API (host copies included), eager and with CUDA-graph replay
    from rda_planner_b200.scenarios import make_instance, CONFIGS
    inst = make_instance(4242, T=10, N=11, E=4, lateral=(1.5, 6.0))
    ref = [inst['ref'][:, t:t + 1] for t in range(11)]
    lat = {}
    for name, graph in (('eager', False), ('graph', True)):
        sv = RDA_solver(10, rectangle_robot(), max_edge_num=4, max_obs_num=11, iter_num=2, time_print=False, device=dev, graph=graph,
                        ro1=300)
        for _ in range(3):
            sv.iterative_solve(inst['nom_s'], inst['nom_u'], ref, 4.0, list(inst['obstacles']))
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(20):
            sv.iterative_solve(inst['nom_s'], inst['nom_u'], ref, 4.0, list(inst['obstacles']))
        torch.cuda.synchronize(dev)
        lat[name] = (time.perf_counter() - t0) / 20 * 1e3
    out['path_track_control_step'] = {'latency_ms': lat, 'what': 'T=10, N=11, iter_num=2, one instance, reference signature '
                                      '(numpy in/out, host<->device copies and packing included), warm-started'}
    # BASELINE configs B and C at their stated single-GPU batch (strong-scaling side benches: bench.py --config B|C|D|E)
    for cname in ('B', 'C'):
        c = CONFIGS[cname]
        h = build_inputs(c['global_batch'], 7000, cname)
        di = {k: torch.from_numpy(v).to(dev) for k, v in h.items()}
        tv = h['obs_A'].shape[2] > 1
        sv = RDA_solver(c['T'], rectangle_robot(dynamics=c['dynamics']), max_edge_num=c['E'], max_obs_num=c['N'], iter_num=c['iter_num'],
                        iter_threshold=0.0, time_print=False, batch=c['global_batch'], device=dev, **c['tun'])

        def cfg_step():
            sv.cold_start()
            return sv.iterative_solve_batch(di['nom_s'], di['nom_u'], di['ref_s'], di['ref_speed'], di['obs_A'], di['obs_b'],
                                            di['obs_kind'], di['obs_count'], tv)
        msc, r = timed(cfg_step, 2)
        out[f'config_{cname}'] = {'solves_per_s': c['global_batch'] / (msc * 1e-3), 'batch': c['global_batch'], 'what': c['what'],
                                  'kept_previous_iterate': int((r['status'] & 6).ne(0).sum())}
    # the metric shape on the HARSH obstacle band of the parity tests (lateral offsets 0.3-3.5 m instead of 1.8-6 m: more
    # overlapping and active cells, i.e. more work for the searched closed forms and the interior point pass)
    if host_harsh is not None:
        Bh = host_harsh['nom_s'].shape[0]
        dh = {k: torch.from_numpy(v).to(dev) for k, v in host_harsh.items()}
        svh = RDA_solver(T, rectangle_robot(), max_edge_num=E, max_obs_num=N, iter_num=ITERS, iter_threshold=0.0, time_print=False,
                         batch=Bh, device=dev)

        def harsh_step():
            svh.cold_start()
            return svh.iterative_solve_batch(dh['nom_s'], dh['nom_u'], dh['ref_s'], dh['ref_speed'], dh['obs_A'], dh['obs_b'],
                                             dh['obs_kind'], dh['obs_count'], False)
        msh, r = timed(harsh_step, 2)
        from rda_planner_b200 import _cabi as _c
        cn = svh.state_buffer(_c.BUF_COUNTERS).cpu().tolist()
        out['harsh_geometry'] = {'solves_per_s': Bh / (msh * 1e-3), 'batch': Bh, 'what': 'metric shape, obstacle band 0.3-3.5 m beside '
                                 'the path (tests/test_gpu_parity.py) instead of 1.8-6 m', 'kept_previous_iterate': int((r['status'] & 6).ne(0).sum()),
                                 'interior_point_cell_fraction': cn[1] / max(1, cn[0] + cn[1])}
        # same batch size on the default band, for the ratio
        dm = {k: v[:Bh].contiguous() for k, v in devin.items()}
        svm = RDA_solver(T, rectangle_robot(), max_edge_num=E, max_obs_num=N, iter_num=ITERS, iter_threshold=0.0, time_print=False,
                         batch=Bh, device=dev)

        def mild_step():
            svm.cold_start()
            return svm.iterative_solve_batch(dm['nom_s'], dm['nom_u'], dm['ref_s'], dm['ref_speed'], dm['obs_A'], dm['obs_b'],
                                             dm['obs_kind'], dm['obs_count'], False)
        msm, _ = timed(mild_step, 2)
        out['harsh_geometry']['default_band_same_batch_solves_per_s'] = Bh / (msm * 1e-3)
    # the metric shape with a DISC body (car_tuple.cone_type 'norm2', rda_solver.py:1034-1039): closed forms for the inactive
    # hinges, two-cone barrier programmes for the rest (cell_disc_robot.cuh) — a coverage row, not tuned
    from rda_planner_b200.scenarios import disc_robot
    Bd = min(B, 2048)
    dd = {k: v[:Bd].contiguous() for k, v in devin.items()}
    svd = RDA_solver(T, disc_robot(radius=1.2, wheelbase=2.0, dynamics='diff'), max_edge_num=E, max_obs_num=N, iter_num=ITERS,
                     iter_threshold=0.0, time_print=False, batch=Bd, device=dev)

    def disc_step():
        svd.cold_start()
        return svd.iterative_solve_batch(dd['nom_s'], dd['nom_u'], dd['ref_s'], dd['ref_speed'], dd['obs_A'], dd['obs_b'],
                                         dd['obs_kind'], dd['obs_count'], False)
    msd, r = timed(disc_step, 2)
    out['disc_robot'] = {'solves_per_s': Bd / (msd * 1e-3), 'batch': Bd, 'what': 'metric shape, disc body of radius 1.2 m, diff drive',
                         'kept_previous_iterate': int((r['status'] & 6).ne(0).sum())}
    return out


def cpu_arm(inputs, budget_s=12.0):
    """The CPU port on the host cores this process may really use (oracle.cpu_port.host_threads: affinity mask and
    cgroup quota, not os.cpu_count()), threads pinned (OMP_PROC_BIND / OMP_PLACES set before libgomp starts), library
    loaded once outside the timed region, best thread count of a short sweep.  Returns (solves/s, info dict)."""
    os.environ.setdefault('OMP_PROC_BIND', 'close')
    os.environ.setdefault('OMP_PLACES', 'cores')
    os.environ.setdefault('OMP_DYNAMIC', 'false')
    from oracle import cpu_port
    ht = cpu_port.host_threads()
    eff = ht['effective']
    cpu_port._lib()
    n_have = inputs['nom_s'].shape[0]
    cpu_port_rate(inputs, min(n_have, max(eff, 4)), eff, iters=2)               # warm-up: page in, spawn the team
    cands = sorted({eff, max(1, eff // 2), max(1, eff // 4)}, reverse=True)
    sweep = {}
    for th in cands:
        n = min(n_have, max(2 * th, 8))
        v, dt = cpu_port_rate(inputs, n, th)
        sweep[th] = v
    best = max(sweep, key=sweep.get)
    n = min(n_have, max(int(sweep[best] * budget_s), 2 * best, 8))
    n -= n % best if n >= 2 * best else 0
    v, dt = cpu_port_rate(inputs, n, best)
    info = {'cores': best, 'host': ht, 'thread_sweep_solves_per_s': {str(k): round(x, 2) for k, x in sweep.items()},
            'per_core_solves_per_s': v / best, 'sample_instances': n, 'seconds': dt,
            'omp': {k: os.environ.get(k) for k in ('OMP_PROC_BIND', 'OMP_PLACES')}}
    return v, info


def run_reference(args):
    """CPU arm: the path on the host cores.  The reference's own implementation (cvxpy/ECOS/pathos) is
    not installable in this image (DESIGN.md §0), so this times the compiled port — the SAME algorithm as
    the CUDA kernels (kind "port"), not the reference's solver."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import cpu_port
    eff = cpu_port.host_threads()['effective']
    inputs = build_inputs(max(64, 8 * eff), 1000 * 9)
    v0, info = cpu_arm(inputs, budget_s=6.0)
    sample, th = info['sample_instances'], info['cores']
    for _ in range(max(args.warmup - 1, 0)):
        cpu_port_rate(inputs, min(sample, 2 * th), th)
    t = 0.0
    for _ in range(args.steps):
        _, dt = cpu_port_rate(inputs, sample, th)
        t += dt
    value = sample * args.steps / t
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'solves/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64/f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'batch_per_step': sample},
            'cpu_baseline': {'value': value, 'unit': 'solves/s', 'cores': th, 'kind': 'port',
                             'what': 'compiled C++ port of THIS repo\'s algorithm (oracle/cpu_port), not cvxpy/ECOS',
                             'host': info['host'], 'thread_sweep_solves_per_s': info['thread_sweep_solves_per_s'],
                             'per_core_solves_per_s': value / th,
                             'sample': f'{sample} instances x {ITERS} ADMM iterations per step, OpenMP over instances, '
                                       f'{th} pinned threads'},
            'e2e': {'value': value, 'unit': 'solves/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=16384, help='instances per GPU per step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--config', default='metric', choices=['metric', 'B', 'C', 'D', 'E'],
                    help='BASELINE.json config (default: the metric row, the headline); B-E are strong-scaling side benches')
    ap.add_argument('--global-batch', type=int, default=0, help='override the global batch of --config B..E')
    ap.add_argument('--scatter-from-rank0', action='store_true',
                    help='--config B..E: rank 0 owns the batch; scatter + solve + gather inside the timed region')
    ap.add_argument('--precision-sweep', action='store_true', help='--config B..E: float32 vs float64 su-QP by iteration')
    ap.add_argument('--su-fp32', action='store_true', help='float32 su-QP arithmetic (lower bound probe, not the metric)')
    ap.add_argument('--no-probes', action='store_true', help='skip early-stop / single-instance / closed-loop probes')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the results of the last timed step (rank 0\'s instances) as DIR/<name>.npy, at most 64 MB')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the results of the GPU path; the reference arm has none')
    if args.impl == 'reference':
        return run_reference(args)
    if args.config != 'metric':
        return run_config(args)

    import torch
    import torch.distributed as dist
    from rda_planner_b200.rda_solver import RDA_solver
    from rda_planner_b200.scenarios import rectangle_robot
    from rda_planner_b200 import build as rbuild
    from rda_planner_b200.sharding import gather_batch

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.warmup < 3:
        args.warmup = 3
    B = args.batch
    # host inputs first (process pool over the host cores: before CUDA / NCCL are initialised).  Every instance unique.
    host = build_inputs(B, 1000 * 9 + rank * B)              # per-rank shard, generated in place (weak scaling)
    host_harsh = None
    if rank == 0 and not args.no_probes:
        host_harsh = build_inputs(min(B, 2048), 5000 * 9, lateral=(0.3, 3.5))      # the parity tests' obstacle band
    torch.cuda.set_device(local)
    dev = torch.device(f'cuda:{local}')
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')      # keep stdout to the one JSON line
        dist.init_process_group('nccl', device_id=dev)
    rbuild.build()
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
    devin = {k: v.to(dev) for k, v in pinned.items()}
    solver = RDA_solver(T, rectangle_robot(), max_edge_num=E, max_obs_num=N, iter_num=ITERS, iter_threshold=0.0,
                        time_print=False, batch=B, device=dev, su_fp64=not args.su_fp32)

    def step(inp):
        solver.cold_start()
        return solver.iterative_solve_batch(inp['nom_s'], inp['nom_u'], inp['ref_s'], inp['ref_speed'], inp['obs_A'],
                                            inp['obs_b'], inp['obs_kind'], inp['obs_count'], False)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step(devin)
    launches_per_step = solver.launch_count() + 1           # + the cold-start fill kernel
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step(devin)
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)        # before the probes below reuse the solver's output buffers
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    status = out['status'].clone()
    # ---- end to end: pinned host inputs -> H2D -> solve -> D2H of the result, every step ----
    hout = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()}
    h2d = sum(v.numel() * v.element_size() for v in pinned.values())
    d2h = sum(v.numel() * v.element_size() for v in hout.values())

    def e2e_step():
        inp = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
        o = step(inp)
        for k, v in o.items():
            hout[k].copy_(v, non_blocking=True)
    for _ in range(2):
        e2e_step()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        e2e_step()
    e3.record()
    barrier()
    ms2 = torch.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms2 = float(ms2.item())
    clocks = sampler.stop() if rank == 0 else None
    # trajectories to rank 0 (the only collective of the path; outside the ADMM loop)
    full_u = gather_batch(out['u'], B * world) if world > 1 else out['u']
    # ---- per-kernel durations for the roofline (CUDA events on the launching stream) ----
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(ITERS)]
    solver.cold_start()
    solver.begin(devin['nom_s'], devin['nom_u'], devin['ref_s'], devin['ref_speed'], devin['obs_A'], devin['obs_b'],
                 devin['obs_kind'], devin['obs_count'], False, 0.0)
    for i in range(ITERS):
        ev[i][0].record(); solver.step_su(); ev[i][1].record(); solver.step_lammuz(); ev[i][2].record()
    solver.finish()
    torch.cuda.synchronize(dev)
    t_su = float(np.mean([ev[i][0].elapsed_time(ev[i][1]) for i in range(1, ITERS)]))       # ms
    t_cells = float(np.mean([ev[i][1].elapsed_time(ev[i][2]) for i in range(1, ITERS)]))    # cells + finalize
    from rda_planner_b200 import _cabi
    counters = solver.state_buffer(_cabi.BUF_COUNTERS).cpu().numpy().tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    k2b, k1b = algorithmic_bytes()
    dominant = 'k_su' if t_su >= t_cells else 'k_cells'
    dur = max(t_su, t_cells) * 1e-3
    alg = (k1b if dominant == 'k_su' else k2b) * B
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(dominant)
    achieved = alg / dur / 1e9
    total = B * world * args.steps
    line = {
        'metric': METRIC, 'value': total / (ms * 1e-3), 'unit': 'solves/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32 state / f64 su-QP interior point', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'batch_per_gpu': B, 'global_batch': B * world, 'unique_instances_per_gpu': B,
                   'parallelism': f'instances sharded over {world} GPU(s), no collective in the ADMM loop',
                   'l2_policy': f'per-step working set {41 * B // 1000} MB of warm-start state > 126 MB L2'
                   if B >= 3200 else 'working set below L2 size (small batch)'},
        'e2e': {'value': total / (ms2 * 1e-3), 'unit': 'solves/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
        'gpu_launches': launches_per_step * args.steps,
        'clocks': clocks,
        'roofline': {'bound': 'hbm', 'kernel': dominant, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                     'algorithmic_bytes_per_launch': alg, 'kernel_ms': {'k_su': t_su, 'k_cells+k_finalize': t_cells},
                     'k_cells': {'achieved': k2b * B / (t_cells * 1e-3) / 1e9, 'frac': k2b * B / (t_cells * 1e-3) / 1e9 / peak},
                     'k_su': {'achieved': k1b * B / (t_su * 1e-3) / 1e9, 'frac': k1b * B / (t_su * 1e-3) / 1e9 / peak}},
        'counters': {'cells_fast': counters[0], 'cells_slow': counters[1], 'cells_failed': counters[2],
                     'su_ipm_iterations': counters[3], 'su_solves': counters[4], 'su_pruned_solves_repeated': counters[5]},
        'status_nonzero': int((status.cpu() != 0).sum()),
        'status_bits': {'su_iteration_cap(1)': int(((status.cpu() & 1) != 0).sum()),
                        'su_nonfinite_keep_previous(2)': int(((status.cpu() & 2) != 0).sum()),
                        'cell_failed_keep_previous(4)': int(((status.cpu() & 4) != 0).sum()),
                        'early_stop(8)': int(((status.cpu() & 8) != 0).sum())},
        'gathered_u_shape': list(full_u.shape),
    }
    if world == 1 and not args.no_cpu_baseline:
        v, info = cpu_arm(host, budget_s=12.0)
        line['cpu_baseline'] = {'value': v, 'unit': 'solves/s', 'cores': info['cores'], 'kind': 'port',
                                'what': 'compiled C++ port of THIS repo\'s algorithm (oracle/cpu_port), not cvxpy/ECOS',
                                'host': info['host'], 'thread_sweep_solves_per_s': info['thread_sweep_solves_per_s'],
                                'per_core_solves_per_s': info['per_core_solves_per_s'],
                                'sample': f"{info['sample_instances']} of the same instances x {ITERS} ADMM iterations, OpenMP over "
                                          f"instances, {info['cores']} pinned threads, {info['seconds']:.1f} s"}
    if not args.no_probes:
        try:
            line.update(extra_probes(dev, solver, devin, B, host_harsh))
        except Exception as ex:
            line['early_stop'] = {'error': repr(ex)[:200]}
        try:
            line['closed_loop'] = closed_loop_probe(dev, B)
        except Exception as ex:          # the probe must never cost the headline line
            line['closed_loop'] = {'error': repr(ex)[:200]}
    print(json.dumps(line), flush=True)
    bad = line['status_bits']['su_nonfinite_keep_previous(2)'] + line['status_bits']['cell_failed_keep_previous(4)']
    if bad:
        raise SystemExit(f'bench: {bad} instances kept a previous iterate (status bits 2/4) — the metric is void')
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
