#!/usr/bin/env python3
"""bench.py — env-steps/s of the batched FeedingJaco-v1 physics step (BASELINE.json metric).

A "step" is one `env.step` over the whole batch: action -> PD targets -> 5 physics substeps ->
obs / reward / done read-back (reference envs/feeding.py:12-37, envs/env.py:174-235).

  python bench.py --gpus N --steps K --warmup W        (torchrun launches it for N > 1)
  python bench.py --impl reference ...                 CPU arm: the oracle restatement on host cores
                                                       (PyBullet, the real reference path, is not installable here)

Prints ONE JSON line on rank 0.  `value` = device-resident throughput (actions already in HBM),
`e2e` = the same metric through the host-buffer C-ABI call (H2D of actions, D2H of obs/reward/done
inside the timed region), `roofline` = the dominant kernel's algorithmic bytes / measured device
time against the measured HBM peak, `cpu_baseline` = the oracle timed on a bounded sample.
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

B_SUBSTEP = 2458          # algorithmic bytes per env-substep (SURVEY.md §8(d): 12 288 B per env-step / 5)
B_STEP = 12288
BATCH_PER_GPU = 4096
METRIC = 'env-steps/sec FeedingJaco-v1 @batch4096'


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu):
        self.gpu = gpu
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': float(np.max(mx)) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def usable_cores():
    """Host threads this process may really use: the affinity mask capped by the cgroup CPU quota (a 1-GPU lease can be
    a slice of a 128-thread host: os.cpu_count() over-subscribed it 20x and the CPU arm swung 5.7x between boxes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_oracle_rate(fb, n_envs, env_steps, threads, seed=0):
    """env-steps/s of the CPU oracle on a bounded sample of the same workload."""
    from assistive_gym_b200 import capi
    from oracle.oracle_py import OracleSim
    from tests.parity_cases import take_step_targets
    cpu = OracleSim(fb.scene, capi.default_config(), n_envs, threads=threads)
    rng = np.random.default_rng(seed)
    fb.reset(cpu, rng, settle_steps=25)
    t0 = time.perf_counter()
    for _ in range(env_steps):
        act = rng.uniform(-1, 1, size=(n_envs, 7))
        tgt = take_step_targets(cpu.get_joint_states(fb.arm_links)[0], act, fb.arm_lower, fb.arm_upper)
        cpu.set_motor_targets(fb.arm_links, tgt)
        cpu.step(5)
        # read-back that feeds obs / reward (same queries the reference issues per step)
        cpu.get_link_states([fb.ee_link, int(fb.scene['body_link0'][fb.tool])])
        for hb in fb.humans.values():
            cpu.contact_force_sum(fb.tool, hb)
            cpu.contact_force_sum(fb.robot, hb)
    dt = time.perf_counter() - t0
    return n_envs * env_steps / dt, dt


def pybullet_rate(env_steps):
    """The real reference, if it can be imported on this box: gym.make('assistive_gym:FeedingJaco-v1') stepped with
    random actions in one process (BASELINE.md section 2 step 1).  None when PyBullet / the reference are absent."""
    try:
        import pybullet  # noqa: F401
        import gym
        import assistive_gym  # noqa: F401  (the reference package, not this repo's shim)
        if getattr(assistive_gym, '__agphys_shim__', False):
            return None
        env = gym.make('assistive_gym:FeedingJaco-v1')
        env.seed(1001)
        env.reset()
        rng = np.random.default_rng(0)
        t0 = time.perf_counter()
        for _ in range(env_steps):
            env.step(rng.uniform(-1, 1, size=7))
        return env_steps / (time.perf_counter() - t0)
    except Exception:
        return None


def run_reference(args):
    """--impl reference: the reference's CPU path on the box's host cores.  PyBullet is tried first (never installable
    in the build container, SURVEY.md 8(c)); otherwise the oracle port is timed, kind = "port", on the SAME workload
    size as the product arm (batch envs per GPU), with all usable host threads and with one."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from assistive_gym_b200.feeding_batch import FeedingBatch
    fb = FeedingBatch()
    cores = usable_cores()
    n_envs = args.batch
    pb = pybullet_rate(200)
    env_steps = 2                                     # per timed sample: bounded so that --steps K ends within minutes
    cpu_oracle_rate(fb, max(cores, 8), 1, cores)      # warm-up (library load, first-touch)
    rates, times = [], []
    for _ in range(max(1, min(args.steps, 3))):
        r, t = cpu_oracle_rate(fb, n_envs, env_steps, cores)
        rates.append(r)
        times.append(t)
    v = float(np.median(rates))
    r1, t1 = cpu_oracle_rate(fb, max(n_envs // max(cores, 1), 32), env_steps, 1)
    sample = '%d envs x %d env-steps per timed sample, %d samples, oracle port (CPU restatement - PyBullet %s), %d threads' % (
        n_envs, env_steps, len(rates), 'timed separately' if pb else 'unavailable', cores)
    out = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
           'warmup': args.warmup, 'ms_per_step': 1000.0 * float(np.median(times)) / env_steps, 'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
           'config': {'workload': 'FeedingJaco-v1, batch %d, CPU restatement (PyBullet %s)' % (n_envs, 'also timed' if pb else 'unavailable'),
                      'global_batch': n_envs, 'l2': 'n/a (CPU)'},
           'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port', 'sample': sample,
                            'one_thread': {'value': float(r1), 'cores': 1},
                            'pybullet_one_process': ({'value': float(pb), 'cores': 1, 'kind': 'reference'} if pb else None)},
           'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
           'gpu_launches': 0}
    print(json.dumps(out))


def run_bedbathing(args):
    """BASELINE.json configs[2]: BedBathingSawyer-v1 @ batch 4096 on one B200, fused step, from a start pose with the
    wiping pad 3 mm above the forearm (random joint actions press it onto the skin): device-timed value + host-buffer e2e."""
    import torch
    from assistive_gym_b200 import capi
    from assistive_gym_b200.bed_bathing_batch import BedBathingBatch
    from assistive_gym_b200.sim import BatchSim
    if args.impl == 'reference':
        print(json.dumps({'impl': 'reference', 'unavailable': 'the bedbathing line has no CPU arm (the oracle is timed on the headline workload only)'}))
        return
    n, K, W = args.batch, args.steps, max(args.warmup, 3)
    bb = BedBathingBatch()
    sim = BatchSim(bb.scene, capi.default_config(), n)
    rng = np.random.default_rng(0)
    t0 = time.time()
    s = bb.reset(sim, rng, toc_attempts=args.toc_attempts)
    ik_err = bb.hover_over_forearm(sim, s, rng, gap=-args.press_mm * 1e-3)      # SURVEY.md 8(d) C2: the pad starts pressed into the forearm
    bb.start_fused(sim, s)
    reset_s = time.time() - t0
    stream = torch.cuda.ExternalStream(sim.stream_ptr())
    dev = torch.device('cuda')
    act = (torch.rand((K + W, n, 7), device=dev) * 2 - 1) * args.action_scale
    obs = torch.zeros((n, 24), device=dev); rew = torch.zeros(n, device=dev); done = torch.zeros(n, device=dev); info = torch.zeros((n, 4), device=dev)
    torch.cuda.synchronize()
    for i in range(W):
        sim.bathing_step_dev(act[i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
    torch.cuda.synchronize()
    clocks = ClockSampler(0); clocks.start()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cs, fs = [], []
    with torch.cuda.stream(stream):
        a.record(stream)
    for i in range(K):
        sim.bathing_step_dev(act[W + i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
    with torch.cuda.stream(stream):
        b.record(stream)
    torch.cuda.synchronize()
    clk = clocks.stop()
    ms = a.elapsed_time(b) / K
    cnt, it = sim.solver_stats()
    host_a = (np.random.default_rng(1).uniform(-1, 1, size=(K, n, 7)) * args.action_scale).astype(np.float32)
    sim.bathing_step_host(host_a[0])
    t0 = time.perf_counter()
    for i in range(K):
        sim.bathing_step_host(host_a[i])
    e2e = n * K / (time.perf_counter() - t0)
    force = info[:, 2].cpu().numpy()
    print(json.dumps({'metric': 'env-steps/sec BedBathingSawyer-v1 @batch%d' % n, 'value': n / ms * 1e3, 'unit': 'env-steps/s', 'n_gpus': 1, 'steps': K, 'warmup': W,
                      'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': {'workload': 'BedBathingSawyer-v1, batch %d, fused step, wiping pad started pressed %.0f mm into the forearm, random actions x %.2f' % (n, args.press_mm, args.action_scale),
                                 'global_batch': n, 'l2': 'not flushed (back-to-back steps)', 'reset_s': reset_s,
                                 'ik_unresolved': int((ik_err >= 0.03).sum()),
                                 'contacts_per_env': {'mean': float(cnt.mean()), 'p99': float(np.percentile(cnt, 99)), 'max': int(cnt.max())},
                                 'envs_with_tool_force': float((force > 0).mean()), 'tool_force_mean_N': float(force[force > 0].mean()) if (force > 0).any() else 0.0,
                                 'pgs_iters_per_env': {'mean': float(it.mean()), 'max': int(it.max())}},
                      'clocks': clk, 'e2e': {'value': e2e, 'unit': 'env-steps/s', 'h2d_bytes_per_step': n * 7 * 4, 'd2h_bytes_per_step': n * 30 * 4},
                      'gpu_launches': int(sim.kernel_launches())}))


def run_dressing(args):
    """BASELINE.json configs[3]: DressingPR2-v1 @ batch 2048 on one B200 (cloth-capsule contact path), fused step: device-timed
    value, host-buffer e2e, the roofline of k_cloth (the one HBM-shaped kernel of the repo: SURVEY.md 8(d), 190 KB of cloth
    state per env and substep) and the CPU oracle on a bounded sample."""
    import torch
    from assistive_gym_b200 import capi
    from assistive_gym_b200.dressing_batch import DressingBatch
    from assistive_gym_b200.sim import BatchSim
    n, K, W = (args.batch if args.batch != BATCH_PER_GPU else 2048), args.steps, max(args.warmup, 3)
    db = DressingBatch()
    cfg = DressingBatch.config()
    rng = np.random.default_rng(0)
    if args.impl == 'reference':
        from oracle.oracle_py import OracleSim
        cores = usable_cores()
        ne = max(cores, 8)
        gpu_free = None
        try:                                   # the reset needs the device IK: replay a stored reset when there is no GPU
            gsim = BatchSim(db.scene, cfg, ne)
            smp = db.reset(gsim, rng, attempts=10, settle_steps=0)
            gsim.close()
        except Exception as ex:                # pragma: no cover
            print(json.dumps({'impl': 'reference', 'unavailable': 'dressing CPU arm needs the device IK for its reset: %s' % ex}))
            return
        orc = OracleSim(db.scene, cfg, ne, threads=cores)
        db.reset(orc, rng, sample=smp, settle_steps=0)
        t0 = time.perf_counter()
        steps = 0
        while time.perf_counter() - t0 < 15.0 or steps < 1:
            orc.step(1); orc.cloth_anchor_follow(db.ee_link); steps += 1
        dt = time.perf_counter() - t0
        v = ne * steps / 5.0 / dt
        print(json.dumps({'metric': 'env-steps/sec DressingPR2-v1 @batch%d' % n, 'impl': 'reference', 'value': v, 'unit': 'env-steps/s', 'n_gpus': 1, 'steps': K, 'warmup': W,
                          'ms_per_step': 1e3 * n / v, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                          'config': {'workload': 'DressingPR2-v1, CPU restatement (PyBullet unavailable), %d envs x %d stepSimulation calls' % (ne, steps)},
                          'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port', 'sample': '%d envs x %d stepSimulation (%.1f s)' % (ne, steps, dt)},
                          'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return
    sim = BatchSim(db.scene, cfg, n)
    t0 = time.time()
    smp = db.reset(sim, rng, attempts=args.toc_attempts, settle_steps=50)
    db.start_fused(sim, smp)
    reset_s = time.time() - t0
    stream = torch.cuda.ExternalStream(sim.stream_ptr())
    dev = torch.device('cuda')
    act = torch.rand((K + W, n, 7), device=dev) * 2 - 1
    obs = torch.zeros((n, 24), device=dev); rew = torch.zeros(n, device=dev); done = torch.zeros(n, device=dev); info = torch.zeros((n, 4), device=dev)
    torch.cuda.synchronize()
    for i in range(W):
        sim.dressing_step_dev(act[i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
    torch.cuda.synchronize()
    clocks = ClockSampler(0); clocks.start()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sim.kernel_launches()
    with torch.cuda.stream(stream):
        a.record(stream)
    for i in range(K):
        sim.dressing_step_dev(act[W + i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
    with torch.cuda.stream(stream):
        b.record(stream)
    torch.cuda.synchronize()
    launches = sim.kernel_launches() - l0
    clk = clocks.stop()
    ms = a.elapsed_time(b) / K
    # per-kernel split in a separate pass (events around every launch, no graph)
    sim.profile_enable(True)
    for i in range(2):
        sim.dressing_step_dev(act[i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
    torch.cuda.synchronize()
    prof = sim.profile_get()
    sim.profile_enable(False)
    per_kernel = {k_: v[0] / 2 for k_, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    cloth_ms = prof['k_cloth'][0] / prof['k_cloth'][1]
    # e2e over the SAME env steps as `value`: the stored reset is replayed (same base poses, start angles, gown) and the batch is driven
    # with the same actions, W untimed + K timed steps from host buffers
    host_a = act.cpu().numpy().astype(np.float32)
    over_steps, over_settle = int(sim.overflow_count()), int(db.settle_overflow)       # (the flags are cleared when read)
    db.reset(sim, np.random.default_rng(0), sample=smp, settle_steps=50)
    db.start_fused(sim, smp)
    for i in range(W):
        sim.dressing_step_host(host_a[i])
    t0 = time.perf_counter()
    for i in range(K):
        sim.dressing_step_host(host_a[W + i])
    e2e = n * K / (time.perf_counter() - t0)
    over_steps = max(over_steps, int(sim.overflow_count()))
    ccnt = sim.cloth_get_contacts(1)[0]
    rcnt, it = sim.solver_stats()
    peak, peak_src = measured_peak()
    nn = db.cloth.n_nodes
    alg = n * 8 * nn * 6 * 4 * 2                     # x and v of every node read and written once per substep, 8 substeps per launch
    ach = alg / cloth_ms / 1e6
    traffic, traffic_src = ncu_traffic('k_cloth')
    info_h = info.cpu().numpy()
    print(json.dumps({'metric': 'env-steps/sec DressingPR2-v1 @batch%d' % n, 'value': n / ms * 1e3, 'unit': 'env-steps/s', 'n_gpus': 1, 'steps': K, 'warmup': W,
                      'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': {'workload': 'DressingPR2-v1, batch %d, fused step: 5 x (8 rigid substeps + 1 cloth launch), gown 3966 nodes / 11640 links, 5 position iterations, random actions' % n,
                                 'global_batch': n, 'l2': 'not flushed; the per-step working set (cloth state %d MB) exceeds L2' % (n * nn * 6 * 4 // 2 ** 20),
                                 'reset_s': reset_s, 'toc_attempts': args.toc_attempts, 'goals_reached_mean': float(np.mean(db.goals_reached)), 'base_unresolved': int(db.unresolved),
                                 'cloth_contacts_per_env': {'mean': float(ccnt.mean()), 'p99': float(np.percentile(ccnt, 99)), 'max': int(ccnt.max())},
                                 'rigid_contacts_per_env': {'mean': float(rcnt.mean()), 'max': int(rcnt.max())},
                                 'envs_over_budget': over_steps, 'envs_over_budget_during_settle': over_settle, 'e2e_same_steps_as_value': True,
                                 'sleeve_state_counts': {str(k_): int((info_h[:, 3] == k_).sum()) for k_ in (0, 1, 2, 3)},
                                 'cloth_force_mean_N': float(obs[:, 23].mean().item())},
                      'clocks': clk, 'e2e': {'value': e2e, 'unit': 'env-steps/s', 'h2d_bytes_per_step': n * 7 * 4, 'd2h_bytes_per_step': n * 30 * 4},
                      'gpu_launches': int(launches),
                      'roofline': {'bound': 'hbm', 'kernel': 'k_cloth', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': traffic, 'traffic_source': traffic_src,
                                   'peak_source': peak_src, 'kernel_ms_per_launch': cloth_ms, 'kernel_share_of_step': 5 * cloth_ms / ms,
                                   'algorithmic_bytes_per_launch': alg, 'per_kernel_ms_per_step': per_kernel,
                                   'note': 'algorithmic bytes = 190 KB per env and substep (SURVEY.md 8(d)); the kernel keeps the cloth in shared memory over the 8 substeps of a launch, so its DRAM traffic is ~1/8 of that'}}))


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Write each per-env output array (rows = envs) as `out_dir/<name>.npy` in float32.  Above DUMP_BYTES in all, the same
    fixed, seeded sample of envs (sorted) is taken from every array, so two runs with the same arguments stay comparable."""
    n = len(next(iter(arrays.values())))
    row_bytes = sum(4 * a[0].size for a in arrays.values())
    rows = np.arange(n)
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a[rows], dtype=np.float32))


def ncu_traffic(kernel):
    """DRAM bytes (read + write) of one launch of `kernel` from the newest committed `ncu --set full` summary
    (profiles/r*_ncu_<kernel>.csv, written by tools/ncu_summary.py); (None, None) if there is none."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_ncu_%s.csv' % kernel)))
    if not files:
        return None, None
    unit = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    tot = 0.0
    for r in csv.reader(open(files[-1])):
        if len(r) >= 4 and r[1] in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
            tot += float(r[3].replace(',', '')) * unit.get(r[2], 1.0)
    return (tot if tot > 0 else None), os.path.relpath(files[-1], ROOT)


def ncu_metrics(kernel, names):
    """selected metrics of the newest committed ncu summary of `kernel` ({} if there is none)"""
    import csv
    import glob
    files = sorted(f for f in glob.glob(os.path.join(ROOT, 'profiles', 'r*_ncu_%s.csv' % kernel)))
    out = {}
    if files:
        for r in csv.reader(open(files[-1])):
            if len(r) >= 4 and r[1] in names:
                try:
                    out[names[r[1]]] = float(r[3].replace(',', ''))
                except ValueError:
                    pass
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='agphys')
    ap.add_argument('--batch', type=int, default=BATCH_PER_GPU, help='envs per GPU')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--profile-kernels', type=int, default=1)
    ap.add_argument('--workload', default='feeding', choices=['feeding', 'bedbathing', 'dressing'], help="'bedbathing': BASELINE.json configs[2] (dense tool-skin contact), 'dressing': configs[3] (cloth); secondary lines")
    ap.add_argument('--press-mm', type=float, default=5.0, help='bedbathing: start depth of the wiping pad in the forearm (SURVEY.md 8(d) C2: 5 mm)')
    ap.add_argument('--action-scale', type=float, default=0.2, help='bedbathing: scale of the random actions (small actions keep the pad on the skin)')
    ap.add_argument('--toc-attempts', type=int, default=10, help='dressing / bedbathing: random base poses ranked per reset (the reference uses 50)')
    ap.add_argument('--sub-batches', type=int, default=int(os.environ.get('AG_SUB_BATCHES', '1')), help='independent sub-batches per GPU, each on its own stream')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='feeding: write obs / reward / done / info of the last timed step (rank 0) as DIR/<name>.npy, float32; '
                         'above 64 MB a fixed, seeded sample of envs')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.workload != 'feeding' or args.impl == 'reference'):
        ap.error('--dump-outputs covers the device path of the feeding workload only')
    if args.workload == 'bedbathing':
        return run_bedbathing(args)
    if args.workload == 'dressing':
        return run_dressing(args)
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the physics step has no CPU fallback')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from assistive_gym_b200 import capi
    from assistive_gym_b200.feeding_batch import FeedingBatch
    from assistive_gym_b200.sim import BatchSimGroup

    n = args.batch
    W = max(args.warmup, 3)
    K = args.steps
    fb = FeedingBatch()
    cfg = capi.default_config()
    G = max(1, args.sub_batches)
    sim = BatchSimGroup(fb.scene, cfg, n, groups=G, device=local_rank)
    # per-env seeds derive from the GLOBAL env id so results do not depend on the partition
    from assistive_gym_b200.sharding import sample_block, shard_range
    lo, hi = shard_range(rank, world, world * n)
    def reset_all():
        for g, sub in enumerate(sim.sims):
            rng = np.random.default_rng(1001 + rank * n + g)       # only used for IK random restarts
            sg = fb.reset(sub, rng, settle_steps=25, sample=sample_block(fb, lo + g * sim.m, lo + (g + 1) * sim.m))
            fb.start_fused(sub, sg, seed=1001 + rank * n + g * sim.m)
    reset_all()
    # `stream`: the bench's own stream; every step forks from it to the sub-batches' streams and joins back
    sub_streams = [torch.cuda.ExternalStream(p, device=local_rank) for p in sim.stream_ptrs()]
    stream = torch.cuda.Stream(device=local_rank)
    dev = torch.device('cuda', local_rank)
    gen = torch.Generator(device=dev)
    gen.manual_seed(rank)
    actions = torch.rand((W + K, n, 7), generator=gen, device=dev) * 2 - 1
    obs = torch.zeros((n, 25), device=dev)
    rew = torch.zeros(n, device=dev)
    done = torch.zeros(n, device=dev)
    info = torch.zeros((n, 4), device=dev)
    # the single collective of the path (SURVEY.md 8(e)): all-gather of the reward tensor, every step, double-buffered
    # and issued on a side stream so that gathering step i overlaps simulating step i+1
    rew_db = [torch.zeros(n, device=dev) for _ in range(2)] if world > 1 else None
    rew_all = [torch.zeros(world * n, device=dev) for _ in range(2)] if world > 1 else None
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)      # 256 MiB > 126 MB L2
    torch.cuda.synchronize()

    def gather_reward(i, src):
        """enqueue: copy the step's reward out of the way (sim stream), gather it on the side stream"""
        with torch.cuda.stream(stream):
            rew_db[i % 2].copy_(src, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        with torch.cuda.stream(side):
            side.wait_event(ev)
            dist.all_gather_into_tensor(rew_all[i % 2], rew_db[i % 2])

    def one_step(i):
        for ss in sub_streams:
            ss.wait_stream(stream)
        sim.feeding_step_dev(actions[i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
        for ss in sub_streams:
            stream.wait_stream(ss)
        if world > 1:
            gather_reward(i, rew)

    for i in range(W):
        one_step(i)
    torch.cuda.synchronize()
    launches0 = sim.kernel_launches()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = ClockSampler(local_rank)
    clocks.start()
    # ---- value: device-resident, CUDA-graph replay of the fused step (the path a learner uses), collective included
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for i in range(K):
        flush.fill_(float(i))                 # L2 flush between timed iterations (default stream)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            starts[i].record(stream)
        one_step(W + i)
        with torch.cuda.stream(stream):
            if world > 1:
                stream.wait_stream(side)      # the step is done when its reward is gathered
            stops[i].record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clk = clocks.stop()
    launches = sim.kernel_launches() - launches0
    elapsed_ms = float(sum(a.elapsed_time(b) for a, b in zip(starts, stops)))
    t = torch.tensor([elapsed_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = world * n * K / (elapsed_ms / 1000.0)
    rew_value_path = rew.detach().cpu().numpy().copy()        # reward of the last timed step (compared with the e2e path below)
    # the later passes step on in the same buffers: keep what the last timed step handed back
    last_step = {'obs': obs.cpu().numpy(), 'reward': rew_value_path, 'done': done.cpu().numpy(), 'info': info.cpu().numpy()} if args.dump_outputs else None
    # the same K steps timed back to back (no flush, no per-step sync): how much the pipeline overlap is worth
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        e0 = torch.cuda.Event(enable_timing=True); e0.record(stream)
    for i in range(K):
        one_step(W + i)
    with torch.cuda.stream(stream):
        if world > 1:
            stream.wait_stream(side)
        e1 = torch.cuda.Event(enable_timing=True); e1.record(stream)
    torch.cuda.synchronize()
    b2b_ms = e0.elapsed_time(e1) / K

    # ---- per-kernel split: a separate pass with direct launches and an event pair around every kernel
    prof = {}
    if args.profile_kernels:
        sim.profile_enable(True)
        for i in range(min(K, 5)):
            sim.feeding_step_dev(actions[W + i].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
            torch.cuda.synchronize()          # sub-batch after sub-batch: the per-kernel times are not overlapped
        torch.cuda.synchronize()
        prof = sim.profile_get()
        sim.profile_enable(False)
        sc_ = K / float(min(K, 5))
        prof = {k: (v[0] * sc_, int(round(v[1] * sc_))) for k, v in prof.items()}     # scaled to K steps (the code below divides by K)

    # ---- e2e: host buffers through the reference-facing call (H2D + D2H inside the timed region, collective included)
    # The SAME env steps as the device-resident measurement: the batch is reset to the same start state and driven with the same
    # actions (W untimed steps, then K timed ones), so the two numbers differ by the transfers and the per-step synchronisation only
    # (a batch stepped on with random actions drifts towards more contacts: steps 50+ cost ~10 % more than steps 5-25).
    host_actions = actions.detach().cpu().numpy().astype(np.float32)
    torch.cuda.synchronize()
    reset_all()
    for i in range(W):
        sim.feeding_step_host(host_actions[i])
    r_dev = torch.zeros(n, device=dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(K):
        o_h, r_h, d_h, i_h = sim.feeding_step_host(host_actions[W + i])
        if world > 1:
            with torch.cuda.stream(stream):
                r_dev.copy_(torch.from_numpy(r_h), non_blocking=True)
            gather_reward(i, r_dev)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * K / float(t.item())
    e2e_diff = float(np.max(np.abs(r_h - rew_value_path)))     # same start state, same actions: the two paths must agree
    overflow = sim.overflow_count()
    ccount, citers = sim.solver_stats()
    stream_bytes = 4 * sim.pgs_trips()[1]

    if rank == 0:
        peak, peak_src = measured_peak()
        roof = None
        if prof:
            top = max(prof.items(), key=lambda kv: kv[1][0])
            name, (ms, cnt) = top
            per_launch_ms = ms / max(cnt, 1)
            achieved = (n // G) * B_SUBSTEP / (per_launch_ms * 1e-3) / 1e9
            total_kernel_ms = sum(v[0] for v in prof.values())
            roof = {'bound': 'hbm', 'kernel': name, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                    'traffic': ncu_traffic(name)[0], 'traffic_source': ncu_traffic(name)[1], 'peak_source': peak_src, 'kernel_ms_per_launch': per_launch_ms,
                    'kernel_share_of_step': ms / total_kernel_ms if total_kernel_ms else None,
                    'step_frac': value * B_STEP / 1e9 / peak / world,
                    'per_kernel_ms_per_step': {k: v[0] / K for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])},
                    # what actually bounds the kernel: issue slots x lane utilisation (from the committed ncu summary)
                    'issue': ncu_metrics(name, {'smsp__thread_inst_executed_per_inst_executed.ratio': 'active_lanes_per_instruction',
                                                'smsp__issue_active.avg.pct_of_peak_sustained_active': 'issue_active_pct',
                                                'smsp__inst_executed.sum': 'warp_instructions_per_launch',
                                                'lts__t_sector_hit_rate.pct': 'l2_hit_pct'}),
                    # bytes the kernel really streams per launch: every env's row stream once per PGS sweep
                    'row_stream_gb_per_launch': float(stream_bytes.astype(np.float64).dot(citers.astype(np.float64)) / 1e9),
                    'note': 'the step is latency/issue bound, not HBM bound (SURVEY.md 8(d)); frac is reported per contract'}
        out = {'metric': METRIC, 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'warmup': W,
               'ms_per_step': elapsed_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
               'data': 'synthetic',
               'config': {'workload': 'FeedingJaco-v1, batch %d per GPU, 5 substeps/step, 50 PGS iters (early exit 1e-7), random actions' % n,
                          'global_batch': world * n, 'parallelism': 'env-sharded x%d' % world,
                          'l2': 'flushed between timed steps (256 MiB fill)', 'contact_budget': int(cfg.max_contacts),
                          'envs_over_contact_budget': overflow,
                          'contacts_per_env': {'mean': float(ccount.mean()), 'p50': float(np.percentile(ccount, 50)), 'p99': float(np.percentile(ccount, 99)), 'max': int(ccount.max())},
                          'pgs_iters_per_env': {'mean': float(citers.mean()), 'p50': float(np.percentile(citers, 50)), 'p99': float(np.percentile(citers, 99)), 'max': int(citers.max())},
                          'pgs_lanes_per_env': 8,
                          'collective': 'all_gather(reward) every step, double-buffered on a side stream (inside both timed regions)' if world > 1 else 'none',
                          'ms_per_step_back_to_back': b2b_ms,
                          'e2e_same_steps_as_value': True, 'e2e_reward_max_abs_diff_vs_value_path': e2e_diff},
               'clocks': clk,
               'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': n * 7 * 4, 'd2h_bytes_per_step': n * 31 * 4},
               'gpu_launches': int(launches), 'roofline': roof}
        if not args.no_cpu:
            cores = usable_cores()
            ne, ns = max(32 * cores, 64), 40                  # ~20 k env-steps = 15-25 s of CPU work spread over the threads
            v, tsec = cpu_oracle_rate(fb, ne, ns, cores)
            v1, t1 = cpu_oracle_rate(fb, 64, ns, 1)
            out['cpu_baseline'] = {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
                                   'sample': '%d envs x %d env-steps (%.2f s wall, %.0f core-seconds), CPU restatement (PyBullet unavailable), %d threads (affinity / cgroup quota)' % (ne, ns, tsec, tsec * cores, cores),
                                   'one_thread': {'value': v1, 'cores': 1, 'sample': '64 envs x %d env-steps (%.2f s)' % (ns, t1)}}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
