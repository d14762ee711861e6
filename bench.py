#!/usr/bin/env python
"""Benchmark of the NES generation hot path (BASELINE.json: generations/s and policy-evals/s, pop 64k).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--pop 65536] [--hidden 256] [--tape-len 256] [--precision fp32|f16|f16x3] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, NCCL)

A "step" is one NES generation (natural_es.py:62-96) over synthetic inputs: sample eps for the whole
population, batched policy forward over population x tape, centered ranks, fitness x noise reduction,
(1-wd)/Adam/step.  The population is fixed as GPUs are added (strong scaling, as BASELINE.json quotes
the metric "at pop 64k, 1/2/4/8 B200").  Prints ONE JSON line on rank 0.

  value        policy-evals/s of the headline workload with everything resident in HBM (generations/s = value / pop)
  e2e          same metric through the host-buffer API (tape H2D, theta+fitness D2H inside the timed region)
  roofline     the dominant kernel (fused sample+forward+fitness).  eps is regenerated, not stored, so the kernel moves
               ~1e-5 of the materialised-noise bytes of SURVEY §8d and the binding roof is the tensor pipe:
               frac = F_fwd / kernel time / measured bf16 peak (F_fwd = 2 n T (d0 H + H^2 + H A), the algorithmic flops;
               f16x3 issues three MMAs per k-step — `tensor_issued_frac`).  The §8d HBM contract (8 n P algorithmic
               bytes per launch) is carried as `hbm_contract`.
  configs      every configuration north_star / BASELINE.json names, measured by this same run: NES at pop 4 096 (2x64),
               16 384 and 65 536 (2x256), CMA-ES generations/s at n=1024 / lambda=256 and the rank-mu update at n=4096 /
               lambda=1024 (sharded over the N GPUs), each with its own roofline and cpu_baseline
  parity       self-check of this run: N > 1: fitness of generation 0 against a 1-GPU evaluation of the same members (bit
               equality) and the update against the 1-GPU update (1e-5); N = 1: tensor-core fitness against the fp32 path
  cpu_baseline the reference's own natural_es.train() run verbatim (oracle/_ref, kind "reference") on the host cores,
               bounded sample, with the numpy port of the same generation beside it (N=1, rank 0)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
# the tree may be read-only where the benchmark runs: no bytecode caches beside the sources, here or in the CPU legs
sys.dont_write_bytecode = True
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'

import numpy as np  # noqa: E402

EMIT = print


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--pop', type=int, default=65536)
    ap.add_argument('--hidden', type=int, default=256)
    ap.add_argument('--state-dim', type=int, default=24)
    ap.add_argument('--action-dim', type=int, default=4)
    ap.add_argument('--tape-len', type=int, default=256)
    ap.add_argument('--precision', default=os.environ.get('DES_BENCH_PRECISION', 'f16x3'),
                    help='policy-forward arithmetic: f16x3 (tensor cores, fp32-grade, default), f16 (tensor cores, fp16 operands), fp32 (CUDA cores)')
    ap.add_argument('--no-other-modes', action='store_true', help='skip the extra context measurements (other precision, closed loop)')
    ap.add_argument('--no-configs', action='store_true', help='skip the secondary configurations (pop 4k/16k, CMA)')
    ap.add_argument('--cpu-sample', type=int, default=0, help='members per CPU-baseline step (0 = auto)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed generation of the headline workload computed (fitness, theta, update, '
                         'gradient partial sum) as DIR/<name>.npy, float32; inputs are seeded, so runs with the same '
                         'arguments compare output for output')
    return ap.parse_args()


def workload_name(d0, H, A, T, pop):
    return 'nes_synth_tape d0=%d H=%d A=%d T=%d pop=%d (SURVEY 8d; strong scaling)' % (d0, H, A, T, pop)


def peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), float(d.get('bf16_tflops', 0.0)), float(d.get('bf16_tflops_sustained', 0.0)), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


FP32_FFMA_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FFMA/clk x 1.965 GHz = 74.4 (nominal CUDA-core peak)


# --------------------------------------------------------------------------------------------------------
# CPU legs (their own processes: no torch / CUDA state in them)
# --------------------------------------------------------------------------------------------------------
def _run_json(cmd, timeout):
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError('%s failed: %s' % (cmd[2], r.stderr[-1500:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def cpu_port(d0, H, A, T, pop, steps, warmup, target_seconds, sample=0):
    """The numpy port of the generation (oracle/cpu_baseline.py), one worker process per core."""
    return _run_json([sys.executable, '-m', 'oracle.cpu_baseline', '--d0', str(d0), '--hidden', str(H), '--action-dim', str(A),
                      '--tape-len', str(T), '--pop', str(pop), '--steps', str(steps), '--warmup', str(warmup),
                      '--sample', str(sample), '--target-seconds', str(target_seconds)], 900)


def cpu_reference(d0, H, A, T, pop, gens, skip=0):
    """The reference's natural_es.train() verbatim (oracle/ref_cpu_baseline.py over oracle/_ref)."""
    return _run_json([sys.executable, '-m', 'oracle.ref_cpu_baseline', '--d0', str(d0), '--hidden', str(H), '--action-dim', str(A),
                      '--tape-len', str(T), '--pop', str(pop), '--gens', str(gens), '--skip', str(skip)], 1800)


def have_reference():
    return os.path.exists(os.path.join(REPO, 'oracle', '_ref', 'natural_es.py'))


def cpu_baseline_for(d0, H, A, T, pop, ref_pop=0, port_seconds=4.0):
    """cpu_baseline object of one NES configuration: the verbatim reference where oracle/_ref exists (value), the numpy
    port beside it.  Never raises: the CPU leg must not take the GPU line down with it."""
    out = {'value': None, 'unit': 'policy-evals/s', 'cores': None, 'kind': 'port', 'sample': None}
    try:
        r = cpu_port(d0, H, A, T, pop, 2, 1, port_seconds)
        out.update(value=r['evals_per_sec'], cores=r['cores'], sample=r['sample'])
        out['port'] = {'value': r['evals_per_sec'], 'cores': r['cores'], 'sample': r['sample'],
                       'note': 'numpy port: per-member BLAS forward over the whole tape, one process per core — faster than the reference itself'}
    except Exception as e:
        out['sample'] = 'port failed: %s' % str(e)[:200]
    if have_reference():
        try:
            cores = out['cores'] or os.cpu_count() or 8
            rp = ref_pop or max(16, 8 * max(1, cores - 1))
            r = cpu_reference(d0, H, A, T, rp, 2)
            out.update(value=r['evals_per_sec'], cores=r['cores'], kind='reference', sample=r['sample'],
                       seconds_per_generation_at_sample=r['seconds_per_generation'])
        except Exception as e:
            out['reference_error'] = str(e)[:200]
    return out


def cma_cpu_baseline(n, lam):
    """fp64 numpy restatement of the rank-mu update (BLAS, all host threads): pycma is unavailable."""
    try:
        from oracle import cma_oracle as co
        rs = np.random.RandomState(0)
        Y = rs.randn(lam, n)
        w = rs.rand(lam)
        C = np.eye(n)
        pc = rs.randn(n)
        co.cov_update(C, co.rank_mu_delta(Y, w), pc, 0.001, 0.009, w.sum())
        t0 = time.perf_counter()
        reps = 3 if n <= 1024 else 1
        for _ in range(reps):
            co.cov_update(C, co.rank_mu_delta(Y, w), pc, 0.001, 0.009, w.sum())
        sec = (time.perf_counter() - t0) / reps
        return {'value': 1.0 / sec, 'unit': 'updates/s', 'cores': os.cpu_count(), 'kind': 'port',
                'sample': 'fp64 numpy restatement (BLAS Y^T diag(w) Y + covariance update), %d repetition(s); pycma unavailable' % reps}
    except Exception as e:
        return {'value': None, 'unit': 'updates/s', 'cores': None, 'kind': 'port', 'sample': 'failed: %s' % str(e)[:200]}


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the path (natural_es.train verbatim from oracle/_ref),
    all host cores, a bounded sample of the population per step; rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    d0, H, A, T = a.state_dim, a.hidden, a.action_dim, a.tape_len
    port = None
    try:
        port = cpu_port(d0, H, A, T, a.pop, 2, 1, 4.0)
    except Exception as e:
        port = {'error': str(e)[:200]}
    if have_reference():
        cores = (port or {}).get('cores') or os.cpu_count() or 8
        sample = a.cpu_sample or max(16, 8 * max(1, cores - 1))
        r = cpu_reference(d0, H, A, T, sample, a.steps + a.warmup, skip=a.warmup)
        value, sec, kind, cores, desc = r['evals_per_sec'], r['seconds_per_generation'], 'reference', r['cores'], r['sample']
    else:       # oracle/_ref did not travel: fall back to the port, and say so
        r = cpu_port(d0, H, A, T, a.pop, a.steps, a.warmup, 150.0 / max(1, a.steps + a.warmup + 2), a.cpu_sample)
        value, sec, kind, cores, desc = r['evals_per_sec'], r['seconds_per_step'], 'port', r['cores'], r['sample']
        sample = r['sample_members']
    line = {
        'impl': 'reference', 'metric': 'nes_policy_evals_per_sec', 'value': value, 'unit': 'policy-evals/s',
        'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': sec * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64/f32 (numpy + torch CPU)',
        'data': 'synthetic', 'generations_per_sec': value / a.pop,
        'config': {'workload': workload_name(d0, H, A, T, a.pop), 'sample_members_per_step': sample,
                   'note': 'ms_per_step is one generation over the SAMPLE (%d members), not over the population; value = '
                           'sample / seconds, generations_per_sec = value / pop' % sample},
        'cpu_baseline': {'value': value, 'unit': 'policy-evals/s', 'cores': cores, 'kind': kind, 'sample': desc,
                         'port': port},
        'e2e': {'value': value, 'unit': 'policy-evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    EMIT(json.dumps(line))


# --------------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '100'], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower() == 'active':
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(np.max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


DUMP_MAX_ELEMS = 3 << 20      # per array: 12 MiB of float32, so the four dumped arrays stay under 64 MB


def dump_outputs(outdir, arrays):
    """Write each device array as outdir/<name>.npy; one larger than DUMP_MAX_ELEMS is cut to a fixed, seeded sample."""
    os.makedirs(outdir, exist_ok=True)
    for name, t in arrays.items():
        x = t.detach().cpu().numpy().astype(np.float32).reshape(-1)
        if x.size > DUMP_MAX_ELEMS:
            x = x[np.sort(np.random.RandomState(0).choice(x.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(outdir, name + '.npy'), x)


def build_hash():
    """Identity of the library the numbers were taken on (keys profiles/roofline_traffic.json)."""
    import hashlib
    try:
        from distributedes_b200 import _lib
        return hashlib.sha256(open(_lib.LIB_PATH, 'rb').read()).hexdigest()[:12]
    except Exception:
        return None


def run_ours(a):
    import torch
    import torch.distributed as dist
    from distributedes_b200.envs import TapeEnv                 # synthetic tape (SURVEY 8d), RandomState(1234)
    from distributedes_b200.model import StandardFCNet          # nn.Linear-style init, RandomState(0)
    from distributedes_b200.engine import NESEngine
    from distributedes_b200 import _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)')
    _lib.load()
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if world != a.gpus and rank == 0:
        print('bench.py: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE' % (a.gpus, world), file=sys.stderr)

    hbm_peak, bf16_peak, bf16_sustained, peak_kind = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """K steps, each bracketed by CUDA events on the launching stream; L2 flushed between steps
        (outside the events).  Returns (sum of step ms, list)."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for s, e in ev:
            flush.zero_()
            s.record()
            fn()
            e.record()
        barrier()
        ms = [s.elapsed_time(e) for s, e in ev]
        return float(np.sum(ms)), ms

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    traffic_table = {}
    tp = os.path.join(REPO, 'profiles', 'roofline_traffic.json')
    if os.path.exists(tp):
        try:
            traffic_table = json.load(open(tp))
        except Exception:
            traffic_table = {}

    def make_engine(d0, H, A, T, N, precision):
        env = TapeEnv(d0, A, T)
        theta0 = StandardFCNet(d0, A, H, seed=0).get_weight()
        eng = NESEngine(state_dim=d0, hidden=H, action_dim=A, pop_size=N, theta0=theta0, obs=env.obs, target=env.target,
                        sigma=0.1, learning_rate=0.1, weight_decay=0.005, clip=1.0, seed=0, precision=precision,
                        device=dev, use_graph=not a.no_graph)
        return eng, env, theta0

    def measure_nes(d0, H, A, T, N, precision, steps, warmup, outputs=None):
        """Device-resident generations of one configuration + its dominant kernel alone -> (dict, engine, env).
        `outputs`, if given, receives copies of what the last timed generation left for its caller."""
        eng, env, _ = make_engine(d0, H, A, T, N, precision)
        P = eng.P
        for _ in range(max(warmup, 3)):
            eng.generation()
        total_ms, _ = timed(eng.generation, steps)
        ms_per_step = max_over_ranks(total_ms) / steps
        if outputs is not None:
            outputs.update(fitness=eng.fitness_all.clone(), theta=eng.theta.clone(), update=eng.update.clone(),
                           partial=eng.partial.clone())

        def eval_only():
            eng.k.nes_eval(eng.theta, eng.obs, eng.target, hidden=H, sigma=eng.sigma, clip=eng.clip, seed=eng.seed,
                           state=eng.state, member_offset=eng.offset, n_local=eng.n_local, precision=eng.precision,
                           out=eng.fitness_shard_out, workspace=eng.eval_ws)
        for _ in range(2):
            eval_only()
        # The kernel is timed INSIDE eager generations (events around the launch, the rest of the generation behind it): the
        # host runs ahead during the long kernels, so no launch latency is billed to the kernel, and the kernel runs under the
        # power / clock conditions of the step it is a share of.  (Timed in a loop of its own — nothing but this kernel,
        # back to back — the same launch takes ~5 % longer: the GPU sits at its power cap.)
        def step_with_eval_events(s_ev, e_ev):
            if eng.world > 1 and eng.comm is None:
                eng.fitness_all.zero_()
            s_ev.record()
            eval_only()
            e_ev.record()
            eng._gather_fitness()
            eng.rank_and_reduce()
            eng.apply()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for s_ev, e_ev in evs:
            flush.zero_()
            step_with_eval_events(s_ev, e_ev)
        barrier()
        ev_ms = float(np.sum([s_ev.elapsed_time(e_ev) for s_ev, e_ev in evs]))
        ev_ms = max_over_ranks(ev_ms) / steps
        alg_bytes = 8.0 * eng.n_local * P                                  # write eps once + read it in the forward
        fwd_flops = 2.0 * eng.n_local * T * (d0 * H + H * H + H * A)
        tf = fwd_flops / (ev_ms * 1e-3) / 1e12
        gbs = alg_bytes / (ev_ms * 1e-3) / 1e9
        traffic = traffic_table.get('%s_H%d_n%d' % (precision, H, eng.n_local))
        tensor_path = precision in ('f16', 'f16x3')
        if tensor_path:
            roofline = {'kernel': 'des_nes_eval[%s]' % precision, 'bound': 'tensor', 'achieved': tf, 'peak': bf16_peak,
                        'unit': 'TFLOP/s', 'frac': tf / bf16_peak if bf16_peak else None,
                        'peak_kind': 'of %s bf16 burst (cuBLAS)' % peak_kind,
                        'frac_of_sustained_peak': tf / bf16_sustained if bf16_sustained else None,
                        'algorithmic_flops_per_launch': fwd_flops,
                        'tensor_issued_frac': (3.0 if precision == 'f16x3' else 1.0) * tf / bf16_peak if bf16_peak else None}
        else:
            roofline = {'kernel': 'des_nes_eval[fp32]', 'bound': 'fp32 CUDA cores', 'achieved': tf, 'peak': FP32_FFMA_TFLOPS,
                        'unit': 'TFLOP/s', 'frac': tf / FP32_FFMA_TFLOPS, 'peak_kind': 'nominal 148 x 128 FFMA/clk x 1.965 GHz',
                        'algorithmic_flops_per_launch': fwd_flops}
        roofline.update({
            'traffic': traffic, 'kernel_ms': ev_ms, 'kernel_share_of_step': ev_ms / ms_per_step,
            'hbm_contract': {'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': gbs / hbm_peak,
                             'algorithmic_bytes_per_launch': alg_bytes,
                             'note': 'SURVEY 8d materialised-noise contract (8 n P bytes per launch); eps is regenerated '
                                     'in the kernel, so this is an effective figure and may exceed the HBM peak'},
            'note': 'binding roof = tensor pipe: measured DRAM traffic (`traffic`, ncu, profiles/) is ~1e-5 of the HBM '
                    'contract bytes; the kernel is limited by instruction issue / XU(MUFU) / tensor hand-overs (profiles/README.md)'})
        res = {'workload': workload_name(d0, H, A, T, N), 'pop': N, 'hidden': H, 'param_count': P, 'precision': precision,
               'n_gpus': world, 'members_per_gpu': eng.n_local, 'ms_per_step': ms_per_step,
               'value': N / (ms_per_step * 1e-3), 'unit': 'policy-evals/s', 'generations_per_sec': 1e3 / ms_per_step,
               'cuda_graph': bool(eng._use_graph), 'roofline': roofline}
        return res, eng, env

    # ================================ headline workload ================================
    d0, H, A, T, N = a.state_dim, a.hidden, a.action_dim, a.tape_len, a.pop
    sampler = ClockSampler(local_rank) if rank == 0 else None
    outputs = {} if a.dump_outputs else None
    main, eng, env = measure_nes(d0, H, A, T, N, a.precision, a.steps, a.warmup, outputs)
    clocks = sampler.stop() if sampler else None
    if outputs and rank == 0:
        dump_outputs(a.dump_outputs, outputs)
    P = eng.P
    ms_per_step, value, roofline = main['ms_per_step'], main['value'], main['roofline']

    # ---- end to end through the host-buffer API ----
    obs_h = torch.from_numpy(env.obs).pin_memory()
    tgt_h = torch.from_numpy(env.target).pin_memory()
    theta_h = torch.empty(P, dtype=torch.float32).pin_memory()
    fit_h = torch.empty(N, dtype=torch.float32).pin_memory()

    def e2e_step():
        eng.generation_host(obs_h, tgt_h, theta_out_host=theta_h, fitness_out_host=fit_h)
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0) / a.steps
    e2e = {'value': N / e2e_s, 'unit': 'policy-evals/s', 'ms_per_step': e2e_s * 1e3,
           'h2d_bytes_per_step': int(obs_h.numel() * 4 + tgt_h.numel() * 4),
           'd2h_bytes_per_step': int(theta_h.numel() * 4 + fit_h.numel() * 4),
           'api': 'NESEngine.generation_host (pinned host tape in, theta + fitness out, synchronous)'}

    # ---- parity self-check of this run ----
    parity = None
    try:
        parity = parity_check(torch, dist, eng, world, dev)
    except Exception as e:
        parity = {'error': str(e)[:300]}
    del eng

    # ================================ every other north_star configuration ================================
    configs = []
    if not a.no_configs:
        sub_steps = max(3, a.steps // 2)
        for (cd0, cH, cA, cT, cN, tag) in [(24, 64, 4, 256, 4096, 'BASELINE configs[1]'),
                                            (24, 256, 4, 256, 16384, 'north_star pop 16k'),
                                            (d0, H, A, T, N, 'BASELINE configs[3] (headline)')]:
            try:
                if (cd0, cH, cA, cT, cN) == (d0, H, A, T, N):
                    r = dict(main)
                else:
                    r, e2, _ = measure_nes(cd0, cH, cA, cT, cN, a.precision, sub_steps, 3)
                    del e2
                r['config_of'] = tag
                if rank == 0 and world == 1 and not a.no_cpu_baseline:
                    r['cpu_baseline'] = cpu_baseline_for(cd0, cH, cA, cT, cN, port_seconds=3.0)
                configs.append(r)
            except Exception as e:
                configs.append({'workload': workload_name(cd0, cH, cA, cT, cN), 'config_of': tag, 'error': str(e)[:300]})
        try:
            configs.extend(measure_cma(torch, dist, timed, max_over_ranks, world, rank, dev, hbm_peak,
                                       not a.no_cpu_baseline))
        except Exception as e:
            configs.append({'workload': 'cma', 'error': str(e)[:300]})

    # ---- the other tensor-core mode and the closed-loop engine, device-resident, for context (not the headline) ----
    other = None
    if not a.no_other_modes and a.precision in ('f16', 'f16x3'):
        oprec = 'f16' if a.precision == 'f16x3' else 'f16x3'
        try:
            r2, eng2, _ = measure_nes(d0, H, A, T, N, oprec, max(3, a.steps // 2), 3)
            del eng2
            other = {oprec: {'ms_per_step': r2['ms_per_step'], 'value': r2['value'], 'unit': 'policy-evals/s',
                             'kernel_ms': r2['roofline']['kernel_ms'],
                             'note': 'fp16-rounded operands (11 significant bits, like TF32): fitness within 4e-3 of the oracle'
                             if oprec == 'f16' else 'hi/lo split operands: fitness within 3e-5 of the oracle'}}
        except Exception as e:
            other = {oprec: {'error': str(e)[:200]}}
    closed = None
    if world == 1 and not a.no_other_modes:
        try:
            from distributedes_b200.engine import RolloutEngine
            cN, cH = min(N, 65536), 64
            ceng = RolloutEngine(hidden=cH, pop_size=cN, theta0=StandardFCNet(3, 1, cH, seed=0).get_weight(), sigma=0.1,
                                 learning_rate=0.1, seed=0, device=dev)
            for _ in range(3):
                ceng.generation()
            c_ms, _ = timed(ceng.generation, max(3, a.steps // 2))
            c_ms /= max(3, a.steps // 2)
            closed = {'workload': 'Pendulum-v0 closed loop: pop %d, 2x%d MLP, 10 episodes x 200 steps per member' % (cN, cH),
                      'ms_per_step': c_ms, 'env_steps_per_sec': cN * 10 * 200 / (c_ms * 1e-3),
                      'policy_evals_per_sec': cN / (c_ms * 1e-3),
                      'fp32_tflops': 2.0 * (3 * cH + cH * cH + cH) * cN * 2000 / (c_ms * 1e-3) / 1e12}
            del ceng
        except Exception as e:
            closed = {'error': str(e)[:200]}

    # ---- CPU baseline of the headline workload (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = next((c.get('cpu_baseline') for c in configs if c.get('config_of', '').endswith('(headline)')), None)
        if cpu is None:
            cpu = cpu_baseline_for(d0, H, A, T, N)

    if rank == 0:
        # memset + eval, rank (2 kernels; 5 on the bucketed path for N > 8192), grad_chunk, grad_reduce, apply, state_advance
        launches_per_step = 5 + (5 if N > 8192 else 2)
        line = {
            'metric': 'nes_policy_evals_per_sec', 'value': value, 'unit': 'policy-evals/s', 'n_gpus': world,
            'steps': a.steps, 'warmup': max(a.warmup, 3), 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': {'fp32': 'f32', 'f16': 'f16 (fp16 operands, f32 accumulate)',
                                                           'f16x3': 'f16x3 (split-fp16 operands ~ f32, f32 accumulate)'}[a.precision],
            'data': 'synthetic', 'generations_per_sec': 1e3 / ms_per_step,
            'forwards_per_sec': value * T,
            'config': {'workload': workload_name(d0, H, A, T, N), 'precision': a.precision, 'param_count': P,
                       'members_per_gpu': main['members_per_gpu'], 'cuda_graph': main['cuda_graph'],
                       'theta0': 'distributedes_b200.model.StandardFCNet(seed=0): nn.Linear-style U(+-1/sqrt(fan_in)) from numpy '
                                 'RandomState(0) — the same distribution as SURVEY 8d\'s torch.manual_seed(0) init, not the same draws',
                       'noise': 'Philox4x32-7 + Box-Muller, counter = (j/4, member, generation, stream)',
                       'l2': 'flushed: 256 MiB memset between steps, outside the per-step CUDA events',
                       'parallelism': 'population sharded over %d GPU(s); all-reduce fitness[N] + all-reduce partial[P]' % world,
                       'library_sha256_12': build_hash()},
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches_per_step * a.steps,
            'roofline': roofline, 'cpu_baseline': cpu, 'parity': parity, 'configs': configs,
            'other_modes': other, 'closed_loop': closed,
        }
        EMIT(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def parity_check(torch, dist, eng, world, dev):
    """Self-check on the engine's own inputs.  N > 1: a fresh generation 0 evaluated (a) sharded + all-reduced, (b) on this
    GPU alone over all members — fitness must be bit-equal; update of the sharded generation against the update formed
    on one GPU from the same fitness — within 1e-5 in both norms (SURVEY 8d iii).  N = 1: tensor-core fitness against the
    fp32 CUDA-core path on 512 members."""
    k = eng.k
    N, H = eng.N, eng.H
    if world == 1:
        n = min(512, N)
        kw = dict(hidden=H, sigma=eng.sigma, clip=eng.clip, seed=eng.seed, generation=0, member_offset=0, n_local=n)
        ref = k.nes_eval(eng.theta, eng.obs, eng.target, precision='fp32', **kw)
        got = k.nes_eval(eng.theta, eng.obs, eng.target, precision=eng.precision, **kw)
        rel = float(((got - ref).abs() / ref.abs()).max())
        bound = {'fp32': 0.0, 'f16': 4e-3, 'f16x3': 3e-5}[eng.precision]
        return {'kind': 'tensor-core fitness vs fp32 CUDA-core path, %d members, same theta/noise' % n,
                'fitness_max_rel': rel, 'bound': bound, 'ok': bool(rel <= bound)}
    import torch as th
    from distributedes_b200.engine import NESEngine
    theta0 = eng.theta.detach().cpu().numpy()
    obs, target = eng.obs_raw.cpu().numpy(), eng.target.cpu().numpy()
    kw = dict(state_dim=eng.d0, hidden=H, action_dim=eng.A, pop_size=N, theta0=theta0, obs=obs, target=target,
              sigma=eng.sigma, learning_rate=eng.lr, weight_decay=eng.wd, clip=eng.clip, seed=eng.seed,
              precision=eng.precision, device=dev, use_graph=False)
    sharded = NESEngine(**kw)
    sharded.generation()                                            # generation 0, sharded over the ranks
    # (b) this GPU alone, all members, same generation counter
    full_fit = k.nes_eval(th.from_numpy(theta0).to(dev), sharded.obs, sharded.target, hidden=H, sigma=eng.sigma,
                          clip=eng.clip, seed=eng.seed, generation=0, member_offset=0, n_local=N, precision=eng.precision)
    fit_equal = bool(th.equal(full_fit, sharded.fitness_all))
    shaped = k.centered_rank(sharded.fitness_all, 0, N)
    partial = k.nes_grad_partial(shaped, sharded.P, seed=eng.seed, generation=0, member_offset=0)
    theta1 = th.from_numpy(theta0.copy()).to(dev)
    m1 = th.zeros(sharded.P, dtype=th.float64, device=dev)
    v1 = th.zeros_like(m1)
    upd1 = th.zeros(sharded.P, dtype=th.float32, device=dev)
    st = k.new_state(dev, 0)
    k.nes_apply(theta1, m1, v1, partial, N, st, sigma=eng.sigma, learning_rate=eng.lr, weight_decay=eng.wd,
                beta1=eng.beta1, beta2=eng.beta2, epsilon=eng.epsilon, update_out=upd1)
    g_s, g_1 = sharded.partial.double(), partial.double()
    g_rel = float((g_s - g_1).norm() / g_1.norm())
    g_max = float((g_s - g_1).abs().max() / g_1.abs().max())
    # Adam's first step is ~sign(g): compare the update where |g| is not at the rounding floor (tests/test_gpu_ops.py)
    keep = g_1.abs() > 1e-4 * g_1.abs().max()
    u_rel = float((sharded.update.double() - upd1.double())[keep].norm() / upd1.double()[keep].norm())
    res = {'kind': 'generation 0 sharded over %d GPUs vs the same members on one GPU' % world,
           'fitness_bit_equal': fit_equal, 'partial_rel_l2': g_rel, 'partial_rel_max': g_max, 'update_rel_l2': u_rel,
           'bound': 1e-5, 'ok': bool(fit_equal and g_rel <= 1e-5 and g_max <= 1e-5 and u_rel <= 1e-5)}
    flags = th.tensor([1.0 if res['ok'] else 0.0], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    res['ok_all_ranks'] = bool(flags.item() == 1.0)
    return res



def cma_roofline(n, lam, lam_local, world):
    """Roofline of the rank-mu update's two kernels, timed separately on this rank (CUDA events): the SYRK
    (tensor pipe when ops picks the split-fp16 tcgen05 path, fp32 CUDA cores below ops.CMA_TC_MIN_N) and the
    HBM-bound covariance blend.  Flops counted as 2 lambda n^2 (the full square; the kernels compute the upper triangle)."""
    import torch
    from distributedes_b200 import ops
    hbm_peak, bf16_peak, _, peak_kind = peaks()
    dev = torch.device('cuda', torch.cuda.current_device())
    Y = torch.randn(lam_local, n, device=dev); w = torch.rand(lam_local, device=dev)
    Cm = torch.eye(n, device=dev); pc = torch.randn(n, device=dev)
    dC = ops.cma_rank_mu(Y, w)
    for _ in range(3):
        ops.cma_rank_mu(Y, w, out=dC); ops.cma_cov_apply(Cm, dC, pc, decay=0.99, c1=0.001, cmu=0.009)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    for _ in range(10):
        ops.cma_rank_mu(Y, w, out=dC)
    ev[1].record()
    for _ in range(10):
        ops.cma_cov_apply(Cm, dC, pc, decay=0.99, c1=0.001, cmu=0.009)
    ev[2].record()
    torch.cuda.synchronize()
    t_mu, t_cov = ev[0].elapsed_time(ev[1]) / 10, ev[1].elapsed_time(ev[2]) / 10
    tc = n >= ops.CMA_TC_MIN_N
    tf = 2.0 * lam_local * n * n / (t_mu * 1e-3) / 1e12
    peak = bf16_peak if tc else FP32_FFMA_TFLOPS
    gbs = 12.0 * n * n / (t_cov * 1e-3) / 1e9
    return {'kernel': 'des_cma_rank_mu_tc (split-fp16 tcgen05 SYRK, TMA-fed)' if tc else 'des_cma_rank_mu (fp32 FFMA)',
            'bound': 'tensor' if tc else 'fp32 CUDA cores', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s',
            'frac': tf / peak if peak else None,
            'peak_kind': ('of %s bf16 burst (cuBLAS)' % peak_kind) if tc else 'nominal 148 x 128 FFMA/clk x 1.965 GHz',
            'tensor_issued_frac': (3.0 * 0.5 * (1 + 256.0 / n) * tf / peak) if (tc and peak) else None,
            'kernel_ms': t_mu, 'members_this_rank': lam_local, 'n_gpus': world,
            'note': 'flops counted as 2 lambda n^2; the kernel issues three MMAs per k-step over the 128x256 tiles that touch the upper triangle',
            'cov_apply': {'bound': 'hbm', 'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': gbs / hbm_peak if hbm_peak else None,
                          'kernel_ms': t_cov, 'algorithmic_bytes': 12.0 * n * n}}


def measure_cma(torch, dist, timed, max_over_ranks, world, rank, dev, hbm_peak, with_cpu):
    """CMA-ES lines: (a) BASELINE configs[2]: whole generations (ask, evaluate sphere, tell) at n=1024, lambda=256 on this
    GPU; (b) configs[4]: the rank-mu covariance update at n=4096, lambda=1024 — shard partial on each GPU, all-reduce of
    the packed upper-triangular tiles, covariance update — max over ranks."""
    from distributedes_b200 import ops
    from distributedes_b200.cma_es import CMAEvolutionStrategy, cma_constants
    out = []
    # ---- (a) generations/s at n = 1024, lambda = 256 (single GPU: every rank runs the same replica; rank 0 reports)
    n, lam = 1024, 256
    x0 = np.random.RandomState(0).randn(n)
    es = CMAEvolutionStrategy(x0, 1.0, lam, seed=0, device=dev, process_group=None) if world == 1 else None
    if es is not None:
        def cma_generation():
            X = es.ask()
            cost = (X.double() ** 2).sum(1)
            es.tell(X, cost)
        for _ in range(3):
            cma_generation()
        ms, _ = timed(cma_generation, 5)
        gen_ms = ms / 5
        Y = torch.randn(lam, n, device=dev)
        w = torch.rand(lam, device=dev)
        Cm = torch.eye(n, device=dev)
        pc = torch.randn(n, device=dev)
        dC = ops.cma_rank_mu(Y, w)

        def upd():
            ops.cma_rank_mu(Y, w, out=dC)
            ops.cma_cov_apply(Cm, dC, pc, decay=0.99, c1=0.001, cmu=0.009)
        for _ in range(3):
            upd()
        ms, _ = timed(upd, 10)
        upd_ms = ms / 10
        flops = 2.0 * lam * n * n
        r = {'workload': 'cma_es sphere n=%d lambda=%d (BASELINE configs[2])' % (n, lam), 'config_of': 'BASELINE configs[2]',
             'n_gpus': 1, 'generation_ms': gen_ms, 'generations_per_sec': 1e3 / gen_ms,
             'rank_mu_update_ms': upd_ms, 'updates_per_sec': 1e3 / upd_ms,
             'roofline': cma_roofline(n, lam, lam, 1),
             'parity': 'oracle/cma_oracle.py (tutorial restatement) pinned by tests/test_cma_pinning.py: constants by hand from Hansen 2016, pycma banner (mu_w, w_1) values, one generation in n=3 by literal arithmetic; pycma itself is absent; kernels vs the restatement <= 1e-5 (tests/test_gpu_cma.py)'}
        if with_cpu and rank == 0:
            r['cpu_baseline'] = cma_cpu_baseline(n, lam)
        out.append(r)
    # ---- (b) rank-mu update at n = 4096, lambda = 1024 sharded over the GPUs
    n, lam = 4096, 1024
    from distributedes_b200.engine import shard_bounds
    off, nl = shard_bounds(lam, world, rank)
    Y = torch.randn(nl, n, device=dev)
    w = torch.rand(nl, device=dev)
    Cm = torch.eye(n, device=dev)
    pc = torch.randn(n, device=dev)
    if world > 1:
        tiles = torch.zeros(ops.cma_packed_elems(n), dtype=torch.float32, device=dev)

        def upd4():
            ops.cma_rank_mu_packed(Y, w, out=tiles)
            dist.all_reduce(tiles)
            ops.cma_cov_apply_packed(Cm, tiles, pc, decay=0.99, c1=0.001, cmu=0.009)
    else:
        dC = ops.cma_rank_mu(Y, w)

        def upd4():
            ops.cma_rank_mu(Y, w, out=dC)
            ops.cma_cov_apply(Cm, dC, pc, decay=0.99, c1=0.001, cmu=0.009)
    for _ in range(3):
        upd4()
    ms, _ = timed(upd4, 10)
    upd_ms = max_over_ranks(ms) / 10
    flops = 2.0 * lam * n * n
    r = {'workload': 'cma rank-mu covariance update n=%d lambda=%d over %d GPU(s) (BASELINE configs[4])' % (n, lam, world),
         'config_of': 'BASELINE configs[4]', 'n_gpus': world, 'rank_mu_update_ms': upd_ms, 'updates_per_sec': 1e3 / upd_ms,
         'collective': None if world == 1 else 'all-reduce of the packed upper-triangular tiles (%d MB)' % (2 * n * n // (1 << 20) + 1),
         'roofline': cma_roofline(n, lam, nl, world),
         'parity': 'oracle/cma_oracle.py (tutorial restatement) pinned by tests/test_cma_pinning.py: constants by hand from Hansen 2016, pycma banner (mu_w, w_1) values, one generation in n=3 by literal arithmetic; pycma itself is absent; kernels vs the restatement <= 1e-5 (tests/test_gpu_cma.py)'}
    if with_cpu and rank == 0 and world == 1:
        r['cpu_baseline'] = cma_cpu_baseline(n, lam)
    out.append(r)
    return out


def _guard_stdout():
    """Keep stdout clean for the ONE JSON line: anything libraries print on fd 1 (NCCL writes its version banner
    there) goes to stderr; the JSON line is written to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real = os.fdopen(saved, 'w')

    def emit(line):
        real.write(line + '\n')
        real.flush()
    return emit


if __name__ == '__main__':
    args = parse()
    EMIT = _guard_stdout()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
