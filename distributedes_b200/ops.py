"""Thin torch-tensor front ends for the C-ABI kernels (include/des_b200.h).

PyTorch is plumbing here: it owns device memory and the stream; every op below passes raw
pointers to libdes_b200.so, which enqueues hand-written sm_100a kernels on the current stream.
CPU tensors are an error (there is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import Dims, Opt, PRECISIONS, State


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype, name, allow_none=False):
    if t is None:
        if allow_none:
            return C.c_void_p(0)
        raise RuntimeError('%s is None' % name)
    if not isinstance(t, torch.Tensor):
        raise RuntimeError('%s must be a torch.Tensor' % name)
    if not t.is_cuda:
        raise RuntimeError('%s is a CPU tensor: distributedes_b200 has no CPU path' % name)
    if t.dtype != dtype:
        raise RuntimeError('%s must be %s, got %s' % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise RuntimeError('%s must be contiguous' % name)
    return C.c_void_p(t.data_ptr())


def _on(t, name):
    """Device guard for the tensor that selects the GPU; CPU tensors are an error, not a fallback."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError('%s is a CPU tensor: distributedes_b200 has no CPU path' % name)
    return torch.cuda.device(t.device)


def _precision(p):
    if isinstance(p, str):
        if p not in PRECISIONS:
            raise RuntimeError('unknown precision %r (choose from %s)' % (p, sorted(PRECISIONS)))
        return PRECISIONS[p]
    return int(p)


def param_count(state_dim, hidden, action_dim):
    n = _lib.load().des_param_count(state_dim, hidden, action_dim)
    if n < 0:
        raise RuntimeError('invalid MLP dims (%r, %r, %r)' % (state_dim, hidden, action_dim))
    return int(n)


def new_state(device, generation=0):
    """Device-resident des_state {generation, adam_t, beta1_t, beta2_t} as a 32-byte tensor."""
    st = torch.empty(C.sizeof(State), dtype=torch.uint8, device=device)
    with torch.cuda.device(st.device):
        _lib.check(_lib.load().des_state_init(C.c_void_p(st.data_ptr()), generation, _stream()), 'des_state_init')
    return st


def state_advance(state, beta1=0.9, beta2=0.999):
    with torch.cuda.device(state.device):
        _lib.check(_lib.load().des_state_advance(_ptr(state, torch.uint8, 'state'), beta1, beta2, _stream()),
                   'des_state_advance')


def read_state(state):
    raw = bytes(state.cpu().numpy().tobytes())
    s = State.from_buffer_copy(raw)
    return dict(generation=s.generation, adam_t=s.adam_t, beta1_t=s.beta1_t, beta2_t=s.beta2_t)


def noise_fill(n_members, P, seed, generation, member_offset=0, stream_tag=0, device='cuda'):
    """eps[n_members, P] fp32 — debug/parity op (natural_es.py:29)."""
    out = torch.empty((n_members, P), dtype=torch.float32, device=device)
    with torch.cuda.device(out.device):
        _lib.check(_lib.load().des_noise_fill(_ptr(out, torch.float32, 'out'), n_members, P, seed, generation,
                                              member_offset, stream_tag, _stream()), 'des_noise_fill')
    return out


def nes_perturb(theta, n_members, sigma, seed, generation, member_offset=0):
    """theta'[n_members, P] = fp32(theta + sigma*eps) — debug/parity op (natural_es.py:28-30)."""
    P = theta.numel()
    out = torch.empty((n_members, P), dtype=torch.float32, device=theta.device)
    with _on(theta, 'theta'):
        _lib.check(_lib.load().des_nes_perturb(_ptr(out, torch.float32, 'out'), _ptr(theta, torch.float32, 'theta'),
                                               n_members, P, sigma, seed, generation, member_offset, _stream()),
                   'des_nes_perturb')
    return out


def obs_stats_merge(stats, obs, n_feed):
    """SharedStats.merge of one generation's online statistics on the tape env (utils.py:85-96), in place."""
    T, d0 = obs.shape
    with _on(obs, 'obs'):
        _lib.check(_lib.load().des_obs_stats_merge(_ptr(stats, torch.float32, 'stats'), _ptr(obs, torch.float32, 'obs'),
                                                   T, d0, float(n_feed), _stream()), 'des_obs_stats_merge')
    return stats


def obs_normalize(obs, stats, out=None):
    """StaticNormalizer.__call__ (utils.py:42-57) over the whole tape: identity while stats are empty."""
    T, d0 = obs.shape
    if out is None:
        out = torch.empty_like(obs)
    with _on(obs, 'obs'):
        _lib.check(_lib.load().des_obs_normalize(_ptr(out, torch.float32, 'out'), _ptr(obs, torch.float32, 'obs'),
                                                 _ptr(stats, torch.float32, 'stats'), T, d0, _stream()), 'des_obs_normalize')
    return out


ENV_DIMS = {0: (3, 1)}      # DES_ENV_PENDULUM: (state_dim, action_dim)


def rollout_eval(theta, *, env=0, hidden, horizon=200, repetitions=10, sigma, clip, action_noise_std=0.0, seed,
                 generation=0, state=None, member_offset=0, n_local, noiseless=False, obs_stats=None, totals_out=None,
                 workspace=None, out=None, episodes_out=None):
    """Closed-loop fitness of members [member_offset, member_offset + n_local): mean return over `repetitions`
    episodes stepped on the device (Evaluator.eval utils.py:116-124 over single_run utils.py:126-139)."""
    if env not in ENV_DIMS:
        raise RuntimeError('unknown environment id %r' % (env,))
    d0, A = ENV_DIMS[env]
    if out is None:
        out = torch.empty(n_local, dtype=torch.float32, device=theta.device)
    if totals_out is not None and workspace is None:
        workspace = torch.empty(max(n_local, 1) * (2 * d0 + 1), dtype=torch.float64, device=theta.device)
    ws_bytes = workspace.numel() * workspace.element_size() if workspace is not None else 0
    with _on(theta, 'theta'):
        _lib.check(_lib.load().des_rollout_eval(
            _ptr(out, torch.float32, 'out'), _ptr(episodes_out, torch.float32, 'episodes_out', True),
            _ptr(totals_out, torch.float64, 'totals_out', True), _ptr(theta, torch.float32, 'theta'),
            _ptr(obs_stats, torch.float32, 'obs_stats', True), int(env), Dims(d0, hidden, A, horizon), int(repetitions),
            float(sigma), float(clip), float(action_noise_std), int(seed), int(generation),
            _ptr(state, torch.uint8, 'state', True), int(member_offset), int(n_local), 1 if noiseless else 0,
            C.c_void_p(workspace.data_ptr()) if workspace is not None else C.c_void_p(0), ws_bytes, _stream()),
            'des_rollout_eval')
    return out


def obs_stats_merge_totals(stats, totals, state_dim):
    """Chan merge of a batch given by fp64 [sum | sum of squares | count] into stats [m|v|n] (utils.py:85-96)."""
    with _on(stats, 'stats'):
        _lib.check(_lib.load().des_obs_stats_merge_totals(_ptr(stats, torch.float32, 'stats'),
                                                          _ptr(totals, torch.float64, 'totals'), int(state_dim), _stream()),
                   'des_obs_stats_merge_totals')
    return stats


def eval_workspace(state_dim, hidden, action_dim, tape_len, precision, device):
    """Optional scratch for des_nes_eval (multi-pass tensor-core shapes); None when the shape needs none."""
    with torch.cuda.device(device):
        nbytes = _lib.load().des_nes_eval_workspace_bytes(Dims(state_dim, hidden, action_dim, tape_len), _precision(precision))
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device) if nbytes else None


def nes_eval(theta, obs, target, *, hidden, sigma, clip, seed, generation=0, state=None, member_offset=0,
             n_local, precision='fp32', out=None, workspace=None):
    """Fused sample+forward+fitness for members [member_offset, member_offset+n_local) -> fitness[n_local]."""
    T, d0 = obs.shape
    A = target.shape[1]
    if target.shape[0] != T:
        raise RuntimeError('obs has %d rows but target has %d' % (T, target.shape[0]))
    if theta.numel() != param_count(d0, hidden, A):
        raise RuntimeError('theta has %d entries, the (%d,%d,%d) MLP needs %d' %
                           (theta.numel(), d0, hidden, A, param_count(d0, hidden, A)))
    if out is None:
        out = torch.empty(n_local, dtype=torch.float32, device=theta.device)
    elif out.numel() != n_local:
        raise RuntimeError('out has %d entries, need n_local=%d' % (out.numel(), n_local))
    with _on(theta, 'theta'):
        _lib.check(_lib.load().des_nes_eval(
            _ptr(out, torch.float32, 'out'), _ptr(theta, torch.float32, 'theta'), _ptr(obs, torch.float32, 'obs'),
            _ptr(target, torch.float32, 'target'), Dims(d0, hidden, A, T), sigma, clip, seed, generation,
            _ptr(state, torch.uint8, 'state', allow_none=True), member_offset, n_local, _precision(precision),
            _ptr(workspace, torch.uint8, 'workspace', allow_none=True), workspace.numel() if workspace is not None else 0,
            _stream()), 'des_nes_eval')
    return out


def pop_eval(solutions, obs, target, *, hidden, clip, out=None):
    """Tape fitness of explicit weight vectors solutions[n, P] (what CMA-ES evaluates, cma_es.py:62-75)."""
    T, d0 = obs.shape
    A = target.shape[1]
    n, P = solutions.shape
    if P != param_count(d0, hidden, A):
        raise RuntimeError('solutions have %d entries, the (%d,%d,%d) MLP needs %d' % (P, d0, hidden, A, param_count(d0, hidden, A)))
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=solutions.device)
    with _on(solutions, 'solutions'):
        _lib.check(_lib.load().des_pop_eval(_ptr(out, torch.float32, 'out'), _ptr(solutions, torch.float32, 'solutions'),
                                            _ptr(obs, torch.float32, 'obs'), _ptr(target, torch.float32, 'target'),
                                            Dims(d0, hidden, A, T), clip, n, _stream()), 'des_pop_eval')
    return out


def rank_workspace(n_local, device, N=None):
    lib = _lib.load()
    nbytes = lib.des_rank_workspace_bytes_n(N, n_local) if N is not None else lib.des_rank_workspace_bytes(n_local)
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def centered_rank(fitness_all, member_offset=0, n_local=None, *, workspace=None, return_ranks=False, out=None):
    """fitness_shift (utils.py:142-148) for a shard of the global fitness vector."""
    _on(fitness_all, 'fitness_all')
    N = fitness_all.numel()
    if n_local is None:
        n_local = N - member_offset
    dev = fitness_all.device
    if out is None:
        out = torch.empty(n_local, dtype=torch.float32, device=dev)
    ranks = torch.empty(n_local, dtype=torch.int32, device=dev) if return_ranks else None
    if workspace is None:
        workspace = rank_workspace(n_local, dev, N)
    with _on(fitness_all, 'fitness_all'):
        _lib.check(_lib.load().des_centered_rank(
            _ptr(out, torch.float32, 'out'), _ptr(ranks, torch.int32, 'ranks', allow_none=True),
            _ptr(fitness_all, torch.float32, 'fitness_all'), N, member_offset, n_local,
            _ptr(workspace, torch.uint8, 'workspace'), workspace.numel(), _stream()), 'des_centered_rank')
    return (out, ranks) if return_ranks else out


def grad_workspace(n_local, P, device):
    nbytes = _lib.load().des_grad_workspace_bytes(n_local, P)
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def nes_grad_partial(shaped_local, P, *, seed, generation=0, state=None, member_offset=0, workspace=None, out=None):
    """partial[P] = sum_i shaped[i] * eps[member_offset+i] (natural_es.py:91, per shard; eps regenerated)."""
    _on(shaped_local, 'shaped_local')
    n_local = shaped_local.numel()
    dev = shaped_local.device
    if out is None:
        out = torch.empty(P, dtype=torch.float32, device=dev)
    if workspace is None:
        workspace = grad_workspace(n_local, P, dev)
    with _on(shaped_local, 'shaped_local'):
        _lib.check(_lib.load().des_nes_grad_partial(
            _ptr(out, torch.float32, 'out'), _ptr(shaped_local, torch.float32, 'shaped_local'), n_local, P, seed,
            generation, _ptr(state, torch.uint8, 'state', allow_none=True), member_offset,
            _ptr(workspace, torch.uint8, 'workspace'), workspace.numel(), _stream()), 'des_nes_grad_partial')
    return out


def nes_apply(theta, adam_m, adam_v, partial_sum, N, state, *, sigma, learning_rate, weight_decay=0.005,
              beta1=0.9, beta2=0.999, epsilon=1e-8, update_out=None, grad_out=None):
    """natural_es.py:92-96 + utils.py:159-166, in place on theta / adam_m / adam_v (fp64 Adam state)."""
    P = theta.numel()
    with _on(theta, 'theta'):
        _lib.check(_lib.load().des_nes_apply(
            _ptr(theta, torch.float32, 'theta'), _ptr(adam_m, torch.float64, 'adam_m'),
            _ptr(adam_v, torch.float64, 'adam_v'), _ptr(update_out, torch.float32, 'update_out', allow_none=True),
            _ptr(grad_out, torch.float64, 'grad_out', allow_none=True),
            _ptr(partial_sum, torch.float32, 'partial_sum'), P, N,
            Opt(sigma, learning_rate, weight_decay, beta1, beta2, epsilon), _ptr(state, torch.uint8, 'state'),
            _stream()), 'des_nes_apply')


_CMA_WS = {}      # (device, n, lambda) -> workspace tensor of the tensor-core rank-mu path
CMA_TC_MIN_N = 2048


def _cma_tc_workspace(n, lam, device):
    key = (str(device), int(n), int(lam))
    ws = _CMA_WS.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.load().des_cma_tc_workspace_bytes(int(n), int(lam))), dtype=torch.uint8, device=device)
        if len(_CMA_WS) > 8:
            _CMA_WS.clear()
        _CMA_WS[key] = ws
    return ws


def _cma_rank_mu(Y, w, out, packed, path):
    lam, n = Y.shape
    lib = _lib.load()
    use_tc = (path == 'tc') or (path is None and n >= CMA_TC_MIN_N and lam >= 1)
    with _on(Y, 'Y'):
        if use_tc:
            ws = _cma_tc_workspace(n, lam, Y.device)
            _lib.check(lib.des_cma_rank_mu_tc(_ptr(out, torch.float32, 'out'), _ptr(Y, torch.float32, 'Y'),
                                              _ptr(w, torch.float32, 'w'), lam, n, 1 if packed else 0,
                                              C.c_void_p(ws.data_ptr()), ws.numel(), _stream()), 'des_cma_rank_mu_tc')
        elif packed:
            _lib.check(lib.des_cma_rank_mu_packed(_ptr(out, torch.float32, 'out'), _ptr(Y, torch.float32, 'Y'),
                                                  _ptr(w, torch.float32, 'w'), lam, n, _stream()), 'des_cma_rank_mu_packed')
        else:
            _lib.check(lib.des_cma_rank_mu(_ptr(out, torch.float32, 'out'), _ptr(Y, torch.float32, 'Y'),
                                           _ptr(w, torch.float32, 'w'), lam, n, _stream()), 'des_cma_rank_mu')
    return out


def cma_rank_mu(Y, w, out=None, path=None):
    """dC[n,n] = sum_i w_i y_i y_i^T for Y[lambda_local, n] (rank-mu term of es.tell, cma_es.py:90).
    path: None = tensor cores (split-fp16 tcgen05 SYRK) for n >= CMA_TC_MIN_N (2048), fp32 FFMA below; 'tc' / 'ffma'
    force one."""
    lam, n = Y.shape
    if w.numel() != lam:
        raise RuntimeError('w has %d entries, Y has %d rows' % (w.numel(), lam))
    if out is None:
        out = torch.empty((n, n), dtype=torch.float32, device=Y.device)
    return _cma_rank_mu(Y, w, out, False, path)


def cma_cov_apply(Cmat, dC, pc, *, decay, c1, cmu):
    """C <- decay*C + c1*pc pc^T + cmu*dC, in place."""
    n = Cmat.shape[0]
    with _on(Cmat, 'C'):
        _lib.check(_lib.load().des_cma_cov_apply(_ptr(Cmat, torch.float32, 'C'), _ptr(dC, torch.float32, 'dC'),
                                                 _ptr(pc, torch.float32, 'pc', allow_none=True), n, decay, c1, cmu,
                                                 _stream()), 'des_cma_cov_apply')
    return Cmat


def cma_packed_elems(n):
    return int(_lib.load().des_cma_packed_elems(int(n)))


def cma_rank_mu_packed(Y, w, out=None, path=None):
    """The rank-mu partial as packed upper-triangular tiles (the multi-GPU all-reduce payload: half of [n, n])."""
    lam, n = Y.shape
    if w.numel() != lam:
        raise RuntimeError('w has %d entries, Y has %d rows' % (w.numel(), lam))
    if out is None:
        out = torch.empty(cma_packed_elems(n), dtype=torch.float32, device=Y.device)
    return _cma_rank_mu(Y, w, out, True, path)


def cma_cov_apply_packed(Cmat, tiles, pc, *, decay, c1, cmu):
    """C <- decay*C + c1*pc pc^T + cmu*dC with dC as packed upper tiles, in place."""
    n = Cmat.shape[0]
    with _on(Cmat, 'C'):
        _lib.check(_lib.load().des_cma_cov_apply_packed(_ptr(Cmat, torch.float32, 'C'), _ptr(tiles, torch.float32, 'tiles'),
                                                        _ptr(pc, torch.float32, 'pc', allow_none=True), n, decay, c1, cmu,
                                                        _stream()), 'des_cma_cov_apply_packed')
    return Cmat
