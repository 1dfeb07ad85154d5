"""Torch-facing wrappers of the C-ABI kernels (device tensors in, device tensors out).

PyTorch is plumbing here: it owns device memory and streams; every operation
below is one call into ``libcoevonet_b200.so`` on the current CUDA stream.
There is no CPU path: non-CUDA tensors raise.
"""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib, layout
from ._lib import RolloutCfg, check, handle, load

MAX_CYCLES = 25

#: kernels launched per C-ABI call (bench.py reports the total as ``gpu_launches``)
_KERNELS_PER_CALL = {"cev_es_update_f32": 2, "cev_es_update_members_f32": 2, "cev_es_update_mirrored_f32": 2,
                     "cev_es_update_diag_f32": 2, "cev_es_subspace_basis_f32": 6, "cev_fp32_peak": 4,
                     "cev_ga_novelty_knn_f64": 2, "cev_ga_safe_scale_f32": 5}
launch_count = 0


def _call(name, *args, launches=None):
    """Invoke one C-ABI entry point, counting the CUDA kernels it launches."""
    global launch_count
    launch_count += _KERNELS_PER_CALL.get(name, 1) if launches is None else launches
    return getattr(load(), name)(*args)


def rollout_plan(device_index, P, K, E, n_cycles=25, variant=0):
    """(kernel variant, kernels launched) of one structured rollout of this shape:
    1 generic, 2 cluster (member weights resident), 3 lockstep (opponents on tcgen05)."""
    used, n = ctypes.c_int(), ctypes.c_int()
    check(load().cev_mpe_rollout_plan(handle(device_index), int(P), int(K), int(E), int(n_cycles),
                                      int(variant), ctypes.byref(used), ctypes.byref(n)),
          "cev_mpe_rollout_plan")
    return used.value, n.value


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _h(dev):
    """The library handle of the device and the CURRENT stream (one scratch workspace per stream)."""
    return handle(dev.index, torch.cuda.current_stream(dev).cuda_stream)


def _need_cuda(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.CevError("coevonet_b200 ops need CUDA tensors (no CPU fallback)")
        if not t.is_contiguous():
            raise _lib.CevError("coevonet_b200 ops need contiguous tensors")
        dev = t.device if dev is None else dev
        if t.device != dev:
            raise _lib.CevError("all tensors of one op must live on the same device")
    return dev


def _need_rows(dev, *rows):
    """Weight rows handed to the kernels with their ``stride(0)`` as the row pitch: CUDA [n, pitch] tensors on
    ``dev`` whose rows are contiguous (column views of a wider buffer qualify)."""
    for t in rows:
        if not t.is_cuda or t.device != dev:
            raise _lib.CevError("weight rows must be CUDA tensors on the device of the other operands")
        if t.dim() != 2 or t.stride(1) != 1:
            raise _lib.CevError("weight rows must be a [n, pitch] tensor with contiguous rows")


def cycles_for_limit(agent_step_limit):
    """World steps executed under ``play_MPE``'s agent-step limit
    (``utils/game_logic_functions.py:127,195-210``; truncation after 25 cycles)."""
    if agent_step_limit is None:
        return MAX_CYCLES
    return int(min(MAX_CYCLES, max(0, int(agent_step_limit)) // 3))


def reward_slots(out, agent_step_limit=None, reference_compat=True):
    """Map the kernel's physical sums ``out[..., 4]`` to the triple ``play_game``
    returns ``(agent_0, agent_1, adversary_0)``.

    ``reference_compat`` reproduces the rotated attribution of
    ``utils/game_logic_functions.py:179-190`` (SURVEY.md Appendix B): agent_0's
    and adversary_0's slots hold the good agents' reward up to the previous
    cycle, agent_1's slot the adversary's.  ``False`` credits each role its own
    reward sum."""
    sg, lg, sa = out[..., 0], out[..., 1], out[..., 2]
    if not reference_compat:
        return sg, sg, sa
    L = 75 if agent_step_limit is None else int(min(75, max(0, int(agent_step_limit))))
    nc = L // 3
    if nc == 0:
        z = torch.zeros_like(sg)
        return z, sa, z
    n_adv = -(-L // 3)
    n_a0 = -(-(L - 1) // 3)
    slot_adv = sg if n_adv - 1 >= nc else sg - lg
    slot_a0 = sg if n_a0 - 1 >= nc else sg - lg
    return slot_a0, sa, slot_adv


def raise_on_status(status):
    """Surface device-detected faults as the reference's ``ValueError``
    (``MPE/fcnetwork.py:39-65``).  Synchronises."""
    code = int(status.item())
    if code & _lib.STATUS_NONFINITE:
        raise ValueError("\n\t Warning: output contains inf or NaN")


def kernel_timing_enable(device_index, on=True):
    """Record CUDA events around every member / opponent kernel of the lockstep rollout."""
    check(load().cev_kernel_timing_enable(handle(device_index), int(bool(on))), "cev_kernel_timing_enable")


def kernel_timing_read(device_index, which):
    """(summed device ms, launches) of the member (which=0) or opponent (which=1) kernel since the
    last read.  Synchronises on the recorded events."""
    ms, n = ctypes.c_double(), ctypes.c_int()
    check(load().cev_kernel_timing_read(handle(device_index), int(which), ctypes.byref(ms), ctypes.byref(n)),
          "cev_kernel_timing_read")
    return ms.value, n.value


def mpe_rollout(member_role, members, opp_a, opp_b, init, *, n_cycles=MAX_CYCLES,
                pos_first=True, init_shared=False, variant=0, out=None, status=None):
    """K1 structured rollout.

    members fp32[P, pitch]; opp_a / opp_b fp32[K, pitch] for the two other seats
    in ascending seat order (adversary_0 < agent_0 < agent_1), rows contiguous, the row
    pitch taken from ``stride(0)``; init fp64 [P, K, E, 11] (or [K, E, 11] with
    ``init_shared``).  Returns fp64 [P, K, E, 4].
    """
    dev = _need_cuda(members, init, out, status)
    _need_rows(dev, opp_a, opp_b)
    seat = layout.SEAT_OF[member_role] if isinstance(member_role, str) else int(member_role)
    P, K = members.shape[0], opp_a.shape[0]
    if opp_b.shape[0] != K:
        raise _lib.CevError("opp_a and opp_b must hold the same number of rows")
    if init_shared:
        if init.dim() != 3 or init.shape[0] != K or init.shape[2] != _lib.INIT_STATE_DIM:
            raise _lib.CevError("shared init must be fp64 [K, E, 11]")
        E = init.shape[1]
    else:
        if init.dim() != 4 or init.shape[:2] != (P, K) or init.shape[3] != _lib.INIT_STATE_DIM:
            raise _lib.CevError("init must be fp64 [P, K, E, 11]")
        E = init.shape[2]
    if members.dtype != torch.float32 or init.dtype != torch.float64:
        raise _lib.CevError("members must be float32 and init float64")
    if out is None:
        out = torch.empty((P, K, E, _lib.ROLLOUT_OUT_DIM), dtype=torch.float64, device=dev)
    if P == 0:
        return out                        # an empty shard plays nothing
    cfg = RolloutCfg(int(n_cycles), int(bool(pos_first)), int(variant), 0)
    _, n_launch = rollout_plan(dev.index, P, K, E, n_cycles, variant)
    check(_call("cev_mpe_rollout_f32",
        _h(dev), seat, _ptr(members), P, members.stride(0),
        _ptr(opp_a), opp_a.stride(0), _ptr(opp_b), opp_b.stride(0), K,
        _ptr(init), int(bool(init_shared)), E, ctypes.byref(cfg), _ptr(out), _ptr(status),
        _stream(dev), launches=n_launch), "cev_mpe_rollout_f32")
    return out


def mpe_rollout_roles(roles, *, n_cycles=MAX_CYCLES, pos_first=True, init_shared=False, variant=0, status=None):
    """K1 for the roles of one generation in one pass (``cev_mpe_rollout_roles_f32``).

    ``roles``: list of (member_role, members fp32[P, pitch], opp_a fp32[K, pitch], opp_b, init fp64[P, K, E, 11])
    with the same P, K, E for every role (opponent rows as in :func:`mpe_rollout`).  Returns the list of fp64
    [P, K, E, 4] results, identical to one :func:`mpe_rollout` per role."""
    outs, recs, keep = [], (_lib.RolloutRole * len(roles))(), []
    P = K = E = None
    dev = None
    for i, (member_role, members, opp_a, opp_b, init) in enumerate(roles):
        dev = _need_cuda(members, init, status)
        _need_rows(dev, opp_a, opp_b)
        seat = layout.SEAT_OF[member_role] if isinstance(member_role, str) else int(member_role)
        p_, k_ = members.shape[0], opp_a.shape[0]
        e_ = init.shape[1] if init_shared else init.shape[2]
        if opp_b.shape[0] != k_:
            raise _lib.CevError("opp_a and opp_b must hold the same number of rows")
        if (init_shared and (init.dim() != 3 or init.shape[0] != k_)) or \
                (not init_shared and (init.dim() != 4 or tuple(init.shape[:2]) != (p_, k_))) or \
                init.shape[-1] != _lib.INIT_STATE_DIM:
            raise _lib.CevError("init must be fp64 [P, K, E, 11] (or [K, E, 11] with init_shared)")
        if members.dtype != torch.float32 or init.dtype != torch.float64:
            raise _lib.CevError("members must be float32 and init float64")
        if P is None:
            P, K, E = p_, k_, e_
        elif (P, K, E) != (p_, k_, e_):
            raise _lib.CevError("every role must have the same P, K, E")
        out = torch.empty((p_, k_, e_, _lib.ROLLOUT_OUT_DIM), dtype=torch.float64, device=dev)
        outs.append(out)
        keep.append((members, opp_a, opp_b, init))
        r = recs[i]
        r.member_seat, r.reserved = seat, 0
        r.members, r.member_pitch = members.data_ptr(), members.stride(0)
        r.opp_a, r.opp_a_pitch = opp_a.data_ptr(), opp_a.stride(0)
        r.opp_b, r.opp_b_pitch = opp_b.data_ptr(), opp_b.stride(0)
        r.init, r.out = init.data_ptr(), out.data_ptr()
    if not roles or P == 0:
        return outs
    cfg = RolloutCfg(int(n_cycles), int(bool(pos_first)), int(variant), 0)
    _, n_launch = rollout_plan(dev.index, P, K, E, n_cycles, variant)
    check(_call("cev_mpe_rollout_roles_f32", _h(dev), len(roles), recs, P, K, int(bool(init_shared)), E,
                ctypes.byref(cfg), _ptr(status), _stream(dev), launches=n_launch * len(roles)),
          "cev_mpe_rollout_roles_f32")
    return outs


def mpe_rollout_trace(member_role, members, opp_a, opp_b, init, *, n_cycles=MAX_CYCLES, pos_first=True,
                      forced_actions=None, status=None):
    """K1 lockstep kernels with parity instrumentation: returns (out fp64 [P,K,E,4], logits fp32
    [n_cycles,3,N,5], actions int32 [n_cycles,3,N]); ``forced_actions`` int32 [n_cycles,3,N] replays
    a given action trace (teacher forcing).  Seats in world order, N = P*K*E."""
    dev = _need_cuda(members, opp_a, opp_b, init, forced_actions, status)
    seat = layout.SEAT_OF[member_role] if isinstance(member_role, str) else int(member_role)
    P, K = members.shape[0], opp_a.shape[0]
    if init.dim() != 4 or init.shape[:2] != (P, K) or init.shape[3] != _lib.INIT_STATE_DIM:
        raise _lib.CevError("init must be fp64 [P, K, E, 11]")
    E = init.shape[2]
    N = P * K * E
    if forced_actions is not None and (forced_actions.dtype != torch.int32 or
                                       tuple(forced_actions.shape) != (n_cycles, 3, N)):
        raise _lib.CevError("forced_actions must be int32 [n_cycles, 3, N]")
    out = torch.empty((P, K, E, _lib.ROLLOUT_OUT_DIM), dtype=torch.float64, device=dev)
    logits = torch.zeros((n_cycles, 3, N, layout.NACT), dtype=torch.float32, device=dev)
    actions = torch.zeros((n_cycles, 3, N), dtype=torch.int32, device=dev)
    cfg = RolloutCfg(int(n_cycles), int(bool(pos_first)), 3, 0)
    check(_call("cev_mpe_rollout_trace_f32", _h(dev), seat, _ptr(members), P, members.stride(0),
                _ptr(opp_a), opp_a.stride(0), _ptr(opp_b), opp_b.stride(0), K, _ptr(init), 0, E,
                ctypes.byref(cfg), _ptr(forced_actions), _ptr(logits), _ptr(actions), _ptr(out), _ptr(status),
                _stream(dev), launches=3 + 3 * int(n_cycles)), "cev_mpe_rollout_trace_f32")
    return out, logits, actions


def mpe_rollout_indexed(w_adv, w_a0, w_a1, idx, init, *, n_cycles=MAX_CYCLES, pos_first=True,
                        out=None, status=None):
    """K1 indexed rollout: episode e is played by rows ``idx[e] = (adv, a0, a1)``."""
    dev = _need_cuda(w_adv, w_a0, w_a1, idx, init, out, status)
    N = idx.shape[0]
    if idx.dtype != torch.int32 or init.dtype != torch.float64 or init.shape != (N, _lib.INIT_STATE_DIM):
        raise _lib.CevError("idx must be int32 [N,3] and init fp64 [N,11]")
    if out is None:
        out = torch.empty((N, _lib.ROLLOUT_OUT_DIM), dtype=torch.float64, device=dev)
    cfg = RolloutCfg(int(n_cycles), int(bool(pos_first)), 1, 0)
    check(_call("cev_mpe_rollout_indexed_f32", 
        _h(dev), _ptr(w_adv), w_adv.stride(0), _ptr(w_a0), w_a0.stride(0),
        _ptr(w_a1), w_a1.stride(0), _ptr(idx), _ptr(init), N, ctypes.byref(cfg), _ptr(out),
        _ptr(status), _stream(dev)), "cev_mpe_rollout_indexed_f32")
    return out


def fc_forward(rows, in_dim, obs, idx=None, *, status=None):
    """Batched ``FCNetwork.forward`` + ``determine_action`` on given observations:
    logits fp32[N,5], actions int32[N]; sample n uses ``rows[idx[n]]`` (row 0 if idx is None)."""
    dev = _need_cuda(rows, obs, idx, status)
    N = obs.shape[0]
    if obs.dtype != torch.float32 or obs.shape[1] != in_dim:
        raise _lib.CevError("fc_forward: obs must be float32 [N, in_dim]")
    if idx is not None and idx.dtype != torch.int32:
        raise _lib.CevError("fc_forward: idx must be int32")
    logits = torch.empty((N, layout.NACT), dtype=torch.float32, device=dev)
    actions = torch.empty(N, dtype=torch.int32, device=dev)
    check(_call("cev_fc_forward_f32", _h(dev), _ptr(rows), rows.stride(0), int(in_dim), _ptr(idx),
                                    _ptr(obs), N, _ptr(logits), _ptr(actions), _ptr(status), _stream(dev)),
          "cev_fc_forward_f32")
    return logits, actions


def _sigma_args(sigma):
    """(by-value float, device pointer) of a mutation power given as a Python float or as a
    one-element fp64 DEVICE tensor (a slot of the generation state, read by the kernel)."""
    if torch.is_tensor(sigma):
        if sigma.dtype != torch.float64 or sigma.numel() != 1 or not sigma.is_cuda:
            raise _lib.CevError("a device sigma must be a one-element float64 CUDA tensor")
        return 0.0, _ptr(sigma)
    return float(sigma), ctypes.c_void_p(0)


def ga_repopulate(elites, dim, sigma, seed, role, gen, row0, n_rows, *, out=None, noise_out=None,
                  crossover_rate=0.0, scale=None):
    """K3: rows [row0, row0+n_rows) of the next GA population.  ``crossover_rate`` > 0 adds uniform
    crossover between two elites before the mutation (an extension; 0 = the reference).  ``scale`` fp32 [E, pitch]
    (``ga_safe_scale`` of the elites) turns the mutation of parameter j into fl(fl(sigma * z_j) * c_j), c_j from the
    elite the parameter was copied from (``cev_ga_repopulate_safe_f32``); None = the plain K3."""
    dev = _need_cuda(elites, out, noise_out, scale)
    sig, sig_dev = _sigma_args(sigma)
    pitch = elites.stride(0)
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    if scale is None:
        check(_call("cev_ga_repopulate_f32", 
            _h(dev), _ptr(elites), elites.shape[0], int(dim), pitch, sig, sig_dev, float(crossover_rate),
            int(seed), role_id, int(gen), int(row0), int(n_rows), _ptr(out), _ptr(noise_out),
            _stream(dev)), "cev_ga_repopulate_f32")
        return out
    if scale.dtype != torch.float32 or tuple(scale.shape) != tuple(elites.shape) or scale.stride(0) != pitch:
        raise _lib.CevError(f"ga_repopulate: scale must be float32 {tuple(elites.shape)}, laid out like the elites")
    check(_call("cev_ga_repopulate_safe_f32", _h(dev), _ptr(elites), _ptr(scale), elites.shape[0], int(dim), pitch,
                sig, sig_dev, float(crossover_rate), int(seed), role_id, int(gen), int(row0), int(n_rows), _ptr(out),
                _ptr(noise_out), _stream(dev)), "cev_ga_repopulate_safe_f32")
    return out


def gather_rows(src, idx, *, row0=0, n_local=None, out=None):
    """dst[i] = src[idx[i] - row0]; with ``n_local`` the ids are GLOBAL and rows outside this rank's
    block [row0, row0+n_local) come back as zeros (summed over ranks = the elite broadcast)."""
    dev = _need_cuda(idx, out, src if src.numel() else None)
    if idx.dtype != torch.int64:
        raise _lib.CevError("gather_rows: idx must be int64")
    pitch = src.stride(0) if src.dim() == 2 and src.shape[0] > 0 else src.shape[-1]
    if out is None:
        out = torch.empty((idx.shape[0], pitch), dtype=torch.float32, device=dev)
    check(_call("cev_gather_rows_f32", _h(dev), _ptr(src) if src.numel() else ctypes.c_void_p(0), pitch, _ptr(idx),
                idx.shape[0], int(row0), -1 if n_local is None else int(n_local), _ptr(out), _stream(dev)),
          "cev_gather_rows_f32")
    return out


def select_topk(fitness, k, order=_lib.ORDER_STABLE_DESC):
    """K4: int64[k] indices of the k largest fitness values, descending.  ``order`` 0: ties -> lower
    index, NaN last; 1 (``ORDER_REFERENCE``): the reference's ``np.argsort(f)[::-1]`` with a stable
    sort: ties -> higher index, NaN first."""
    dev = _need_cuda(fitness)
    if fitness.dtype != torch.float64 or fitness.dim() != 1:
        raise _lib.CevError("select_topk: fitness must be float64 [P]")
    idx = torch.empty(k, dtype=torch.int64, device=dev)
    check(_call("cev_select_topk_f64", _h(dev), _ptr(fitness), fitness.shape[0], int(k), int(order),
                                     _ptr(idx), _stream(dev)), "cev_select_topk_f64")
    return idx


def es_perturb(theta, in_dim, sigma, seed, role, gen, row0, n_rows, *, out=None, noise_out=None):
    """K5: perturbed member rows theta + sigma*N(0,1) (Linear parameters only)."""
    return _es_perturb("cev_es_perturb_f32", theta, in_dim, sigma, seed, role, gen, row0, n_rows, out, noise_out)


def es_perturb_mirrored(theta, in_dim, sigma, seed, role, gen, row0, n_rows, *, out=None, noise_out=None):
    """K5 with mirrored sampling: global member c = theta + s*sigma*z_q, pair q = c >> 1, s = +1 for even c and
    -1 for odd c (one normal draw per pair); ``noise_out`` receives s*z."""
    return _es_perturb("cev_es_perturb_mirrored_f32", theta, in_dim, sigma, seed, role, gen, row0, n_rows, out,
                       noise_out)


def _es_perturb(name, theta, in_dim, sigma, seed, role, gen, row0, n_rows, out, noise_out):
    dev = _need_cuda(theta, out, noise_out)
    pitch = layout.fc_pitch(in_dim)
    if theta.numel() < pitch:
        raise _lib.CevError("es_perturb: theta must be a padded flat row")
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    sig, sig_dev = _sigma_args(sigma)
    check(_call(name,
        _h(dev), _ptr(theta), int(in_dim), sig, sig_dev, int(seed), role_id, int(gen),
        int(row0), int(n_rows), pitch, _ptr(out), _ptr(noise_out), _stream(dev)), name)
    return out


def es_perturb_dqn(theta, c_in, n_actions, sigma, seed, role, gen, row0, n_rows, *, out=None):
    """K5 for DeepQN rows: theta + sigma*N(0,1) on the conv / Linear parameters (a prefix of the row),
    BatchNorm gamma / beta copied (``Atari/deepqn.py:158-172``)."""
    dev = _need_cuda(theta, out)
    pitch, total = layout.dqn_pitch(c_in, n_actions), layout.dqn_dim(c_in, n_actions)
    d_pert = total - 2 * (32 + 64 + 64)
    if theta.numel() < pitch:
        raise _lib.CevError("es_perturb_dqn: theta must be a padded flat row")
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    sig, sig_dev = _sigma_args(sigma)
    check(_call("cev_es_perturb_prefix_f32", _h(dev), _ptr(theta), d_pert, total, sig, sig_dev, int(seed), role_id,
                int(gen), int(row0), int(n_rows), pitch, _ptr(out), _stream(dev)), "cev_es_perturb_prefix_f32")
    return out


def es_update(fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, *, out=None):
    """K6: delta fp32[pitch] = lr/(n_total*sigma) * sum_i (sigma z_i) fitness_i over the
    local members [row0, row0+len(fitness))."""
    return _es_update("cev_es_update_f32", fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, out)


def es_update_mirrored(fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, *, out=None):
    """K6 with mirrored sampling, noise regenerated: the delta of :func:`es_update` for the members
    :func:`es_perturb_mirrored` writes (sigma z_i = s_i * sigma z_{i >> 1}, one draw per pair)."""
    return _es_update("cev_es_update_mirrored_f32", fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, out)


def _es_update(name, fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, out):
    dev = _need_cuda(fitness, out)
    if fitness.dtype != torch.float64:
        raise _lib.CevError("es_update: fitness must be float64")
    pitch = layout.fc_pitch(in_dim)
    if out is None:
        out = torch.empty(pitch, dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    sig, sig_dev = _sigma_args(sigma)
    check(_call(name,
        _h(dev), _ptr(fitness), int(in_dim), sig, sig_dev, float(lr), int(n_total),
        int(seed), role_id, int(gen), int(row0), fitness.shape[0], _ptr(out), _stream(dev)), name)
    return out


def es_update_members(fitness, members, theta, in_dim, sigma, lr, n_total, *, out=None):
    """K6 from the materialised members: delta fp32[pitch] = lr/(n_total*sigma) * sum_i (members[i] - theta)
    * fitness_i (the reference's `noises` array read back instead of regenerated)."""
    dev = _need_cuda(theta, out, fitness if fitness.numel() else None, members if members.numel() else None)
    if fitness.dtype != torch.float64 or fitness.shape[0] != members.shape[0]:
        raise _lib.CevError("es_update_members: fitness must be float64 [n_rows]")
    pitch = layout.fc_pitch(in_dim) if in_dim else members.stride(0)      # in_dim 0: any row layout (DeepQN)
    if (members.shape[0] > 0 and members.stride(0) != pitch) or theta.numel() < pitch:
        raise _lib.CevError("es_update_members: members / theta must use the padded row pitch")
    if out is None:
        out = torch.empty(pitch, dtype=torch.float32, device=dev)
    sig, sig_dev = _sigma_args(sigma)
    empty = members.shape[0] == 0
    check(_call("cev_es_update_members_f32", _h(dev), ctypes.c_void_p(0) if empty else _ptr(fitness),
                ctypes.c_void_p(0) if empty else _ptr(members), pitch, _ptr(theta),
                int(in_dim), sig, sig_dev, float(lr), int(n_total), members.shape[0], _ptr(out), _stream(dev)),
          "cev_es_update_members_f32")
    return out


def weight_stats(rows, in_dim, *, out=None):
    """fp32 [n_rows, 4] = (mean, min, max, population std) of every row's perturbable weights
    (``MPEAgent.log_weight_statistics``, ``MPE/mpe_agent.py:30-50``)."""
    n = rows.shape[0]
    if out is None:
        out = torch.empty((n, 4), dtype=torch.float32, device=rows.device)
    if n == 0:
        return out
    dev = _need_cuda(rows, out)
    check(_call("cev_weight_stats_f32", _h(dev), _ptr(rows), n, rows.stride(0), int(in_dim), _ptr(out),
                _stream(dev)), "cev_weight_stats_f32")
    return out


def generation_state(sigmas, hist_capacity, device):
    """A fresh device generation state (fp64; ``CEV_GS_*`` slots): generation 0, the three mutation
    powers (agent_0, agent_1, adversary_0), best = -inf, empty histories."""
    n = int(load().cev_generation_state_doubles(int(hist_capacity)))
    gs = torch.zeros(n, dtype=torch.float64)
    gs[_lib.GS_SIGMA:_lib.GS_SIGMA + 3] = torch.tensor([float(x) for x in sigmas], dtype=torch.float64)
    gs[_lib.GS_BEST:_lib.GS_BEST + 3] = float("-inf")
    sh = _lib.GS_HIST + 3 * int(hist_capacity)
    gs[sh:sh + 3] = gs[_lib.GS_SIGMA:_lib.GS_SIGMA + 3]
    return gs.to(device)


def generation_end(eval_out, gstate, hist_capacity, *, agent_step_limit=None, reference_compat=True,
                   adaptive=False, sigma_max=0.5, sigma_min=0.001, early_stopping=False, min_delta=0.1,
                   patience=300):
    """End-of-generation bookkeeping on the device (evaluation mean, reward history, adaptive sigma,
    early-stopping counters); see ``cev_generation_end_f64``."""
    dev = _need_cuda(eval_out, gstate)
    if eval_out.dtype != torch.float64 or gstate.dtype != torch.float64:
        raise _lib.CevError("generation_end: eval_out and gstate must be float64")
    n_games = eval_out.numel() // _lib.ROLLOUT_OUT_DIM
    check(_call("cev_generation_end_f64", _h(dev), _ptr(eval_out), n_games,
                -1 if agent_step_limit is None else int(agent_step_limit), int(bool(reference_compat)),
                _ptr(gstate), int(hist_capacity), int(bool(adaptive)), float(sigma_max), float(sigma_min),
                int(bool(early_stopping)), float(min_delta), int(patience), _stream(dev)),
          "cev_generation_end_f64")
    return gstate


def centered_ranks(fitness, row0=0, n_rows=None, *, out=None):
    """Centered-rank fitness shaping: fp64[n_rows] = rank_i / (P-1) - 0.5 for the rows [row0, row0 + n_rows) of
    the GLOBAL fitness fp64[P] (average ranks for ties, -0.0 == +0.0, NaNs tie below every number)."""
    dev = _need_cuda(fitness, out)
    if fitness.dtype != torch.float64 or fitness.dim() != 1:
        raise _lib.CevError("centered_ranks: fitness must be float64 [P]")
    P = fitness.shape[0]
    n_rows = P - int(row0) if n_rows is None else int(n_rows)
    if out is None:
        out = torch.empty(n_rows, dtype=torch.float64, device=dev)
    check(_call("cev_centered_ranks_f64", _h(dev), _ptr(fitness), P, int(row0), n_rows, _ptr(out), _stream(dev)),
          "cev_centered_ranks_f64")
    return out


def es_apply(theta, delta, in_dims, *, optimizer="sgd", lr, l2_coeff=0.0, t=1, m=None, v=None):
    """Fused ES apply over the FCNetwork rows of ``in_dims`` concatenated in ``theta`` / ``delta`` (and the Adam
    moments ``m`` / ``v``, same layout): g = delta - l2_coeff * theta, then ``sgd``: theta += lr * g, or ``adam``
    at step ``t`` (updates applied including this one).  Only the Linear entries change."""
    dev = _need_cuda(theta, delta, m, v)
    n = sum(layout.fc_pitch(d) for d in in_dims)
    if any(x is not None and (x.dtype != torch.float32 or x.numel() != n) for x in (theta, delta, m, v)):
        raise _lib.CevError(f"es_apply: theta / delta / m / v must be float32 [{n}]")
    opt = {"sgd": _lib.ES_SGD, "adam": _lib.ES_ADAM}[optimizer]
    dims = (ctypes.c_int * len(in_dims))(*[int(d) for d in in_dims])
    check(_call("cev_es_apply_f32", _h(dev), _ptr(theta), _ptr(delta), _ptr(m), _ptr(v), len(in_dims), dims, opt,
                float(lr), float(l2_coeff), int(t), _stream(dev)), "cev_es_apply_f32")
    return theta


def _need_f32(name, x, n):
    if x.dtype != torch.float32 or x.dim() != 1 or x.numel() != n:
        raise _lib.CevError(f"{name}: need a float32 [{n}] vector, got {tuple(x.shape)} {x.dtype}")


def es_perturb_diag(theta, sigma, in_dim, seed, role, gen, row0, n_rows, *, mirrored=False, out=None,
                    noise_out=None):
    """K5 of separable NES: member rows theta + fl(sigma * z) with the per-parameter sigma row fp32[pitch] (Linear
    parameters only).  z is the normal stream of :func:`es_perturb` (``mirrored`` False) or of
    :func:`es_perturb_mirrored` (True), so a sigma row of sigma0 gives their rows bit for bit; ``noise_out``
    receives s*z."""
    dev = _need_cuda(theta, sigma, out, noise_out)
    pitch = layout.fc_pitch(in_dim)
    _need_f32("es_perturb_diag: theta", theta, pitch)
    _need_f32("es_perturb_diag: sigma", sigma, pitch)
    for name, t in (("out", out), ("noise_out", noise_out)):
        if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != (int(n_rows), pitch)):
            raise _lib.CevError(f"es_perturb_diag: {name} must be float32 [{n_rows}, {pitch}]")
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    check(_call("cev_es_perturb_diag_f32", _h(dev), _ptr(theta), _ptr(sigma), int(in_dim), int(bool(mirrored)),
                int(seed), role_id, int(gen), int(row0), int(n_rows), pitch, _ptr(out), _ptr(noise_out),
                _stream(dev)), "cev_es_perturb_diag_f32")
    return out


def es_update_diag(fitness, in_dim, n_total, seed, role, gen, row0, *, mirrored=False, g_mu=None, g_sigma=None):
    """K6 of separable NES, noise regenerated: (g_mu, g_sigma) fp32[pitch] = 1/n_total * sum_i F_i z_i and
    1/n_total * sum_i F_i (z_i^2 - 1) over the local members [row0, row0 + len(fitness)), z the stream of
    :func:`es_perturb_diag` with the same ``mirrored``."""
    dev = _need_cuda(fitness, g_mu, g_sigma)
    if fitness.dtype != torch.float64 or fitness.dim() != 1:
        raise _lib.CevError("es_update_diag: fitness must be float64 [n_rows]")
    pitch = layout.fc_pitch(in_dim)
    g_mu = torch.empty(pitch, dtype=torch.float32, device=dev) if g_mu is None else g_mu
    g_sigma = torch.empty(pitch, dtype=torch.float32, device=dev) if g_sigma is None else g_sigma
    _need_f32("es_update_diag: g_mu", g_mu, pitch)
    _need_f32("es_update_diag: g_sigma", g_sigma, pitch)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    n = fitness.shape[0]
    check(_call("cev_es_update_diag_f32", _h(dev), ctypes.c_void_p(0) if n == 0 else _ptr(fitness), int(in_dim),
                int(bool(mirrored)), int(n_total), int(seed), role_id, int(gen), int(row0), n, _ptr(g_mu),
                _ptr(g_sigma), _stream(dev)), "cev_es_update_diag_f32")
    return g_mu, g_sigma


def es_apply_diag(theta, sigma, g_mu, g_sigma, in_dims, *, lr, sigma_lr, sigma_min, sigma_max):
    """Separable NES apply over the FCNetwork rows of ``in_dims`` concatenated in ``theta`` / ``sigma`` / ``g_mu`` /
    ``g_sigma``: theta += lr * (sigma * g_mu), then sigma *= exp(sigma_lr[s] / 2 * g_sigma) clamped to
    [sigma_min, sigma_max] (``sigma_lr``: one learning rate per row).  Only the Linear entries change."""
    dev = _need_cuda(theta, sigma, g_mu, g_sigma)
    n = sum(layout.fc_pitch(d) for d in in_dims)
    for name, x in (("theta", theta), ("sigma", sigma), ("g_mu", g_mu), ("g_sigma", g_sigma)):
        _need_f32(f"es_apply_diag: {name}", x, n)
    if len(sigma_lr) != len(in_dims):
        raise _lib.CevError("es_apply_diag: one sigma_lr per row")
    dims = (ctypes.c_int * len(in_dims))(*[int(d) for d in in_dims])
    etas = (ctypes.c_double * len(in_dims))(*[float(e) for e in sigma_lr])
    check(_call("cev_es_apply_diag_f32", _h(dev), _ptr(theta), _ptr(sigma), _ptr(g_mu), _ptr(g_sigma), len(in_dims),
                dims, float(lr), etas, float(sigma_min), float(sigma_max), _stream(dev)), "cev_es_apply_diag_f32")
    return theta, sigma


def es_hof_opponents(seed, gen, K, filled, newest, device, *, out=None):
    """Co-ES Hall of Fame: int64[K] archive slots of generation ``gen``'s opponent sets on the device.  Set 0 is
    ``newest`` (the current base agents); sets 1..K-1 are drawn uniformly with replacement from the ``filled``
    slots [0, filled) by the Philox stream of kind ``KIND_HOF`` keyed by (seed, gen), the same on every rank."""
    if out is None:
        out = torch.empty(int(K), dtype=torch.int64, device=device)
    dev = _need_cuda(out)
    if out.dtype != torch.int64 or tuple(out.shape) != (int(K),):
        raise _lib.CevError(f"es_hof_opponents: out must be int64 [{K}]")
    check(_call("cev_es_hof_opponents_i64", _h(dev), int(seed), int(gen), int(K), int(filled), int(newest), _ptr(out),
                _stream(dev)), "cev_es_hof_opponents_i64")
    return out


def es_perturb_subspace(theta, in_dim, sigma, U, k_eff, alpha, seed, role, gen, row0, n_rows, *, mirrored=False,
                        out=None, noise_out=None, coef_out=None):
    """K5 of guided search: member rows theta + sigma * eps with eps = A z + B U^T c on the Linear entries,
    A = fp32(sqrt(alpha)), B = fp32(sqrt((1 - alpha) d / k_eff)) (see ``cev_es_perturb_subspace_f32``).  ``U``: fp32
    [k, pitch] rows of the basis (contiguous rows, any row stride, e.g. the role's columns of a wider buffer);
    ``k_eff``: one-element int32 DEVICE tensor, the number of basis rows in use.  z is the stream of
    :func:`es_perturb` (``mirrored`` False) or :func:`es_perturb_mirrored` (True); ``noise_out`` receives s*z and
    ``coef_out`` fp32 [n_rows, k] the coefficients s*c, s = -1 for the odd member of a mirrored pair."""
    dev = _need_cuda(theta, k_eff, out, noise_out, coef_out)
    _need_rows(dev, U)
    pitch = layout.fc_pitch(in_dim)
    k = U.shape[0]
    _need_f32("es_perturb_subspace: theta", theta, pitch)
    if U.dtype != torch.float32 or U.shape[1] != pitch:
        raise _lib.CevError(f"es_perturb_subspace: U must be float32 [k, {pitch}]")
    if k_eff.dtype != torch.int32 or k_eff.numel() != 1:
        raise _lib.CevError("es_perturb_subspace: k_eff must be a one-element int32 tensor")
    for name, t, cols in (("out", out, pitch), ("noise_out", noise_out, pitch), ("coef_out", coef_out, k)):
        if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != (int(n_rows), cols)):
            raise _lib.CevError(f"es_perturb_subspace: {name} must be float32 [{n_rows}, {cols}]")
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    sig, sig_dev = _sigma_args(sigma)
    check(_call("cev_es_perturb_subspace_f32", _h(dev), _ptr(theta), int(in_dim), sig, sig_dev, _ptr(U), U.stride(0),
                int(k), _ptr(k_eff), float(alpha), int(bool(mirrored)), int(seed), role_id, int(gen), int(row0),
                int(n_rows), pitch, _ptr(out), _ptr(noise_out), _ptr(coef_out), _stream(dev)),
          "cev_es_perturb_subspace_f32")
    return out


def es_subspace_basis(ring, newest, filled, in_dims, *, out=None, k_eff=None):
    """Orthonormal basis of the guided-search subspace of each FCNetwork row of ``in_dims`` concatenated in ``ring``
    (fp32 [k, n]; slots [0, filled) filled, ``newest`` the newest estimate): CholeskyQR2 in fp64 over the estimates
    newest first, dropping an estimate whose residual norm is <= 1e-4 of its own norm.  Returns (U fp32 [k, n],
    k_eff int32 [len(in_dims)]) on the device (see ``cev_es_subspace_basis_f32``)."""
    dev = _need_cuda(ring, out, k_eff)
    k, n = ring.shape
    if ring.dtype != torch.float32 or n != sum(layout.fc_pitch(d) for d in in_dims):
        raise _lib.CevError("es_subspace_basis: ring must be float32 [k, summed pitch of in_dims]")
    out = torch.empty_like(ring) if out is None else out
    k_eff = torch.empty(len(in_dims), dtype=torch.int32, device=dev) if k_eff is None else k_eff
    if out.dtype != torch.float32 or out.shape != ring.shape:
        raise _lib.CevError(f"es_subspace_basis: out must be float32 [{k}, {n}]")
    if k_eff.dtype != torch.int32 or k_eff.numel() != len(in_dims):
        raise _lib.CevError(f"es_subspace_basis: k_eff must be int32 [{len(in_dims)}]")
    dims = (ctypes.c_int * len(in_dims))(*[int(d) for d in in_dims])
    check(_call("cev_es_subspace_basis_f32", _h(dev), _ptr(ring), int(k), int(newest), int(filled), len(in_dims),
                dims, _ptr(out), _ptr(k_eff), _stream(dev)), "cev_es_subspace_basis_f32")
    return out, k_eff


def _need_status(name, status):
    if status is not None and (status.dtype != torch.int32 or status.numel() != 1):
        raise _lib.CevError(f"{name}: status must be a one-element int32 tensor")


def _need_sigma_dev(name, sigma):
    if not (isinstance(sigma, torch.Tensor) and sigma.dtype == torch.float64 and sigma.numel() == 1):
        raise _lib.CevError(f"{name}: sigma must be a one-element float64 device tensor (the generation state slot)")


def es_lmma_project(M, k, G, cd, in_dim, seed, role, gen, row0, n_rows, *, beta=None, s_out=None, status=None):
    """LM-MA-ES projection and transform coefficients (see ``cev_es_lmma_project_f32``): s = M[:k] z_i in fp64 for the
    members [row0, row0 + n_rows) (z the stream of :func:`es_perturb`), then the compact form of the sequential
    transform with the Gram ``G`` fp64 [m, m] and ``cd`` (host, the k values c_d,j).  ``M``: fp32 [>= k, pitch] rows
    (contiguous rows, any row stride).  Returns beta fp32 [n_rows, k]; ``s_out`` (optional) receives s fp64
    [n_rows, k]; a non-finite s or beta sets ``status``."""
    dev = _need_cuda(G, beta, s_out, status)
    _need_rows(dev, M)
    pitch = layout.fc_pitch(in_dim)
    k, n_rows = int(k), int(n_rows)
    if M.dtype != torch.float32 or M.shape[1] != pitch or not 1 <= k <= min(M.shape[0], _lib.SUBSPACE_MAX_DIM):
        raise _lib.CevError(f"es_lmma_project: M must be float32 [>= k, {pitch}] and 1 <= k <= 32")
    if G.dtype != torch.float64 or G.dim() != 2 or G.shape[0] != G.shape[1] or G.shape[0] < k:
        raise _lib.CevError("es_lmma_project: G must be float64 [m, m] with m >= k")
    if len(cd) != k:
        raise _lib.CevError(f"es_lmma_project: need k = {k} values of c_d")
    for name, t, dt in (("beta", beta, torch.float32), ("s_out", s_out, torch.float64)):
        if t is not None and (t.dtype != dt or tuple(t.shape) != (n_rows, k)):
            raise _lib.CevError(f"es_lmma_project: {name} must be {dt} [{n_rows}, {k}]")
    _need_status("es_lmma_project", status)
    if beta is None:
        beta = torch.empty((n_rows, k), dtype=torch.float32, device=dev)
    n_chunks = -(-layout.fc_dim(in_dim) // _lib.LMMA_PROJECT_CHUNK)
    part = torch.empty(max(n_chunks * n_rows * k, 1), dtype=torch.float64, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    cd_arr = (ctypes.c_double * k)(*[float(c) for c in cd])
    check(_call("cev_es_lmma_project_f32", _h(dev), _ptr(M), M.stride(0), k, _ptr(G), G.shape[0], cd_arr, int(in_dim),
                int(seed), role_id, int(gen), int(row0), n_rows, _ptr(part), _ptr(beta), _ptr(s_out), _ptr(status),
                _stream(dev), launches=2), "cev_es_lmma_project_f32")
    return beta


def es_perturb_lmma(theta, in_dim, sigma, M, k, beta, alpha, seed, role, gen, row0, n_rows, *, out=None):
    """LM-MA K5 (see ``cev_es_perturb_lmma_f32``): member rows theta + fl(sigma eps) with eps = fl(fl(fp32(alpha) z) +
    sum_{l < k} fl(M[l] beta_l)) on the Linear entries, z the stream of :func:`es_perturb`.  ``sigma``: the
    one-element fp64 DEVICE slot; ``beta``: fp32 [n_rows, k] from :func:`es_lmma_project`."""
    dev = _need_cuda(theta, sigma, beta, out)
    _need_rows(dev, M)
    _need_sigma_dev("es_perturb_lmma", sigma)
    pitch = layout.fc_pitch(in_dim)
    k, n_rows = int(k), int(n_rows)
    _need_f32("es_perturb_lmma: theta", theta, pitch)
    if M.dtype != torch.float32 or M.shape[1] != pitch or not 1 <= k <= min(M.shape[0], _lib.SUBSPACE_MAX_DIM):
        raise _lib.CevError(f"es_perturb_lmma: M must be float32 [>= k, {pitch}] and 1 <= k <= 32")
    if beta.dtype != torch.float32 or tuple(beta.shape) != (n_rows, k):
        raise _lib.CevError(f"es_perturb_lmma: beta must be float32 [{n_rows}, {k}]")
    if out is not None and (out.dtype != torch.float32 or tuple(out.shape) != (n_rows, pitch)):
        raise _lib.CevError(f"es_perturb_lmma: out must be float32 [{n_rows}, {pitch}]")
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    check(_call("cev_es_perturb_lmma_f32", _h(dev), _ptr(theta), int(in_dim), _ptr(sigma), _ptr(M), M.stride(0), k,
                _ptr(beta), float(alpha), int(seed), role_id, int(gen), int(row0), n_rows, pitch, _ptr(out),
                _stream(dev)), "cev_es_perturb_lmma_f32")
    return out


def es_lmma_reduce(ids, w, beta, in_dim, seed, role, gen, row0, n_rows, *, zbar=None, betabar=None):
    """LM-MA weighted recombination over this rank's rows (see ``cev_es_lmma_reduce_f32``): ``ids`` int64 [mu] the
    selected members best first, ``w`` fp32 [mu] their weights, ``beta`` fp32 [n_rows, k] (k may be 0).  Returns
    (zbar fp32 [pitch], betabar fp32 [k]), this rank's share of sum_i w_i z_(i) and sum_i w_i beta_(i)."""
    dev = _need_cuda(ids, w, beta if beta.numel() else None, zbar, betabar)
    pitch = layout.fc_pitch(in_dim)
    mu, k = ids.numel(), beta.shape[1]
    if ids.dtype != torch.int64 or w.dtype != torch.float32 or w.numel() != mu or mu < 1:
        raise _lib.CevError("es_lmma_reduce: ids must be int64 [mu >= 1] and w float32 [mu]")
    if beta.dtype != torch.float32 or beta.dim() != 2 or beta.shape[0] != int(n_rows) or k > _lib.SUBSPACE_MAX_DIM:
        raise _lib.CevError(f"es_lmma_reduce: beta must be float32 [{n_rows}, k <= 32]")
    zbar = torch.empty(pitch, dtype=torch.float32, device=dev) if zbar is None else zbar
    betabar = torch.empty(k, dtype=torch.float32, device=dev) if betabar is None else betabar
    _need_f32("es_lmma_reduce: zbar", zbar, pitch)
    _need_f32("es_lmma_reduce: betabar", betabar, k)
    part = torch.empty(_lib.LMMA_REDUCE_SPLIT * pitch, dtype=torch.float64, device=dev)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    check(_call("cev_es_lmma_reduce_f32", _h(dev), _ptr(ids), _ptr(w), mu, _ptr(beta) if k else ctypes.c_void_p(0), k,
                int(in_dim), int(seed), role_id, int(gen), int(row0), int(n_rows), _ptr(part), _ptr(zbar),
                _ptr(betabar) if k else ctypes.c_void_p(0), _stream(dev), launches=2), "cev_es_lmma_reduce_f32")
    return zbar, betabar


def es_lmma_apply(theta, M, p, zbar, betabar, in_dims, *, k, alpha, c_sigma, mu_w, c_m, c_c, G, gstate, sigma_min,
                  sigma_max, stats=None, status=None):
    """LM-MA apply over the FCNetwork rows of ``in_dims`` concatenated in ``theta`` / ``p`` / ``zbar`` (fp32 [n]) and
    the rows of ``M`` (fp32 [m, n]); see ``cev_es_lmma_apply_f32``.  ``betabar`` fp32 [len(in_dims), m] (the first k of
    each row used); ``alpha``, ``c_sigma``, ``mu_w``: one per row; ``c_c``: [len(in_dims)][m].  Steps theta with the old
    M, updates p and every vector, writes the new Gram into ``G`` fp64 [len(in_dims), m, m] and the adapted sigma into
    the generation state ``gstate``.  Returns ``stats`` fp64 [len(in_dims), 2] = (|p|^2 / n, sigma after)."""
    dev = _need_cuda(theta, M, p, zbar, betabar, G, gstate, stats, status)
    n = sum(layout.fc_pitch(d) for d in in_dims)
    ns = len(in_dims)
    m = M.shape[0]
    for name, x in (("theta", theta), ("p", p), ("zbar", zbar)):
        _need_f32(f"es_lmma_apply: {name}", x, n)
    if M.dtype != torch.float32 or tuple(M.shape) != (m, n) or not 1 <= m <= _lib.SUBSPACE_MAX_DIM:
        raise _lib.CevError(f"es_lmma_apply: M must be float32 [m <= 32, {n}]")
    if betabar.dtype != torch.float32 or betabar.numel() != ns * m:
        raise _lib.CevError(f"es_lmma_apply: betabar must be float32 [{ns}, {m}]")
    if G.dtype != torch.float64 or tuple(G.shape) != (ns, m, m):
        raise _lib.CevError(f"es_lmma_apply: G must be float64 [{ns}, {m}, {m}]")
    if gstate.dtype != torch.float64:
        raise _lib.CevError("es_lmma_apply: gstate must be float64")
    if not 0 <= int(k) <= m or any(len(x) != ns for x in (alpha, c_sigma, mu_w, c_c)) or any(len(c) != m for c in c_c):
        raise _lib.CevError("es_lmma_apply: need 0 <= k <= m and one alpha / c_sigma / mu_w / c_c row per row")
    _need_status("es_lmma_apply", status)
    if stats is None:
        stats = torch.empty((ns, 2), dtype=torch.float64, device=dev)
    n_chunks = -(-max(layout.fc_pitch(d) for d in in_dims) // _lib.LMMA_APPLY_CHUNK)
    part = torch.empty(ns * n_chunks * (m * (m + 1) // 2 + 1), dtype=torch.float64, device=dev)

    def arr(vals):
        return (ctypes.c_double * len(vals))(*[float(v) for v in vals])
    dims = (ctypes.c_int * ns)(*[int(d) for d in in_dims])
    check(_call("cev_es_lmma_apply_f32", _h(dev), _ptr(theta), _ptr(M), m, int(k), _ptr(p), _ptr(zbar), _ptr(betabar),
                ns, dims, arr(alpha), arr(c_sigma), arr(mu_w), float(c_m), arr([c for row in c_c for c in row]), _ptr(G),
                _ptr(gstate), float(sigma_min), float(sigma_max), _ptr(part), _ptr(stats), _ptr(status), _stream(dev),
                launches=2), "cev_es_lmma_apply_f32")
    return stats


def novelty_probe_obs(init, role, *, out=None):
    """Probe observations of the novelty search: fp32 [n, in_dim] = what ``role`` observes in the world state of each
    initial-state record of ``init`` fp64 [n, 11] (zero velocities), bit for bit the rollout's observation."""
    dev = _need_cuda(init, out)
    if init.dtype != torch.float64 or init.dim() != 2 or init.shape[1] != _lib.INIT_STATE_DIM:
        raise _lib.CevError(f"novelty_probe_obs: init must be float64 [n, {_lib.INIT_STATE_DIM}]")
    in_dim, n = layout.OBS_DIM[role], init.shape[0]
    if out is None:
        out = torch.empty((n, in_dim), dtype=torch.float32, device=dev)
    if out.dtype != torch.float32 or tuple(out.shape) != (n, in_dim):
        raise _lib.CevError(f"novelty_probe_obs: out must be float32 [{n}, {in_dim}]")
    check(_call("cev_novelty_probe_obs_f32", _h(dev), _ptr(init), n, layout.SEAT_OF[role], _ptr(out), _stream(dev)),
          "cev_novelty_probe_obs_f32")
    return out


def novelty_bc(rows, in_dim, probe_obs, *, out=None, status=None):
    """Behaviour characterisation of the novelty search: fp32 [P, 160], row m = the softmax action distributions of
    network row m on the 32 probe observations ``probe_obs`` fp32 [32, in_dim], probe after probe.  ``rows``: fp32
    [P, >= fc_dim] with contiguous rows (any row stride that is a multiple of 4, e.g. a view of a wider buffer);
    ``out``: fp32 [P, 160] with contiguous rows (e.g. a slot of the archive ring).  A non-finite logit sets ``status``."""
    dev = _need_cuda(probe_obs, status)
    _need_rows(dev, rows)
    P = rows.shape[0]
    if rows.dtype != torch.float32 or rows.shape[1] < layout.fc_dim(in_dim) or (P and rows.stride(0) % 4):
        raise _lib.CevError(f"novelty_bc: rows must be float32 [P, >= {layout.fc_dim(in_dim)}], row stride a "
                            "multiple of 4")
    if probe_obs.dtype != torch.float32 or tuple(probe_obs.shape) != (_lib.NOVELTY_PROBES, in_dim):
        raise _lib.CevError(f"novelty_bc: probe_obs must be float32 [{_lib.NOVELTY_PROBES}, {in_dim}]")
    if out is None:
        out = torch.empty((P, _lib.NOVELTY_BC_DIM), dtype=torch.float32, device=dev)
    _need_rows(dev, out)
    if out.dtype != torch.float32 or tuple(out.shape) != (P, _lib.NOVELTY_BC_DIM):
        raise _lib.CevError(f"novelty_bc: out must be float32 [{P}, {_lib.NOVELTY_BC_DIM}]")
    if P == 0:
        return out
    check(_call("cev_novelty_bc_f32", _h(dev), _ptr(rows), rows.stride(0), int(in_dim), P, _ptr(probe_obs), _ptr(out),
                out.stride(0), _ptr(status), _stream(dev)), "cev_novelty_bc_f32")
    return out


def novelty_knn(bc, ring, filled, k, *, out=None):
    """k-NN novelty: fp64 [n], entry i = the mean of the min(k, filled) smallest Euclidean distances (fp64) from
    ``bc[i]`` fp32 [n, 160] to the archive entries ``ring[:filled]`` fp32 [A, 160]."""
    dev = _need_cuda(bc, ring, out)
    D = _lib.NOVELTY_BC_DIM
    if bc.dtype != torch.float32 or bc.dim() != 2 or bc.shape[1] != D:
        raise _lib.CevError(f"novelty_knn: bc must be float32 [n, {D}]")
    if ring.dtype != torch.float32 or ring.dim() != 2 or ring.shape[1] != D:
        raise _lib.CevError(f"novelty_knn: ring must be float32 [A, {D}]")
    if not 1 <= int(filled) <= ring.shape[0]:
        raise _lib.CevError(f"novelty_knn: filled must be in [1, {ring.shape[0]}], not {filled}")
    if not 1 <= int(k) <= _lib.NOVELTY_MAX_K:
        raise _lib.CevError(f"novelty_knn: k must be in [1, {_lib.NOVELTY_MAX_K}], not {k}")
    n = bc.shape[0]
    if out is None:
        out = torch.empty(n, dtype=torch.float64, device=dev)
    if out.dtype != torch.float64 or tuple(out.shape) != (n,):
        raise _lib.CevError(f"novelty_knn: out must be float64 [{n}]")
    if n == 0:
        return out
    check(_call("cev_novelty_knn_f64", _h(dev), _ptr(bc), n, _ptr(ring), int(filled), int(k), _ptr(out), _stream(dev)),
          "cev_novelty_knn_f64")
    return out


def _need_bc_rows(name, what, t, dev):
    """Characterisation rows handed to a kernel with their ``stride(0)`` as the row pitch."""
    D = _lib.NOVELTY_BC_DIM
    if not t.is_cuda or t.device != dev:
        raise _lib.CevError(f"{name}: {what} must be a CUDA tensor on the device of the other operands")
    if t.dtype != torch.float32 or t.dim() != 2 or t.shape[1] != D or t.stride(1) != 1 or \
            (t.shape[0] and (t.stride(0) % 4 or t.data_ptr() % 16)):
        raise _lib.CevError(f"{name}: {what} must be float32 [rows, {D}] with contiguous rows, a row stride that is a "
                            "multiple of 4 and 16-byte alignment")


def ga_novelty_knn(x, row0, pop, ring, filled, k, *, splits=0, out=None):
    """Co-GA k-NN novelty: fp64 [n], entry i = the mean of the k_eff = min(k, P - 1 + filled) smallest fp32
    Euclidean distances from ``x[i]`` (the characterisation of global row ``row0 + i``) to the other population
    rows ``pop`` fp32 [P, 160] and the archive slots ``ring[:filled]`` fp32 [A, 160], summed in fp64 in ascending
    order of (distance, index) (``cev_ga_novelty_knn_f64``).  ``x`` / ``pop``: contiguous rows, any row stride
    that is a multiple of 4 (e.g. one role's column of a gathered [P, 3, 160] block).  ``splits``: candidate
    ranges searched by separate CTAs (0 = chosen from the shape); the result does not depend on it."""
    dev = _need_cuda(ring, out)
    if dev is None:
        raise _lib.CevError("ga_novelty_knn: needs CUDA tensors (no CPU fallback)")
    _need_bc_rows("ga_novelty_knn", "x", x, dev)
    _need_bc_rows("ga_novelty_knn", "pop", pop, dev)
    D = _lib.NOVELTY_BC_DIM
    if ring.dtype != torch.float32 or ring.dim() != 2 or ring.shape[1] != D:
        raise _lib.CevError(f"ga_novelty_knn: ring must be float32 [A, {D}]")
    n, P = x.shape[0], pop.shape[0]
    if P < 1:
        raise _lib.CevError("ga_novelty_knn: the population needs at least one row")
    if not 0 <= int(filled) <= min(ring.shape[0], _lib.NOVELTY_MAX_ARCHIVE):
        raise _lib.CevError(f"ga_novelty_knn: filled must be in [0, {min(ring.shape[0], _lib.NOVELTY_MAX_ARCHIVE)}], "
                            f"not {filled}")
    if P - 1 + int(filled) < 1:
        raise _lib.CevError("ga_novelty_knn: a member needs at least one other candidate (P = 1 needs filled >= 1)")
    if not 1 <= int(k) <= _lib.NOVELTY_MAX_K:
        raise _lib.CevError(f"ga_novelty_knn: k must be in [1, {_lib.NOVELTY_MAX_K}], not {k}")
    if not 0 <= int(row0) <= P - n:
        raise _lib.CevError(f"ga_novelty_knn: rows [row0, row0 + {n}) must lie in [0, {P}), row0 = {row0}")
    if int(splits) < 0:
        raise _lib.CevError(f"ga_novelty_knn: splits must be >= 0, not {splits}")
    if out is None:
        out = torch.empty(n, dtype=torch.float64, device=dev)
    if out.dtype != torch.float64 or tuple(out.shape) != (n,):
        raise _lib.CevError(f"ga_novelty_knn: out must be float64 [{n}]")
    if n == 0:
        return out
    check(_call("cev_ga_novelty_knn_f64", _h(dev), _ptr(x), x.stride(0), n, int(row0), _ptr(pop), pop.stride(0), P,
                _ptr(ring), int(filled), int(k), int(splits), _ptr(out), _stream(dev)),
          "cev_ga_novelty_knn_f64")
    return out


def ga_novelty_draw(seed, gen, role, m, P, device, *, out=None):
    """Co-GA novelty archive: int64 [m] population ids in [0, P) whose characterisations enter ``role``'s archive
    after generation ``gen``'s selection, in draw order, from the Philox stream of kind ``KIND_GA_NOVELTY`` keyed
    by (seed, gen, role), the same on every rank."""
    if out is None:
        out = torch.empty(int(m), dtype=torch.int64, device=device)
    dev = _need_cuda(out)
    if dev is None:
        raise _lib.CevError("ga_novelty_draw: needs a CUDA device (no CPU fallback)")
    if out.dtype != torch.int64 or tuple(out.shape) != (int(m),):
        raise _lib.CevError(f"ga_novelty_draw: out must be int64 [{m}]")
    if not 1 <= int(P) <= 1 << 32:
        raise _lib.CevError(f"ga_novelty_draw: P must be in [1, 2^32], not {P}")
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    check(_call("cev_ga_novelty_draw_i64", _h(dev), int(seed), int(gen), role_id, int(m), int(P), _ptr(out),
                _stream(dev)), "cev_ga_novelty_draw_i64")
    return out


def ga_safe_scale(elites, in_dim, probe_obs, floor, *, out=None, status=None):
    """Safe-mutation scales (SM-G-SUM): fp32 [E, pitch], entry j of row e = 1 / max(s_j, floor), or 1 where s_j = 0,
    with s_j = sqrt(sum_k (sum_t dy_k(x_t) / dW_j)^2) the response of the 5 logits of network row ``elites[e]`` to
    parameter j on the 32 probe observations ``probe_obs`` fp32 [32, in_dim]; padding entries are 0
    (``cev_ga_safe_scale_f32``).  ``elites``: fp32 [E, pitch >= fc_dim] with contiguous rows, 16-byte aligned.
    A non-finite logit or gradient sets ``status``."""
    dev = _need_cuda(probe_obs, status)
    _need_rows(dev, elites)
    E, D = elites.shape[0], layout.fc_dim(in_dim)
    if in_dim not in (8, 10):
        raise _lib.CevError(f"ga_safe_scale: in_dim must be 8 or 10, not {in_dim}")
    if elites.dtype != torch.float32 or elites.shape[1] < D or (E and (elites.stride(0) % 4 or elites.data_ptr() % 16)):
        raise _lib.CevError(f"ga_safe_scale: elites must be float32 [E, >= {D}], row stride a multiple of 4, "
                            "16-byte aligned")
    if probe_obs.dtype != torch.float32 or tuple(probe_obs.shape) != (_lib.NOVELTY_PROBES, in_dim):
        raise _lib.CevError(f"ga_safe_scale: probe_obs must be float32 [{_lib.NOVELTY_PROBES}, {in_dim}]")
    f = float(floor)
    if not (math.isfinite(f) and f > 0.0):
        raise _lib.CevError(f"ga_safe_scale: floor must be finite and > 0, not {floor}")
    if out is None:
        out = torch.empty((E, elites.shape[1]), dtype=torch.float32, device=dev)
    _need_rows(dev, out)
    if out.dtype != torch.float32 or out.shape[0] != E or out.shape[1] < D or (E and out.stride(0) % 4):
        raise _lib.CevError(f"ga_safe_scale: out must be float32 [{E}, >= {D}], row stride a multiple of 4")
    if status is not None and (status.dtype != torch.int32 or status.numel() != 1):
        raise _lib.CevError("ga_safe_scale: status must be a one-element int32 tensor")
    if E == 0:
        return out
    check(_call("cev_ga_safe_scale_f32", _h(dev), _ptr(elites), elites.stride(0), int(in_dim), E, _ptr(probe_obs),
                f, _ptr(out), out.stride(0), _ptr(status), _stream(dev)), "cev_ga_safe_scale_f32")
    return out


def axpy(a, x, y):
    dev = _need_cuda(x, y)
    check(_call("cev_axpy_f32", _h(dev), float(a), _ptr(x), _ptr(y), min(x.numel(), y.numel()),
                              _stream(dev)), "cev_axpy_f32")
    return y


def diversity_dist(pop, ref, in_dim, *, out=None):
    """K7: fp32[P] distances || pop[i] - ref || over the Linear parameters."""
    dev = _need_cuda(ref, out, pop if pop.numel() else None)
    if out is None:
        out = torch.empty(pop.shape[0], dtype=torch.float32, device=dev)
    if pop.shape[0] == 0:
        return out
    check(_call("cev_diversity_dist_f32", _h(dev), _ptr(pop), pop.shape[0], pop.stride(0),
                                        _ptr(ref), int(in_dim), _ptr(out), _stream(dev)),
          "cev_diversity_dist_f32")
    return out


def diversity_from_dist(dist):
    """The scalar of ``diversity_penalty`` (``utils/game_logic_functions.py:22-37``)
    from the distances: sigma = mean(d), sum(max(0, 1 - d/sigma)).  P scalars of
    glue arithmetic, done with torch on the device."""
    sigma = dist.mean()
    return torch.clamp(1 - dist / sigma, min=0).sum()


def deepqn_forward(members, frames, c_in, n_actions):
    """K2: logits fp32[P,B,A] and first-max actions int32[P,B].  ``members`` fp32[P, >= dqn_dim] with
    contiguous rows; the row pitch is ``stride(0)`` (rows of a wider buffer qualify)."""
    dev = _need_cuda(frames)
    _need_rows(dev, members)
    P, B = frames.shape[0], frames.shape[1]
    if frames.dtype != torch.uint8 or tuple(frames.shape[2:]) != (c_in, 84, 84):
        raise _lib.CevError("deepqn_forward: frames must be uint8 [P,B,C,84,84]")
    if members.dtype != torch.float32 or members.shape[0] != P or members.shape[1] < layout.dqn_dim(c_in, n_actions):
        raise _lib.CevError("deepqn_forward: members must be fp32 [P, >= dqn_dim(c_in, n_actions)]")
    logits = torch.empty((P, B, n_actions), dtype=torch.float32, device=dev)
    actions = torch.empty((P, B), dtype=torch.int32, device=dev)
    if P == 0:
        return logits, actions
    check(_call("cev_deepqn_forward", _h(dev), _ptr(members), P, members.stride(0),
                                    _ptr(frames), B, int(c_in), int(n_actions), _ptr(logits),
                                    _ptr(actions), _stream(dev)), "cev_deepqn_forward")
    return logits, actions


def atari_synth_step(seed, ep0, ring, t, a_first=None, a_second=None, *, reward_out=None):
    """Synthetic emulator step: frame ``t`` of every episode into slot t % 4 of ``ring`` (u8 [n, 4, 7056]);
    returns the zero-sum reward r_first fp32[n] of the step (None for t = 0)."""
    dev = _need_cuda(ring, a_first, a_second, reward_out)
    n = ring.shape[0]
    if ring.dtype != torch.uint8 or tuple(ring.shape[1:]) != (4, 7056):
        raise _lib.CevError("atari_synth_step: ring must be uint8 [n, 4, 7056]")
    if t > 0:
        if a_first is None or a_second is None or a_first.dtype != torch.int32 or a_second.dtype != torch.int32:
            raise _lib.CevError("atari_synth_step: int32 actions of both agents are needed for t >= 1")
        if reward_out is None:
            reward_out = torch.empty(n, dtype=torch.float32, device=dev)
    check(_call("cev_atari_synth_step_u8", _h(dev), int(seed), int(ep0), n, int(t), _ptr(a_first), _ptr(a_second),
                _ptr(ring), _ptr(reward_out), _stream(dev)), "cev_atari_synth_step_u8")
    return reward_out


def atari_observe(ring, t, seat, *, out=None):
    """What agent ``seat`` (0 first_0, 1 second_0) observes after ``t`` emulator steps: u8 [n, 6, 84, 84]
    (4 stacked frames, oldest first, + 2 agent-indicator planes)."""
    dev = _need_cuda(ring, out)
    n = ring.shape[0]
    if out is None:
        out = torch.empty((n, 6, 84, 84), dtype=torch.uint8, device=dev)
    check(_call("cev_atari_observe_u8", _h(dev), _ptr(ring), n, int(t), int(seat), _ptr(out), _stream(dev)),
          "cev_atari_observe_u8")
    return out


def fc_init(in_dim, seed, role, row0, n_rows, device, *, out=None):
    """Device-side founders: float32[n_rows, pitch] rows with PyTorch's default-init
    distribution (Philox stream; global member ids row0 .. row0+n_rows-1)."""
    pitch = layout.fc_pitch(in_dim)
    if out is None:
        out = torch.empty((n_rows, pitch), dtype=torch.float32, device=device)
    dev = _need_cuda(out)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    check(_call("cev_fc_init_f32", _h(dev), int(in_dim), int(seed), role_id, int(row0), int(n_rows),
                pitch, _ptr(out), _stream(dev)), "cev_fc_init_f32")
    return out


def init_states(seed, stream_id, n, device, rec0=0):
    """Device-generated initial env states fp64[n,11] (Appendix A.3 distribution):
    records rec0 .. rec0+n-1 of Philox stream ``stream_id``."""
    out = torch.empty((n, _lib.INIT_STATE_DIM), dtype=torch.float64, device=device)
    dev = out.device
    check(_call("cev_init_states_f64", _h(dev), int(seed), int(stream_id), int(rec0), n, _ptr(out),
                                     _stream(dev)), "cev_init_states_f64")
    return out


def random_frames(seed, shape, device):
    out = torch.empty(shape, dtype=torch.uint8, device=device)
    if out.numel() % 16:
        raise _lib.CevError("random_frames: byte count must be a multiple of 16")
    dev = out.device
    check(_call("cev_random_frames_u8", _h(dev), int(seed), out.numel(), _ptr(out),
                                      _stream(dev)), "cev_random_frames_u8")
    return out


def philox_words(seed, kind, role, gen, member0, n_members, n4, device):
    out = torch.empty((n_members, n4, 4), dtype=torch.int32, device=device)
    dev = out.device
    check(_call("cev_philox_words", _h(dev), int(seed), int(kind), int(role), int(gen),
                                  int(member0), int(n_members), int(n4), _ptr(out), _stream(dev)),
          "cev_philox_words")
    return out


def fp32_peak(device, mode=1):
    """Measured FP32 FMA-pipe peak in TFLOP/s (mode 0 scalar FFMA, 1 packed FFMA2)."""
    dev = torch.device(device)
    val = ctypes.c_double()
    check(_call("cev_fp32_peak", _h(dev), int(mode), ctypes.byref(val), _stream(dev)),
          "cev_fp32_peak")
    return val.value
