"""K2, the grouped DeepQN forward, at the population sizes it runs at, on all three paths, against the float64
oracle.

Every K2 kernel is persistent and loops over jobs: the convolution kernels run min(P*B, n_sm) CTAs over frames,
the tensor-core fc stage min(P, n_sm) CTAs over members (frame blocks of 16 inside a member), the fp32 kernel
min(P, n_sm) CTAs over members.  These shapes make CTAs run second and later jobs; each is checked four ways:
a. the frames of every later job and of the last, ragged wave (at most REF_CAP of them) against the float64
   oracle, within SCALE_TOL x max(1, max|logit|) of the frame;
b. every frame bit for bit against launches cut into chunks in which every CTA runs one job of one frame block,
   the regime (a) and the smaller tests validate (a frame's logits do not depend on its neighbours);
c. a second launch bit for bit;
d. every action is the first-max argmax of the returned logits, and the float64 argmax where the float64
   top-2 gap exceeds twice the tolerance.
The members are ES perturbations (sigma 0.05, as BASELINE config 5) of one row whose BatchNorm gammas include
negative ones."""
import numpy as np
import pytest
import torch

from conftest import parity_report
from oracle import deepqn as odqn
from oracle import layout as olayout
from oracle import weights
from test_gpu_deepqn import FC_MODES, _pad, fc_mode  # noqa: F401  (fc_mode: the three K2 paths)

pytestmark = pytest.mark.gpu

# Bounds on |logit - float64| / max(1, max|logit|) of the frame.  The ES members (sigma 0.05, three times the
# fc1 init bound) have logits up to ~10.  The fp32 path stays within the suite's 2e-5 there.  The tensor-core fc
# stage does not: its MMAs accumulate fp32 with truncated alignment, not round-to-nearest (Fasi et al., "Numerical
# behavior of NVIDIA tensor cores", 2021), so the error of fc1 grows with the 392 k-steps of K = 3136 and with the
# partial sums, up to 392 * 2^-23 = 4.7e-5 of them.  Observed on a B200: <= 7e-6 (fp32), <= 3.1e-5 (tensor-core
# fc); the fc and conv mutations of 2xTF32 give >= 6e-4.
SCALE_TOL = {"conv_fp32": 6e-5, "fp32": 2e-5, "tc": 6e-5}
SIGMA = 0.05
BN_JITTER = 0.7       # gamma = 1 + 0.7 N(0, 1): about 8 % of them negative
REF_CAP = 200         # frames per shape held to the float64 oracle (a few ms each on the host)
NB = 16               # frames per frame block of the fc stage

# name: (c_in, n_actions, P as a function of n_sm, B, frames, extra floats of row pitch)
SHAPES = {
    "config4_B1": (4, 6, lambda n: 592, 1, "random", 0),
    "config4_B4": (4, 6, lambda n: 592, 4, "random", 0),          # 16 frames per conv CTA, 4 members per fc CTA
    "ragged_waves": (6, 18, lambda n: 2 * n + 3, 17, "random", 0),  # 2 and 3 members per CTA, a 1-frame block
    "opponent_call": (6, 18, lambda n: 1, 300, "atari", 0),       # atari_rollout's opponent: 19 blocks, one CTA
    "actions_1": (4, 1, lambda n: n + 1, 2, "random", 0),
    "actions_17": (4, 17, lambda n: n + 1, 2, "random", 0),
    "actions_32": (4, 32, lambda n: n + 1, 2, "random", 0),
    "row_pitch": (4, 6, lambda n: n + 2, 3, "random", 32),        # rows of a wider buffer
}


def _n_sm(device=0):
    return torch.cuda.get_device_properties(device).multi_processor_count


def _members(c_in, n_act, P, seed, extra_pitch=0, device="cuda"):
    """P distinct members theta + SIGMA z (conv / Linear entries; BatchNorm entries copied), as rows of a buffer
    whose pitch is dqn_pitch + extra_pitch; the extra floats are NaN, so reading them poisons the logits."""
    from coevonet_b200 import layout, ops
    total, dp = layout.dqn_dim(c_in, n_act), layout.dqn_pitch(c_in, n_act)
    base = weights.make_dqn_rows(1, c_in, n_act, seed, bn_jitter=BN_JITTER)[0]
    assert (olayout.unpack_dqn(base, c_in, n_act)["vbn1.weight"] < 0).any()
    theta = torch.zeros(dp, device=device)
    theta[:total] = torch.from_numpy(base).to(device)
    rows = ops.es_perturb_dqn(theta, c_in, n_act, SIGMA, seed, "agent_0", 5, 0, P)
    if not extra_pitch:
        return rows
    buf = torch.full((P, dp + extra_pitch), float("nan"), device=device)
    buf[:, :dp] = rows
    return buf[:, :dp]


def _frames(kind, P, B, c_in, n_act, seed):
    from coevonet_b200 import ops
    if kind == "random":
        return ops.random_frames(seed, (P, B, c_in, 84, 84), "cuda")
    # what atari_rollout hands the opponent's forward after one emulator step: P*E observations of one seat
    # (two zero planes of the not yet filled frame stack, two emulator frames, two constant indicator planes)
    assert P == 1 and c_in == 6
    ring = torch.zeros((B, 4, 84 * 84), dtype=torch.uint8, device="cuda")
    ops.atari_synth_step(seed, 0, ring, 0)
    g = torch.Generator().manual_seed(seed)
    a_first, a_second = (torch.randint(0, n_act, (B,), generator=g, dtype=torch.int32).cuda() for _ in range(2))
    ops.atari_synth_step(seed, 0, ring, 1, a_first, a_second)
    return ops.atari_observe(ring, 1, 1).reshape(1, B, c_in, 84, 84)


def _spread(idx, k):
    """At most k entries of idx, evenly spaced, both ends included."""
    if len(idx) <= k:
        return idx
    return idx[np.unique(np.linspace(0, len(idx) - 1, k).round().astype(np.int64))]


def _subset(P, B, n_sm, cap=REF_CAP):
    """Flat frame indices m * B + f to hold to the float64 oracle: the frames of the last, ragged wave of the
    conv kernels (frames) and of the fc stage (members), and the frames some CTA runs as a second or later job."""
    g = np.arange(P * B)
    m = g // B
    ragged = np.zeros(P * B, dtype=bool)
    if P % n_sm:
        ragged |= m >= P // n_sm * n_sm
    if P * B % n_sm:
        ragged |= g >= P * B // n_sm * n_sm
    later = np.flatnonzero(((g >= n_sm) | (m >= n_sm)) & ~ragged)
    first = _spread(np.flatnonzero(ragged), cap // 2 if len(later) else cap)
    return np.sort(np.concatenate([first, _spread(later, cap - len(first))]))


def _reference(members, frames, sel, c_in, n_act):
    """float64 oracle logits [len(sel), A] of the flat frames sel."""
    P, B = frames.shape[:2]
    fr = frames.reshape(P * B, c_in, 84, 84)[torch.from_numpy(sel).to(frames.device)].cpu().numpy()
    ref = np.empty((len(sel), n_act))
    for m in np.unique(sel // B):
        row = members[int(m)].cpu().numpy()
        for j in np.flatnonzero(sel // B == m):
            ref[j] = odqn.dqn_forward(row, fr[j], c_in, n_act, np.float64)
    return ref


def _check_vs_float64(logits, actions, sel, ref, key, tol):
    n_act = ref.shape[1]
    idx = torch.from_numpy(sel).to(logits.device)
    got = logits.reshape(-1, n_act)[idx].cpu().numpy().astype(np.float64)
    act = actions.reshape(-1)[idx].cpu().numpy()
    scale = np.maximum(1.0, np.abs(ref).max(axis=1))
    err = np.abs(got - ref).max(axis=1)
    parity_report(key, {"frames": int(len(sel)), "max_abs_err": float(err.max()),
                        "max_err_over_scale": float((err / scale).max()), "max_abs_logit": float(np.abs(ref).max())})
    bad = np.flatnonzero(err > tol * scale)
    assert bad.size == 0, (f"{bad.size} of {len(sel)} frames beyond {tol} x max(1, max|logit|): "
                           f"flat frames {sel[bad[:8]].tolist()}, errors {err[bad[:8]].tolist()}")
    if n_act > 1:
        srt = np.sort(ref, axis=1)
        safe = srt[:, -1] - srt[:, -2] > 2 * tol * scale
        assert np.array_equal(act[safe], np.argmax(ref, axis=1)[safe])
    else:
        assert np.all(act == 0)


def _chunked(members, frames, c_in, n_act, n_sm):
    """The forward as launches of at most n_sm frames, n_sm members and NB frames per member each."""
    from coevonet_b200 import ops
    P, B = frames.shape[:2]
    logits = torch.empty((P, B, n_act), dtype=torch.float32, device=frames.device)
    actions = torch.empty((P, B), dtype=torch.int32, device=frames.device)
    bs = min(B, NB)
    for b0 in range(0, B, bs):
        bw = min(bs, B - b0)
        step = min(n_sm, n_sm // bw)
        for m0 in range(0, P, step):
            m1 = min(P, m0 + step)
            lg, ac = ops.deepqn_forward(members[m0:m1], frames[m0:m1, b0:b0 + bw].contiguous(), c_in, n_act)
            logits[m0:m1, b0:b0 + bw] = lg
            actions[m0:m1, b0:b0 + bw] = ac
    return logits, actions


@pytest.fixture(scope="module", params=list(SHAPES))
def case(request):
    c_in, n_act, p_of, B, kind, extra = SHAPES[request.param]
    n_sm = _n_sm()
    P = p_of(n_sm)
    seed = 4100 + list(SHAPES).index(request.param)
    torch.cuda.reset_peak_memory_stats()
    members = _members(c_in, n_act, P, seed, extra)
    frames = _frames(kind, P, B, c_in, n_act, seed)
    sel = _subset(P, B, n_sm)
    d = dict(name=request.param, c_in=c_in, n_act=n_act, P=P, B=B, n_sm=n_sm, members=members, frames=frames,
             sel=sel, ref=_reference(members, frames, sel, c_in, n_act))
    yield d
    parity_report(f"k2_scale_{request.param}_peak_torch_bytes", int(torch.cuda.max_memory_allocated()))
    d.clear()


def test_deepqn_at_scale(case, fc_mode):
    from coevonet_b200 import ops
    c_in, n_act, members, frames = case["c_in"], case["n_act"], case["members"], case["frames"]
    logits, actions = ops.deepqn_forward(members, frames, c_in, n_act)
    # a. later jobs and the ragged wave against float64
    _check_vs_float64(logits, actions, case["sel"], case["ref"], f"k2_scale_{case['name']}_{fc_mode}",
                      SCALE_TOL[fc_mode])
    # b. every frame against launches in which every CTA runs one job
    cl, ca = _chunked(members, frames, c_in, n_act, case["n_sm"])
    diff = torch.nonzero((cl != logits).any(dim=-1).reshape(-1)).reshape(-1)
    assert diff.numel() == 0, f"{diff.numel()} of {cl.shape[0] * cl.shape[1]} frames differ from the chunked " \
                              f"launches, first flat frames {diff[:8].tolist()}"
    assert torch.equal(ca, actions)
    # c. determinism
    l2, a2 = ops.deepqn_forward(members, frames, c_in, n_act)
    assert torch.equal(l2, logits) and torch.equal(a2, actions)
    # d. first-max argmax of the kernel's own logits, on every frame
    lg = logits.cpu().numpy()
    assert np.isfinite(lg).all()
    assert np.array_equal(actions.cpu().numpy(), np.argmax(lg, axis=-1))


def test_deepqn_exact_tie_takes_first_max(fc_mode):
    """Output rows 2 and 5 identical with an equal, dominant bias: both logits come out of the same instruction
    sequence, so they tie exactly, and the action is the first of them on every frame."""
    from coevonet_b200 import layout, ops
    c_in, n_act, P, B = 4, 6, _n_sm() + 1, 2
    members = _members(c_in, n_act, P, 4200)
    off = {name: o for name, o, _, _ in layout.dqn_segments(c_in, n_act)[0]}
    ow, ob = off["output.weight"], off["output.bias"]
    members[:, ow + 5 * 512:ow + 6 * 512] = members[:, ow + 2 * 512:ow + 3 * 512]
    members[:, ob + 2] = 100.0
    members[:, ob + 5] = 100.0
    frames = ops.random_frames(4201, (P, B, c_in, 84, 84), "cuda")
    logits, actions = ops.deepqn_forward(members, frames, c_in, n_act)
    assert torch.equal(logits[..., 2], logits[..., 5])
    assert (logits[..., 2] > logits[..., [0, 1, 3, 4]].amax(dim=-1)).all()
    assert (actions == 2).all()


@pytest.mark.parametrize("c_in,n_act", [(4, 6), (6, 18)])
def test_deepqn_constant_frames_vs_float64(fc_mode, c_in, n_act):
    """All-zero and all-255 frames: every BatchNorm sees zero variance, and the float64 logits depend only on
    the betas and the fc layers.  Rounding noise the kernel leaves in a constant channel is amplified by up to
    1/sqrt(eps) ~ 316 there.  Default-init rows (logits < 1), so the suite's own bound applies."""
    from coevonet_b200 import ops
    P = 3
    rows = weights.make_dqn_rows(P, c_in, n_act, 4300 + c_in, bn_jitter=BN_JITTER)
    members = _pad(rows, c_in, n_act)
    frames = torch.zeros((P, 2, c_in, 84, 84), dtype=torch.uint8, device="cuda")
    frames[:, 1] = 255
    logits, actions = ops.deepqn_forward(members, frames, c_in, n_act)
    sel = np.arange(P * 2)
    _check_vs_float64(logits, actions, sel, _reference(members, frames, sel, c_in, n_act),
                      f"k2_constant_frames_c{c_in}_{fc_mode}", FC_MODES[fc_mode])


def test_deepqn_refusals_and_empty_population():
    from coevonet_b200 import _lib, layout, ops
    c_in, n_act, P, B = 4, 6, 2, 1
    dp = layout.dqn_pitch(c_in, n_act)
    members = torch.zeros((P, dp), device="cuda")
    frames = torch.zeros((P, B, c_in, 84, 84), dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.CevError, match="c_in must be"):
        ops.deepqn_forward(torch.zeros((P, layout.dqn_pitch(6, n_act)), device="cuda"),
                           torch.zeros((P, B, 5, 84, 84), dtype=torch.uint8, device="cuda"), 5, n_act)
    wide = torch.zeros((P, layout.dqn_pitch(c_in, 33)), device="cuda")
    for bad in (0, 33):
        with pytest.raises(_lib.CevError):
            ops.deepqn_forward(wide, frames, c_in, bad)
    with pytest.raises(_lib.CevError):
        ops.deepqn_forward(members, frames[:, :0], c_in, n_act)
    with pytest.raises(_lib.CevError, match="multiple of 4"):
        ops.deepqn_forward(torch.zeros((P, dp + 1), device="cuda"), frames, c_in, n_act)
    flat = torch.zeros(P * dp + 4, device="cuda")
    with pytest.raises(_lib.CevError, match="aligned"):
        ops.deepqn_forward(flat[1:1 + P * dp].view(P, dp), frames, c_in, n_act)
    with pytest.raises(_lib.CevError):
        ops.deepqn_forward(members[:1], frames, c_in, n_act)                # fewer rows than frame groups
    logits, actions = ops.deepqn_forward(members[:0], frames[:0], c_in, n_act)
    assert logits.shape == (0, B, n_act) and actions.shape == (0, B)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_deepqn_two_devices_in_one_process():
    """The fc stage's shared-memory attribute is per device: K2 on cuda:0 and then on cuda:1 in one process."""
    from coevonet_b200 import ops
    n_sm = _n_sm()
    c_in, n_act, P, B = 4, 6, n_sm + 1, 2
    members = _members(c_in, n_act, P, 4400, device="cuda:0")
    frames = ops.random_frames(4401, (P, B, c_in, 84, 84), "cuda:0")
    sel = _subset(P, B, n_sm)
    ref = _reference(members, frames, sel, c_in, n_act)
    out = []
    for dev in ("cuda:0", "cuda:1"):
        lg, ac = ops.deepqn_forward(members.to(dev), frames.to(dev), c_in, n_act)
        _check_vs_float64(lg, ac, sel, ref, f"k2_two_devices_{dev}", SCALE_TOL["tc"])
        out.append((lg.cpu(), ac.cpu()))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])
