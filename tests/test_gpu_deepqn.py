"""K2 parity: grouped per-member DeepQN forward (through the C ABI) vs the
reference's own DeepQN.forward outputs (tests/golden/deepqn.npz) and the oracle.

Three paths are tested, all to the SAME fp32-level tolerance (2e-5 absolute on logits of magnitude ~0.2:
summation order only):
* ``tc`` (default): convolutions and the fully-connected stage on tcgen05 kind::tf32 with every product issued
  three times (3xTF32: lo.hi + hi.lo + hi.hi, fp32 accumulation; K = 3136 in fc1), W1 as the M-side operand;
* ``conv_fp32`` (COEVONET_DQN_CONV=fp32): the CUDA-core fp32 convolutions, then the tensor-core fc stage;
* ``fp32`` (COEVONET_DQN_FC=fp32): the CUDA-core fp32 kernel for the whole forward.
Actions are compared where the reference's top-2 logit gap exceeds twice the tolerance."""
import os

import numpy as np
import pytest
import torch

from oracle import deepqn as odqn
from oracle import weights

pytestmark = pytest.mark.gpu


def _pad(rows, c_in, n_act):
    from coevonet_b200 import layout
    out = np.zeros((rows.shape[0], layout.dqn_pitch(c_in, n_act)), dtype=np.float32)
    out[:, :rows.shape[1]] = rows
    return torch.from_numpy(out).cuda()


FC_MODES = {"conv_fp32": 2e-5, "fp32": 2e-5, "tc": 2e-5}
# the library reads these on every call, so setting them in-process selects the path of the next call
_MODE_ENV = {"conv_fp32": {"COEVONET_DQN_CONV": "fp32"}, "fp32": {"COEVONET_DQN_FC": "fp32"}, "tc": {}}


@pytest.fixture(params=sorted(FC_MODES))
def fc_mode(request):
    old = {k: os.environ.get(k) for k in ("COEVONET_DQN_CONV", "COEVONET_DQN_FC")}
    for k in old:
        os.environ.pop(k, None)
    os.environ.update(_MODE_ENV[request.param])
    yield request.param
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


@pytest.mark.parametrize("c_in,n_act", [(4, 6), (4, 18), (6, 18)])
def test_deepqn_forward_matches_reference_golden(golden, fc_mode, c_in, n_act):
    from coevonet_b200 import ops
    tol = FC_MODES[fc_mode]
    g = golden("deepqn")
    rows = weights.make_dqn_rows(2, c_in, n_act, 600 + c_in + n_act, bn_jitter=float(g["bn_jitter"]))
    rng = np.random.Generator(np.random.PCG64(int(g["frame_seed"])))
    frames = rng.integers(0, 256, (2, 2, c_in, 84, 84), dtype=np.uint8)
    logits, actions = ops.deepqn_forward(_pad(rows, c_in, n_act), torch.from_numpy(frames).cuda(), c_in, n_act)
    want = g[f"c{c_in}a{n_act}.logits"]
    np.testing.assert_allclose(logits.cpu().numpy(), want, rtol=0, atol=tol)
    srt = np.sort(want, axis=-1)
    safe = (srt[..., -1] - srt[..., -2]) > 2 * tol
    assert np.array_equal(actions.cpu().numpy()[safe], np.argmax(want, axis=-1)[safe])


@pytest.mark.parametrize("n_act", [6, 1, 32])     # 32 = the fc epilogue's F3_MAX_ACT (n_out = 512)
def test_deepqn_many_frames_and_members_vs_oracle(fc_mode, n_act):
    from coevonet_b200 import ops
    tol = FC_MODES[fc_mode]
    c_in, P, B = 4, 3, 19                                # B > 16 frames per fc block exercises the frame-block loop
    rows = weights.make_dqn_rows(P, c_in, n_act, 91, bn_jitter=0.1)
    frames = ops.random_frames(5, (P, B, c_in, 84, 84), "cuda")
    logits, actions = ops.deepqn_forward(_pad(rows, c_in, n_act), frames, c_in, n_act)
    want, want_act = odqn.dqn_forward_batch(rows, frames.cpu().numpy(), c_in, n_act)
    np.testing.assert_allclose(logits.cpu().numpy(), want, rtol=0, atol=1.5 * tol)
    srt = np.sort(want, axis=-1)
    safe = (srt[..., -1] - srt[..., -2]) > 4 * tol if n_act > 1 else np.ones((P, B), dtype=bool)
    assert np.array_equal(actions.cpu().numpy()[safe], want_act[safe])
    # per-frame BatchNorm: a frame's logits do not depend on its batch neighbours
    solo, _ = ops.deepqn_forward(_pad(rows, c_in, n_act)[1:2].contiguous(), frames[1:2, 4:5].contiguous(), c_in, n_act)
    assert torch.equal(solo[0, 0], logits[1, 4])


def test_deepqn_module_dropin():
    from coevonet_b200.Atari.deepqn import DeepQN
    torch.manual_seed(3)
    net = DeepQN(4, 6, "float32")
    x = torch.randint(0, 256, (2, 4, 84, 84)).float()
    got = net.forward(x)
    sd = {k: v.numpy() for k, v in net.state_dict().items()}
    from oracle import layout as olayout
    row = olayout.pack_dqn_state_dict(sd, 4, 6)
    want, _ = odqn.dqn_forward_batch(row[None], x.numpy().astype(np.uint8)[None], 4, 6)
    np.testing.assert_allclose(got.numpy(), want[0], rtol=0, atol=3e-5)
    srt = np.sort(want[0, 0])
    if srt[-1] - srt[-2] > 6e-5:
        assert net.determine_action(x[:1]) == int(np.argmax(want[0, 0]))


def test_deepqn_es_perturb_and_update():
    """BASELINE config 5 pieces: K5 on DeepQN rows (conv / Linear prefix perturbed with the Philox stream,
    BatchNorm entries copied) and the layout-agnostic K6 from the materialised members."""
    from coevonet_b200 import layout, ops
    from oracle import philox
    c_in, n_act, P, sigma, lr, seed, gen = 4, 18, 6, 0.05, 0.1, 99, 2
    total, pitch = layout.dqn_dim(c_in, n_act), layout.dqn_pitch(c_in, n_act)
    d_pert = total - 320
    theta = torch.zeros(pitch, device="cuda")
    theta[:total] = torch.from_numpy(weights.make_dqn_rows(1, c_in, n_act, 3, bn_jitter=0.1)[0]).cuda()
    members = ops.es_perturb_dqn(theta, c_in, n_act, sigma, seed, "agent_0", gen, 10, P)
    z = philox.normals(seed, philox.KIND_ES, philox.ROLE_ID["agent_0"], gen, np.arange(10, 10 + P), d_pert)
    th = theta.cpu().numpy()
    want = np.tile(th, (P, 1))
    want[:, :d_pert] = th[:d_pert] + (np.float32(sigma) * z).astype(np.float32)
    got = members.cpu().numpy()
    np.testing.assert_allclose(got[:, :d_pert], want[:, :d_pert], rtol=0, atol=3e-6 * sigma + 1e-9)
    assert np.array_equal(got[:, d_pert:], want[:, d_pert:])          # BatchNorm entries and padding untouched
    fit = torch.randn(P, dtype=torch.float64, device="cuda")
    delta = ops.es_update_members(fit, members, theta, 0, sigma, lr, P).cpu().numpy()
    noise = got - th
    ref = (np.float32(lr / (P * sigma)) * (noise.T.astype(np.float64) @ fit.cpu().numpy())).astype(np.float32)
    np.testing.assert_allclose(delta, ref, rtol=0, atol=2e-5 * np.abs(ref).max())
    assert np.all(delta[d_pert:] == 0)
