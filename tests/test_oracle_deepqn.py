"""The DeepQN oracle's float64 mode (the reference the K2 scale tests hold the kernels to) against its float32
mode, the reference's own logits and the exact values of constant frames."""
import numpy as np
import pytest

from oracle import deepqn as odqn
from oracle import layout, weights


@pytest.mark.parametrize("c_in,n_act", [(4, 6), (6, 18)])
def test_float64_agrees_with_float32_oracle(c_in, n_act):
    rows = weights.make_dqn_rows(2, c_in, n_act, 31 + c_in, bn_jitter=0.5)
    frames = np.random.Generator(np.random.PCG64(5)).integers(0, 256, (2, 2, c_in, 84, 84), dtype=np.uint8)
    l32, a32 = odqn.dqn_forward_batch(rows, frames, c_in, n_act)
    l64, a64 = odqn.dqn_forward_batch(rows, frames, c_in, n_act, np.float64)
    assert l32.dtype == np.float32 and l64.dtype == np.float64
    # float32 summation noise over fan-ins up to 3136 on logits of magnitude ~0.5 (observed <= 1.2e-6)
    np.testing.assert_allclose(l64, l32, rtol=0, atol=5e-6)
    srt = np.sort(l64, axis=-1)
    safe = srt[..., -1] - srt[..., -2] > 1e-5
    assert np.array_equal(a64[safe], a32[safe])


def test_float64_matches_reference_golden(golden):
    g = golden("deepqn")
    for c_in, n_act in ((4, 6), (4, 18), (6, 18)):
        rows = weights.make_dqn_rows(2, c_in, n_act, 600 + c_in + n_act, bn_jitter=float(g["bn_jitter"]))
        rng = np.random.Generator(np.random.PCG64(int(g["frame_seed"])))
        frames = rng.integers(0, 256, (2, 2, c_in, 84, 84), dtype=np.uint8)
        logits, _ = odqn.dqn_forward_batch(rows, frames, c_in, n_act, np.float64)
        np.testing.assert_allclose(logits, g[f"c{c_in}a{n_act}.logits"], rtol=0, atol=2e-5)


@pytest.mark.parametrize("c_in", [4, 6])
@pytest.mark.parametrize("value", [0, 255])
def test_float64_constant_frame_is_exact(c_in, value):
    """A constant frame makes every conv output constant per channel: each BatchNorm sees zero variance and
    outputs exactly relu(beta), so the logits depend only on the betas and the fc layers."""
    n_act = 6
    rows = weights.make_dqn_rows(2, c_in, n_act, 17, bn_jitter=0.7)
    frame = np.full((c_in, 84, 84), value, dtype=np.uint8)
    for row in rows:
        p = layout.unpack_dqn(row, c_in, n_act)
        st = odqn.dqn_layers(row, frame, c_in, n_act, np.float64)
        for i in range(3):
            y, x = st[2 * i], st[2 * i + 1]
            assert np.all(y == y[:, :1, :1]), f"conv{i + 1} output is not constant per channel"
            want = np.maximum(p[f"vbn{i + 1}.bias"].astype(np.float64), 0)[:, None, None]
            assert np.array_equal(x, np.broadcast_to(want, x.shape)), f"BatchNorm-{i + 1} is not exactly relu(beta)"
        h = np.maximum(p["fc1.weight"].astype(np.float64) @ st[5].reshape(-1) + p["fc1.bias"], 0)
        assert np.array_equal(st[-1], p["output.weight"].astype(np.float64) @ h + p["output.bias"])
