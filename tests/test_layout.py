"""Flat-row layouts: product vs oracle, vs a torch module built like the reference, and vs the
outputs of the reference's own modules (tests/golden)."""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import layout as olayout


def test_dims_match_survey():
    assert layout.fc_dim(10) == 139781 and layout.fc_dim(8) == 138757
    assert len(layout.fc_perturbable_index(10)) == 138245
    assert len(layout.fc_perturbable_index(8)) == 137221
    assert layout.fc_pitch(10) % 32 == 0 and layout.fc_pitch(8) % 32 == 0
    assert layout.dqn_dim(4, 6) == 1687526 and layout.dqn_dim(6, 18) == 1697778
    for in_dim in (8, 10):
        a, ta = layout.fc_segments(in_dim)
        b, tb = olayout.fc_segments(in_dim)
        assert a == b and ta == tb
        assert np.array_equal(layout.fc_perturbable_index(in_dim), olayout.fc_perturbable_index(in_dim))
    assert layout.dqn_segments(4, 18) == olayout.dqn_segments(4, 18)


def test_sub_tensors_are_16_byte_aligned():
    for in_dim in (8, 10):
        segs, _ = layout.fc_segments(in_dim)
        offs = {n: o for n, o, _, _ in segs}
        assert offs["fc2.weight"] % 32 == 0          # cp.async / bulk-copy source
        assert offs["fc1.weight"] == 0


def test_pack_unpack_roundtrip_with_module():
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    net = FCNetwork(10, 5, "float32")
    row = layout.pack_state_dict(net.state_dict(), 10)
    flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
    assert torch.equal(row[:layout.fc_dim(10)], flat)               # parameters() order
    sd = layout.unpack_to_state_dict(row, 10)
    for k, v in net.state_dict().items():
        assert torch.equal(sd[k], v)
    # ES view == get_perturbable_weights
    pert = net.get_perturbable_weights()
    assert np.array_equal(row.numpy()[layout.fc_perturbable_index(10)], pert)


# The layout against what the reference's own modules produced (tests/golden, written by
# oracle/make_golden.py, which loaded the rows into the reference's modules by parameter name).
def test_fc_names_offsets_and_shapes_reproduce_reference_logits(golden):
    """Read by this layout's names, offsets and shapes, the weights the reference's FCNetwork held
    give its logits (MPE/fcnetwork.py:37-70: Linear -> LayerNorm -> ReLU, twice, then Linear)."""
    import torch.nn.functional as F
    from oracle import weights
    g = golden("fc_logits")
    for role in ("agent_0", "adversary_0"):
        in_dim = layout.OBS_DIM[role]
        rows = weights.make_fc_rows(3, in_dim, int(g[f"{role}.seed"]), ln_jitter=float(g["ln_jitter"]))
        x = torch.from_numpy(g[f"{role}.obs"])
        for m in range(3):
            p = layout.unpack_to_state_dict(torch.from_numpy(rows[m]), in_dim)
            h = F.linear(x, p["fc1.weight"], p["fc1.bias"])
            h = F.relu(F.layer_norm(h, (layout.H1,), p["ln1.weight"], p["ln1.bias"]))
            h = F.linear(h, p["fc2.weight"], p["fc2.bias"])
            h = F.relu(F.layer_norm(h, (layout.H2,), p["ln2.weight"], p["ln2.bias"]))
            logits = F.linear(h, p["output.weight"], p["output.bias"]).numpy()
            np.testing.assert_allclose(logits, g[f"{role}.logits"][m], rtol=0, atol=2e-6)


def test_fc_parameter_order_and_perturbable_view_reproduce_reference_mutation(golden):
    """Agent.mutate (agent.py:25-29) draws one noise tensor per parameters() entry in registration
    order, so the reference's child equals noise laid out segment by segment in fc_segments order.
    mutate_ES (agent.py:31-70) perturbs get_perturbable_weights() only and returns its noise in that
    order; compute_weight_update's result is in the same order, so fc_perturbable_index must
    reproduce both the reference's perturbed rows and its update vector."""
    from oracle import ga_es, philox, weights
    g = golden("mutation")
    segs, D = layout.fc_segments(10)
    parent = weights.make_fc_rows(1, 10, int(g["parent_seed"]), ln_jitter=float(g["ln_jitter"]))[0]
    assert parent.shape == (D,)
    z = philox.normals(int(g["seed"]), philox.KIND_GA, 0, int(g["ga_gen"]), [int(g["ga_member"])], D)[0]
    sig = np.float32(g["ga_sigma"])
    child, used = parent.copy(), 0
    for _, off, shape, _ in segs:
        n = int(np.prod(shape))
        child[off:off + n] += (sig * z[used:used + n]).astype(np.float32)
        used += n
    assert used == D
    assert int(np.bitwise_xor.reduce(child.view(np.uint32))) == int(g["ga_child_crc"][0])
    assert np.array_equal(child[:64], g["ga_child_head"]) and np.array_equal(child[-64:], g["ga_child_tail"])

    pidx = layout.fc_perturbable_index(10)
    assert len(pidx) == len(g["es_update"])
    P, sigma = int(g["es_P"]), np.float32(g["es_sigma"])
    zs = philox.normals(int(g["seed"]), philox.KIND_ES, 0, int(g["es_gen"]), np.arange(P), D)
    noise = (sigma * zs[:, pidx]).astype(np.float32)
    rows = np.repeat(parent[None], P, axis=0)
    rows[:, pidx] = parent[pidx] + noise
    assert int(np.bitwise_xor.reduce(rows.view(np.uint32).reshape(-1))) == int(g["es_rows_crc"][0])
    upd = ga_es.es_update(noise, g["es_rewards"], float(g["lr"]), float(g["es_sigma"]))
    np.testing.assert_allclose(upd, g["es_update"], rtol=0, atol=1e-6 * np.abs(g["es_update"]).max())


def test_dqn_names_offsets_and_shapes_reproduce_reference_logits(golden):
    """Read by dqn_segments' names, offsets and shapes, the weights the reference's DeepQN held give
    its logits (Atari/deepqn.py:39-48: three conv -> train-mode BatchNorm -> ReLU, fc1 -> ReLU, output)."""
    import torch.nn.functional as F
    from oracle import weights
    g = golden("deepqn")
    for c_in, n_act in ((4, 6), (4, 18), (6, 18)):
        segs, _ = layout.dqn_segments(c_in, n_act)
        rows = weights.make_dqn_rows(2, c_in, n_act, 600 + c_in + n_act, bn_jitter=float(g["bn_jitter"]))
        rng = np.random.Generator(np.random.PCG64(int(g["frame_seed"])))
        frames = rng.integers(0, 256, (2, 2, c_in, 84, 84), dtype=np.uint8)
        for m in range(2):
            row = torch.from_numpy(rows[m])
            p = {name: row[off:off + int(np.prod(shape))].reshape(shape) for name, off, shape, _ in segs}
            x = torch.from_numpy(frames[m].astype(np.float32)) / 255.0
            for i, stride in ((1, 4), (2, 2), (3, 1)):
                x = F.conv2d(x, p[f"conv{i}.weight"], p[f"conv{i}.bias"], stride=stride)
                # batch 1 in the reference: each frame is normalised over its own H x W
                x = torch.cat([F.batch_norm(f[None], None, None, p[f"vbn{i}.weight"], p[f"vbn{i}.bias"],
                                            training=True, eps=1e-5) for f in x])
                x = F.relu(x)
            x = F.relu(F.linear(x.reshape(x.shape[0], -1), p["fc1.weight"], p["fc1.bias"]))
            logits = F.linear(x, p["output.weight"], p["output.bias"]).numpy()
            np.testing.assert_allclose(logits, g[f"c{c_in}a{n_act}.logits"][m], rtol=0, atol=5e-6)
