"""The lattice-network reference (tests/lattice_net.py) pinned on the CPU: it agrees with the oracle and the torch restatement
where rounding is the identity, its preconditions hold on the very data the GPU tests use, and its comparison function flags
a one-step change in any stage of the network."""
import numpy as np
import pytest
import torch

import lattice_net as ln
from helpers import orc, random_playouts, torch_reference_forward

DISTINCT = 256
POWER_BOARDS = 64


def planes_data():
    return ln.random_planes(DISTINCT, seed=1)


def position_data():
    pos, _ = random_playouts(DISTINCT, seed=5, max_plies=120)
    return pos


def test_small_network_matches_the_oracle_and_torch():
    net = ln.small()
    planes = planes_data()[:32]
    rep = ln.reference(net, planes, rounded=False)
    rounded = ln.reference(net, planes, rounded=True)
    assert torch.equal(rep.logits, rounded.logits) and torch.equal(rep.z, rounded.z)   # bf16 rounding is the identity
    p, v = ln.outputs_of(rep.logits, rep.z)
    for name, (rp, rv) in (("oracle", orc.Net(net.arrays).forward_planes(planes)), ("torch", torch_reference_forward(net.arrays, planes))):
        assert np.allclose(p.numpy(), rp, rtol=1e-6, atol=0), name
        assert np.allclose(v.numpy(), rv, rtol=1e-6, atol=1e-7), name


def test_preconditions_hold_for_every_network():
    planes = planes_data()
    for net in ln.networks():
        for rounded in (True, False):
            ln.reference(net, planes, rounded=rounded)   # asserts R1-R4
    pp = orc.to_tensor_batch(position_data())
    for net in ln.position_networks():
        for rounded in (True, False):
            ln.reference(net, pp, rounded=rounded)
    # the dense-live networks between them make every tower layer dense, read every tower channel from a value row and every
    # value_linear_1 input
    dense = [net for net in ln.networks() if net.kind == "dense"]
    assert sorted(net.dense for net in dense) == list(range(20))
    h = ln.HEAD
    assert set().union(*(np.nonzero(net.arrays[h + 8].reshape(8, 128))[1] for net in dense)) == set(range(128))
    assert set().union(*(np.nonzero(net.arrays[h + 14].reshape(512, 64))[0] for net in dense)) == set(range(512))


def test_comparison_accepts_exact_outputs_and_flags_small_errors():
    net = ln.dense_live(3)
    rep = ln.reference(net, planes_data()[:16])
    p, v = ln.outputs_of(rep.logits, rep.z)
    assert ln.compare(p, v, rep.logits, rep.z) == []
    rows = ln.batch_rows(40, 16, seed=2)
    assert ln.compare(p[rows], v[rows], rep.logits, rep.z, rows) == []
    # one logit a lattice step off, one value a lattice step off
    lg = rep.logits.clone()
    lg[5, 777] += ln.LOGIT_Q
    assert ln.compare(p, v, lg, rep.z)
    z = rep.z.clone()
    z[9] += ln.WL1_Q * ln.WL2_Q
    assert ln.compare(p, v, rep.logits, z)


# ---------------------------------------------------------------------------------------------------------- mutation power
def _stages():
    """(stage, network, [(array index, lattice step)]) for the power test: each tower layer in the network where it is dense."""
    h = ln.HEAD
    out = [("input", ln.dense_live(0), [(0, 1.0), (1, 1.0)])]
    for layer in range(20):
        o = ln.tower_index(layer)
        out.append((f"tower{layer}", ln.dense_live(layer), [(o, 1.0), (o + 1, 1.0)]))
    heads_net = ln.sparse_live()
    out += [("W40/b40", heads_net, [(h, 1.0), (h + 1, 1.0), (h + 8, 1.0), (h + 9, 1.0)]),
            ("wp2/bp2", heads_net, [(h + 6, ln.LOGIT_Q), (h + 7, ln.LOGIT_Q)]),
            ("wl1/bl1", heads_net, [(h + 14, ln.WL1_Q), (h + 15, ln.WL1_Q)]),
            ("wl2/bl2", heads_net, [(h + 16, ln.WL2_Q), (h + 17, ln.WL1_Q * ln.WL2_Q)])]
    return out


@pytest.mark.parametrize("stage", [s[0] for s in _stages()])
def test_one_lattice_step_is_flagged(stage):
    """100 random one-step mutations of the stage's weights and biases: the comparison function, applied to the reference of
    the mutated network against the reference of the original, flags at least 90 of them."""
    name, net, arrays = next(s for s in _stages() if s[0] == stage)
    planes = planes_data()[:POWER_BOARDS]
    base = ln.reference(net, planes)
    t = base.tower if not stage.startswith(("input", "tower")) else None
    rng = np.random.default_rng(sum(map(ord, stage)))
    flagged = 0
    for _ in range(100):
        i, q = arrays[int(rng.integers(len(arrays)))]
        m = net.copy()
        j = int(rng.integers(m.arrays[i].size))
        m.arrays[i][j] += np.float32(q * rng.choice([-1.0, 1.0]))
        mut = ln.Report()
        if t is None:
            mut.logits, mut.z = ln.heads(m, ln.tower(m, planes, rep=mut), rep=mut)
        else:
            mut.logits, mut.z = ln.heads(m, t, rep=mut)
        p, v = ln.outputs_of(mut.logits, mut.z)
        flagged += bool(ln.compare(p, v, base.logits, base.z))
    print(f"\n{stage}: {flagged} of 100 flagged")
    assert flagged >= 90, f"{stage}: only {flagged} of 100 one-step mutations flagged"
