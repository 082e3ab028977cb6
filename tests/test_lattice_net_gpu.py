"""Every network kernel against the exact float64 reference of tests/lattice_net.py: networks whose weights, biases and inputs sit
on a power-of-two lattice, so that each accumulation of the tower, head stage 1, the logits and the value pre-activation has
exactly one correct result.  The comparison allows only the error of ex2.approx / expf / __fdividef / tanhf, about 24 times
smaller than one lattice step of a logit; a dropped, duplicated or misplaced term fails it."""
import numpy as np
import pytest
import torch

import alphazero_chess_b200 as az
import lattice_net as ln
from helpers import orc, random_playouts
from test_networks_gpu import _splits

pytestmark = pytest.mark.gpu

DISTINCT = 256   # distinct boards; larger batches repeat them in shuffled order
SIZES = [1, 2, 3, 4, 5, 127, 296, 297, 2072, 2073, 4095, 4096, 4736, 4737, 4801]
CONFIGS = {
    "mma.sync heads": {"AZ_HEADS_TC": "0"},
    "21 launches": {"AZ_TOWER_FUSED": "0", "AZ_INPUT_K32": "0", "AZ_TOWER_WIDE": "0"},
    "input convolution inside the tower launch": {"AZ_TOWER_FUSED": "2", "AZ_INPUT_K32": "0", "AZ_TOWER_WIDE": "0"},
    "three ranges, one launch each": {"AZ_TOWER_SPLIT": "3", "AZ_TOWER_INKERNEL": "0"},
    "16-file boxes": {"AZ_TOWER_WIDE": "1"},
    "alternating input epilogue": {"AZ_INPUT_EPI2": "1"},
    "release arrive": {"AZ_TC_RELEASE_ARRIVE": "1"},
    "140 tower CTAs": {"AZ_TOWER_GRID": "140"},
}
NETS = ln.networks()
_refs = {}


@pytest.fixture(scope="module")
def planes():
    return ln.random_planes(DISTINCT, seed=1)


@pytest.fixture(scope="module")
def positions():
    pos, _ = random_playouts(DISTINCT, seed=5, max_plies=120)
    return pos


def _ref(net, data, rounded):
    """The reference of the distinct boards (computed once per network, path and data), on the GPU for the comparison."""
    key = (net.name, rounded, data.shape)
    if key not in _refs:
        rep = ln.reference(net, data, rounded=rounded)
        rep.logits, rep.z = rep.logits.cuda(), rep.z.cuda()
        _refs[key] = rep
    return _refs[key]


def _run_planes(e, planes, sizes, rounded=True):
    for net in NETS:
        e.load_weights(net.arrays)
        rep = _ref(net, planes, rounded)
        for n in sizes:
            rows = ln.batch_rows(n, DISTINCT, seed=n)
            pol, val = e.forward_planes(planes[rows])
            ln.check(pol, val, rep, rows, what=f"{net.name}, n = {n}")


def test_forward_planes_default_configuration(planes):
    with az.Engine(max_games=max(SIZES), precision=0) as e:
        _run_planes(e, planes, SIZES)


@pytest.mark.parametrize("config", list(CONFIGS))
def test_forward_planes_other_configurations(planes, monkeypatch, config):
    for k, v in CONFIGS[config].items():
        monkeypatch.setenv(k, v)   # the knobs are read when the engine is created
    with az.Engine(max_games=4096, precision=0) as e:
        _run_planes(e, planes, (3, 297, 4096))


def test_forward_planes_fp32_path(planes):
    with az.Engine(max_games=300, precision=1) as e:
        _run_planes(e, planes, (1, 7, 300), rounded=False)


def test_small_network_bf16_and_fp32_paths_agree(planes):
    """The small network never rounds, so the bf16 and the fp32 path compute the same logits and value pre-activations: their
    log-probabilities (relative to each board's largest) and values agree to twice the comparison's bound."""
    small = next(net for net in NETS if net.kind == "small")
    assert torch.equal(_ref(small, planes, True).logits, _ref(small, planes, False).logits)
    out = []
    for precision in (0, 1):
        with az.Engine(max_games=DISTINCT, precision=precision) as e:
            e.load_weights(small.arrays)
            out.append(e.forward_planes(planes))
    (p0, v0), (p1, v1) = out
    l0, l1 = np.log(p0.astype(np.float64)), np.log(p1.astype(np.float64))
    d = np.abs((l0 - l0.max(1, keepdims=True)) - (l1 - l1.max(1, keepdims=True)))
    assert d.max() <= 2 * ln.POLICY_TOL, d.max()
    assert np.abs(v0.astype(np.float64) - v1).max() <= 2 * ln.VALUE_TOL


@pytest.mark.parametrize("precision", [0, 1])
def test_forward_and_forward_networks_from_positions(positions, precision):
    nets = ln.position_networks()
    pl = orc.to_tensor_batch(positions)
    refs = [_ref(net, pl, precision == 0) for net in nets]
    # each network's range of a batch starts on a multiple of four boards
    with az.Engine(max_games=4096, max_batch=4096 + 8, precision=precision) as e:
        e.load_weights(nets[0].arrays)
        e.load_weights(nets[1].arrays, network=1)
        for n in (1, 3, 2073, 4096):
            rows = ln.batch_rows(n, DISTINCT, seed=n)
            pos = positions[rows]
            pol, val = e.forward(pos)
            ln.check(pol, val, refs[0], rows, what=f"forward, n = {n}")
            for name, net in _splits(n, np.random.default_rng(n)):
                pol, val = e.forward_networks(pos, net)
                for s in (0, 1):
                    sel = np.nonzero(net == s)[0]
                    if len(sel):
                        ln.check(pol[sel], val[sel], refs[s], rows[sel], what=f"forward_networks, n = {n}, {name}, network {s}")
