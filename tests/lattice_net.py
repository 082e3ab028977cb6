"""Networks whose arithmetic is exact, and a float64 reference that restates the kernels' rounding points.

Every weight, bias and input sits on a power-of-two lattice and every accumulation is bounded by 2^20 lattice steps, so each
fp32 or tensor-core sum in the network has exactly one correct result, whatever the order of its terms.  BatchNorm folds
exactly (gamma 1, integer beta and mean, var = float32(1 - 1e-5) so that var + 1e-5f == 1.0f) and bf16 round-to-nearest-even
of an integer is an integer, so the tower, head stage 1, the logits and the value pre-activation are determined exactly.  A
dropped, duplicated or misplaced term, a wrong bias channel or a wrong tap at a board edge moves an output by at least one
lattice step, which is far above the error of the only inexact operations (ex2.approx, __fdividef, expf, tanhf).

Rounding points of the bf16 path (precision 0), restated by `reference(..., rounded=True)`:
  input planes -> bf16; folded convolution / stage-1 weights -> bf16; policy_conv_2 and value_linear_1 -> bf16 unfolded;
  value_linear_2 and every bias stay fp32;
  convolution epilogue: accumulator + bias + bf16 residual, ReLU, bf16;
  head stage 1: + b40, ReLU, bf16 for P1 (policy) and V1 (value input);
  logits: accumulator + bp2, softmax;  value: V1 . wl1 + bl1, ReLU, x wl2, summed, + bl2, tanh.
The fp32 path (precision 1) is the same without any bf16 rounding (`rounded=False`).
"""
import numpy as np
import torch

N_ARRAYS = 144
HEAD = 6 + 10 * 12          # first array of the heads
VAR = np.float32(1.0 - 1e-5)
LOGIT_Q = 2.0 ** -12        # lattice step of policy_conv_2 (the logits' step with integer P1)
WL1_Q = 2.0 ** -6           # lattice steps of value_linear_1 and value_linear_2: the value pre-activation's step is 2^-12
WL2_Q = 2.0 ** -6

SIZES = [128 * 19 * 9] + [128] * 5 + ([128 * 128 * 9] + [128] * 5) * 20 + \
        [32 * 128, 32, 32, 32, 32, 32, 64 * 32, 64, 8 * 128, 8, 8, 8, 8, 8, 512 * 64, 64, 64, 1]
assert len(SIZES) == N_ARRAYS


def tower_index(layer):
    """First array (weight) of tower convolution `layer` (0..19: conv1 / conv2 of block layer // 2)."""
    return 6 + (layer // 2) * 12 + (layer % 2) * 6


# ------------------------------------------------------------------------------------------------------------- builders
class LatticeNet:
    """144 float32 arrays in az_weight_name order, plus what the tests need to know about them."""

    def __init__(self, name, arrays, kind, live, dense=None):
        self.name, self.arrays, self.kind = name, arrays, kind
        self.live = live     # tower layers with nonzero weights
        self.dense = dense   # the dense tower layer of a dense-live network

    def copy(self):
        return LatticeNet(self.name, [a.copy() for a in self.arrays], self.kind, list(self.live), self.dense)


def _bn(arrays, i, c, rng, spread):
    """BatchNorm i..i+3 that folds exactly: gamma 1, integer beta and mean, var + 1e-5f == 1.0f."""
    arrays[i] = np.ones(c, np.float32)
    arrays[i + 1] = rng.integers(-spread, spread + 1, c).astype(np.float32)
    arrays[i + 2] = rng.integers(-spread, spread + 1, c).astype(np.float32)
    arrays[i + 3] = np.full(c, VAR, np.float32)


def _sparse(rng, co, k, per_row):
    """[co][k] with `per_row` entries of +-1 per row at random places."""
    w = np.zeros((co, k), np.float32)
    for o in range(co):
        idx = rng.choice(k, per_row, replace=False)
        w[o, idx] = rng.choice([-1.0, 1.0], per_row)
    return w


def _dense(rng, shape, p_zero=1 / 3):
    return rng.choice([-1.0, 0.0, 1.0], shape, p=[(1 - p_zero) / 2, p_zero, (1 - p_zero) / 2]).astype(np.float32)


def _centre_identity():
    w = np.zeros((128, 128, 3, 3), np.float32)
    w[np.arange(128), np.arange(128), 1, 1] = 1.0
    return w


# The value head reads few of its inputs (R3 bounds the value pre-activation to 2^13 lattice steps): value_conv one tower channel
# per row, value_linear_1 64 of its 512 inputs.  Head set `part` takes slice `part` of two fixed covers, so that the dense-live
# networks between them read every tower channel from a value row (16 parts) and every V1 input from value_linear_1 (8 parts).
_cover = np.random.default_rng(7)
VALUE_CHANNELS = _cover.permutation(128)
# V1 inputs c * 64 + sq in pairs of two squares of one channel: [32 pair slots][8 channels][2]
V1_PAIRS = np.stack([c * 64 + _cover.permutation(64).reshape(32, 2) for c in range(8)], 1)


def _heads(arrays, rng, part, policy_fan=4):
    """Heads that read every tower channel from policy_conv_1 (row r reads `policy_fan` channels, each channel once, signs balanced
    so that about half of the outputs live); policy_conv_2 +-2^-12 with two entries per row; value_conv row r reads tower channel
    VALUE_CHANNELS[8 part + r]; value_linear_1 reads the V1 inputs of pair slots 4 part .. 4 part + 3 (steps 2^-6, below)."""
    h = HEAD
    perm = rng.permutation(128)
    w1 = np.zeros((32, 128), np.float32)
    for r in range(32):
        w1[r, perm[r * policy_fan:(r + 1) * policy_fan]] = rng.permutation([(-1.0) ** k for k in range(policy_fan)])   # balanced signs
    arrays[h] = w1.ravel()
    arrays[h + 1] = rng.integers(0, 4, 32).astype(np.float32)
    _bn(arrays, h + 2, 32, rng, 1)
    arrays[h + 6] = (_sparse(rng, 64, 32, 2) * LOGIT_Q).ravel()
    arrays[h + 7] = (rng.integers(-64, 65, 64) * LOGIT_Q).astype(np.float32)
    wv = np.zeros((8, 128), np.float32)
    wv[np.arange(8), VALUE_CHANNELS[(8 * part + np.arange(8)) % 128]] = 1.0
    arrays[h + 8] = wv.ravel()
    arrays[h + 9] = rng.integers(4, 8, 8).astype(np.float32)   # > 0: V1 lives on every square, so does every hidden unit
    _bn(arrays, h + 10, 8, rng, 1)
    # [in][out], y = x W + b: hidden unit o reads one input with +2^-6, so that it lives wherever that input does; units 2k and
    # 2k + 1 read two squares of one value channel and enter the value with opposite signs, which keeps the value pre-activation
    # a sum of differences of like-scaled numbers
    wl1 = np.zeros((512, 64), np.float32)
    pairs = V1_PAIRS[(4 * part + np.arange(4)) % 32].reshape(32, 2)[rng.permutation(32)]
    wl1[pairs.ravel(), np.arange(64)] = 1.0
    arrays[h + 14] = (wl1 * WL1_Q).ravel()
    arrays[h + 15] = (rng.integers(-8, 9, 64) * WL1_Q).astype(np.float32)
    sign = rng.choice([-1.0, 1.0], 32)
    arrays[h + 16] = (np.stack([sign, -sign], 1).ravel() * WL2_Q).astype(np.float32)
    arrays[h + 17] = np.array([rng.integers(-64, 65) * WL1_Q * WL2_Q], np.float32)


def _empty():
    return [np.zeros(s, np.float32) for s in SIZES]


def _zero_tower(arrays):
    for layer in range(20):
        o = tower_index(layer)
        arrays[o] = np.zeros(128 * 128 * 9, np.float32)
        arrays[o + 1] = np.zeros(128, np.float32)
        arrays[o + 2] = np.ones(128, np.float32)
        arrays[o + 3] = np.zeros(128, np.float32)
        arrays[o + 4] = np.zeros(128, np.float32)
        arrays[o + 5] = np.full(128, VAR, np.float32)


def _input_conv(arrays, rng, from_positions, w):
    w = w.reshape(128, 19, 9)
    if from_positions:
        w[:, 17:19] = 0.0     # the halfmove / fullmove planes (hm / 100, fm / 200) are off the lattice
    arrays[0] = w.ravel()
    arrays[1] = rng.integers(0, 4, 128).astype(np.float32) if from_positions else rng.integers(-1, 3, 128).astype(np.float32)
    _bn(arrays, 2, 128, rng, 1)


def dense_live(layer, seed=0, from_positions=False):
    """Dense input convolution, tower convolution `layer` dense, its block partner the centre-tap identity, every other block
    the identity (all-zero weights and biases: block inputs are >= 0)."""
    rng = np.random.default_rng(1000 + 37 * layer + seed)
    a = _empty()
    _input_conv(a, rng, from_positions, _dense(rng, (128, 19 * 9)))
    _zero_tower(a)
    o = tower_index(layer)
    a[o] = _dense(rng, (128, 128 * 9), p_zero=0.8).ravel()
    a[o + 1] = rng.integers(100, 250, 128).astype(np.float32)
    _bn(a, o + 2, 128, rng, 4)
    p = tower_index(layer ^ 1)
    a[p] = _centre_identity().ravel()
    a[p + 1] = rng.integers(0, 3, 128).astype(np.float32)
    _bn(a, p + 2, 128, rng, 0)
    _heads(a, rng, part=layer + (20 if from_positions else 0))
    return LatticeNet(f"dense{layer}" + ("_pos" if from_positions else ""), a,
                      "positions" if from_positions else "dense", sorted({layer, layer ^ 1}), layer)


def sparse_live(seed=0, from_positions=False, per_row=3):
    """All 21 convolutions live with `per_row` nonzero +-1 entries per output channel."""
    rng = np.random.default_rng(2000 + seed)
    a = _empty()
    _input_conv(a, rng, from_positions, _sparse(rng, 128, 19 * 9, per_row))
    if from_positions:   # keep the live entries of the input convolution on the planes that carry the position
        w = _sparse(rng, 128, 17 * 9, per_row).reshape(128, 17, 9)
        a[0] = np.concatenate([w, np.zeros((128, 2, 9), np.float32)], 1).ravel()
        a[1] = rng.integers(0, 4, 128).astype(np.float32)
    for layer in range(20):
        o = tower_index(layer)
        a[o] = _sparse(rng, 128, 128 * 9, per_row).ravel()
        a[o + 1] = rng.integers(-2, 1, 128).astype(np.float32)
        _bn(a, o + 2, 128, rng, 0)
    _heads(a, rng, part=21 + from_positions)
    return LatticeNet("sparse" + ("_pos" if from_positions else ""), a, "positions" if from_positions else "sparse", list(range(20)))


def small(seed=0):
    """A network whose activations all stay <= 256, so bf16 rounding is the identity on every one of them."""
    rng = np.random.default_rng(3000 + seed)
    a = _empty()
    _input_conv(a, rng, False, _sparse(rng, 128, 19 * 9, 1))
    for layer in range(20):
        o = tower_index(layer)
        a[o] = _sparse(rng, 128, 128 * 9, 2).ravel()
        a[o + 1] = rng.integers(-1, 1, 128).astype(np.float32)
        _bn(a, o + 2, 128, rng, 0)
    _heads(a, rng, part=23, policy_fan=1)
    return LatticeNet("small", a, "small", list(range(20)))


def networks():
    """Every network the planes-fed GPU tests run: 20 dense-live (one per tower layer), one sparse all-live, the small one."""
    return [dense_live(l) for l in range(20)] + [sparse_live(), small()]


def position_networks():
    """Two different networks fed from positions (zero weights on the halfmove / fullmove planes)."""
    return [dense_live(7, seed=5, from_positions=True), sparse_live(seed=5, from_positions=True)]


# ------------------------------------------------------------------------------------------------------------- inputs
def random_planes(n, seed):
    """[n, 19, 8, 8] float32 planes of random integers in {0, 1, 2} on every square."""
    return np.random.default_rng(seed).integers(0, 3, (n, 19, 8, 8)).astype(np.float32)


def batch_rows(n, distinct, seed):
    """Row i of a batch of n is distinct board rows[i]: all of them in shuffled order, repeated when n > distinct."""
    rng = np.random.default_rng(seed)
    reps = -(-n // distinct)
    return np.concatenate([rng.permutation(distinct) for _ in range(reps)])[:n]


# ------------------------------------------------------------------------------------------------------------- reference
def _bf(t):
    """bf16 round-to-nearest-even of float64 values that are exact in float32."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def _step(t):
    """The largest power of two 2^e (e <= 0) of which every value of t is an integer multiple; 1 for an all-zero t."""
    for e in range(0, -41, -1):
        s = 2.0 ** e
        if bool(torch.all(torch.remainder(t, s) == 0)):
            return s
    raise AssertionError("value off every lattice down to 2^-40")


def _on(t, q):
    return bool(torch.all(torch.remainder(t, q) == 0))


class Report:
    """Reference outputs (float64) and what the precondition checks measured."""

    def __init__(self):
        self.positive, self.changed, self.ties = {}, {}, {}
        self.logits = self.z = self.tower = None


def _fold(a, i, co, k):
    """BatchNorm i+2.. folded into conv weight a[i] ([co][k]) / bias a[i+1] the way nn.cu:fold does, asserting that the scale is
    exactly one (so the folded arrays equal weight and bias - mean + beta)."""
    g, b, m, v = (np.asarray(a[i + j], np.float32) for j in range(2, 6))
    s = g / np.sqrt(v + np.float32(1e-5))
    assert np.all(s == np.float32(1.0)), "BatchNorm does not fold with scale 1"
    w = np.asarray(a[i], np.float32).reshape(co, k).astype(np.float64)
    bias = (np.asarray(a[i + 1], np.float32) - m) * s + b
    return torch.from_numpy(w), torch.from_numpy(bias.astype(np.float64))


def _bound(what, terms_abs, q):
    mx = float(terms_abs.max()) if terms_abs.numel() else 0.0
    assert mx <= 2.0 ** 20 * q, f"R1: {what}: sum of |terms| {mx} exceeds 2^20 x step {q}"


def _conv(x, w, bias, residual, rounded, what, rep):
    """3x3 same convolution + bias (+ residual), ReLU, (bf16): x [n, ci, 8, 8], w [co][ci*9]."""
    co = w.shape[0]
    w4 = w.reshape(co, -1, 3, 3)
    if rounded:
        w4 = _bf(w4)
    q = _step(w4) * _step(x)
    assert _on(bias, q) and (residual is None or _on(residual, q)), f"R1: {what}: bias / residual off the lattice step {q}"
    terms = torch.nn.functional.conv2d(x.abs(), w4.abs(), padding=1) + bias.abs().view(1, -1, 1, 1)
    acc = torch.nn.functional.conv2d(x, w4, padding=1) + bias.view(1, -1, 1, 1)
    if residual is not None:
        terms = terms + residual.abs()
        acc = acc + residual
    _bound(what, terms, q)
    out = torch.relu(acc)
    rep.positive[what] = float((out > 0).double().mean())
    if rounded:
        r = _bf(out)
        rep.changed[what] = float((r != out).double().mean())
        pos = out[out >= 256]
        ulp = torch.exp2(torch.floor(torch.log2(pos)) - 7)
        rep.ties[what] = int((torch.remainder(pos, ulp) == ulp / 2).sum())
        out = r
    return out


def _is_zero(w, b):
    return not np.any(w) and not np.any(b)


def _is_centre_identity(w, b):
    w = w.reshape(128, 128, 9)
    return np.array_equal(w[:, :, 4], np.eye(128, dtype=np.float32)) and not np.any(np.delete(w, 4, 2)) and np.all(b >= 0)


def tower(net, planes, rounded=True, device="cpu", rep=None):
    """Tower output [n, 128, 64] (float64) of `planes` [n, 19, 8, 8]."""
    rep = rep or Report()
    a = net.arrays
    x = torch.as_tensor(np.asarray(planes, np.float32), device=device).to(torch.float64).reshape(-1, 19, 8, 8)
    w, b = _fold(a, 0, 128, 19 * 9)
    dead = [c for c in range(19) if not np.any(w.numpy().reshape(128, 19, 9)[:, c])]
    if dead:   # planes with zero weights add exact zeros (the halfmove / fullmove planes of positions are off the lattice)
        x = x.clone()
        x[:, dead] = 0.0
    if rounded:
        x = _bf(x)
    x = _conv(x, w.to(device), b.to(device), None, rounded, "input", rep)
    for blk in range(10):
        o1, o2 = tower_index(2 * blk), tower_index(2 * blk + 1)
        w1, b1 = _fold(a, o1, 128, 128 * 9)
        w2, b2 = _fold(a, o2, 128, 128 * 9)
        if _is_zero(w1.numpy(), b1.numpy()) and _is_zero(w2.numpy(), b2.numpy()):
            continue    # relu(0 + 0 + x) = x for x >= 0
        if _is_centre_identity(w1.numpy(), b1.numpy()):
            y = x + b1.to(device).view(1, -1, 1, 1)   # relu(x + b) with x, b >= 0; exact in bf16 below 2^8 x ulp
            y = _bf(y) if rounded else y
        else:
            y = _conv(x, w1.to(device), b1.to(device), None, rounded, f"tower{2 * blk}", rep)
        x = _conv(y, w2.to(device), b2.to(device), x, rounded, f"tower{2 * blk + 1}", rep)
    return x.reshape(-1, 128, 64)


def heads(net, t, rounded=True, rep=None):
    """(logits [n, 4096], value pre-activation [n]) in float64 from the tower output t [n, 128, 64]."""
    rep = rep or Report()
    a, h, dev = net.arrays, HEAD, t.device
    wp, bp = _fold(a, h, 32, 128)
    wv, bv = _fold(a, h + 8, 8, 128)
    w40, b40 = torch.cat([wp, wv]).to(dev), torch.cat([bp, bv]).to(dev)
    if rounded:
        w40 = _bf(w40)
    q = _step(w40) * _step(t)
    assert _on(b40, q), "R1: stage 1: bias off the lattice"
    _bound("stage 1", torch.einsum("oc,ncs->nos", w40.abs(), t.abs()) + b40.abs().view(1, -1, 1), q)
    d1 = torch.relu(torch.einsum("oc,ncs->nos", w40, t) + b40.view(1, -1, 1))
    rep.positive["stage 1 policy"] = float((d1[:, :32] > 0).double().mean())
    rep.positive["stage 1 value"] = float((d1[:, 32:] > 0).double().mean())
    if rounded:
        r = _bf(d1)
        rep.changed["stage 1"] = float((r != d1).double().mean())
        d1 = r
    p1, v1 = d1[:, :32], d1[:, 32:].reshape(-1, 512)
    # logits[co * 64 + sq] = wp2[co] . P1[:, sq] + bp2[co]
    wp2 = torch.from_numpy(np.asarray(a[h + 6], np.float64).reshape(64, 32)).to(dev)
    bp2 = torch.from_numpy(np.asarray(a[h + 7], np.float64)).to(dev)
    if rounded:
        wp2 = _bf(wp2)
    q = _step(wp2) * _step(p1)
    assert _on(bp2, q), "R1: logits: bias off the lattice"
    assert q >= 2.0 ** -12, f"R2: logit step {q} < 2^-12"
    _bound("logits", torch.einsum("ok,nks->nos", wp2.abs(), p1.abs()) + bp2.abs().view(1, -1, 1), q)
    logits = (torch.einsum("ok,nks->nos", wp2, p1) + bp2.view(1, -1, 1)).reshape(-1, 4096)
    spread = float((logits.max(1).values - logits.min(1).values).max()) if logits.shape[0] else 0.0
    assert spread <= 48, f"R2: logit spread {spread} > 48 within a board"
    # value: V1 [512] . wl1 [512][64] + bl1, ReLU, . wl2 + bl2
    wl1 = torch.from_numpy(np.asarray(a[h + 14], np.float64).reshape(512, 64)).to(dev)
    bl1 = torch.from_numpy(np.asarray(a[h + 15], np.float64)).to(dev)
    wl2 = torch.from_numpy(np.asarray(a[h + 16], np.float64)).to(dev)
    bl2 = torch.from_numpy(np.asarray(a[h + 17], np.float64)).to(dev)
    if rounded:
        wl1 = _bf(wl1)
    q1 = _step(wl1) * _step(v1)
    assert _on(bl1, q1), "R1: value_linear_1: bias off the lattice"
    _bound("value_linear_1", v1.abs() @ wl1.abs() + bl1.abs(), q1)
    h1 = torch.relu(v1 @ wl1 + bl1)
    rep.positive["value hidden"] = float((h1 > 0).double().mean())
    q2 = q1 * _step(wl2)
    assert _on(bl2, q2), "R1: value_linear_2: bias off the lattice"
    assert q2 >= 2.0 ** -12, f"R3: value step {q2} < 2^-12"
    _bound("value_linear_2", h1.abs() @ wl2.abs() + bl2.abs(), q2)
    z = h1 @ wl2 + bl2
    zmax = float(z.abs().max()) if z.numel() else 0.0
    assert zmax <= 2.0, f"R3: |value pre-activation| {zmax} > 2"
    return logits, z


def reference(net, planes, rounded=True, device="cpu", check_live=True):
    """Reference outputs of `planes` [n, 19, 8, 8]: a Report with .logits [n, 4096] and .z [n] (float64 tensors on `device`).
    Asserts R1-R3 (inside) and R4: at least 25 % of the live outputs are positive after ReLU, and in the dense-live networks bf16
    rounding changes at least 10 % of the outputs of the dense tower layer, some of them exact ties."""
    rep = Report()
    rep.tower = tower(net, planes, rounded, device, rep)
    rep.logits, rep.z = heads(net, rep.tower, rounded, rep)
    if check_live:
        for k, v in rep.positive.items():
            assert v >= 0.25, f"R4: {net.name}: only {v:.1%} of the outputs of {k} are positive"
        if rounded and net.kind == "dense":
            k = f"tower{net.dense}"
            assert rep.changed[k] >= 0.10, f"R4: {net.name}: bf16 rounding changes only {rep.changed[k]:.1%} of {k}"
            assert rep.ties[k] > 0, f"R4: {net.name}: no exact ties in {k}"
        if rounded and net.kind == "small":
            assert not any(rep.changed.values()), f"{net.name}: bf16 rounding changes an activation"
    return rep


# ------------------------------------------------------------------------------------------------------------- comparison
POLICY_TOL = 1e-5
VALUE_TOL = 1e-6


def compare(policy, value, logits, z, rows=None):
    """The kernel's (policy [n, 4096], value [n]) against the reference (logits [m, 4096], z [m]) of the distinct boards,
    row i of the batch being distinct board rows[i].  Returns a list of failures (empty when the outputs agree):
      policy: |(ln p_i - ln p_max) - (l_i - l_max)| <= 1e-5 for every move, every p_i > 0, |sum p - 1| <= 1e-5;
      value:  |v - tanh(z)| <= 1e-6."""
    dev = logits.device
    p = torch.as_tensor(np.asarray(policy), device=dev).to(torch.float64)
    v = torch.as_tensor(np.asarray(value), device=dev).to(torch.float64)
    if rows is not None:
        idx = torch.as_tensor(np.asarray(rows), device=dev, dtype=torch.long)
        logits, z = logits[idx], z[idx]
    bad = []
    if not bool(torch.all(p > 0)):
        r = int(torch.nonzero(~(p > 0))[0, 0])
        bad.append(f"row {r}: a probability is not > 0")
        return bad
    s = (p.sum(1) - 1).abs()
    if float(s.max()) > POLICY_TOL:
        bad.append(f"row {int(s.argmax())}: |sum p - 1| = {float(s.max()):.3g}")
    lp = p.log()
    d = ((lp - lp.max(1, keepdim=True).values) - (logits - logits.max(1, keepdim=True).values)).abs()
    if float(d.max()) > POLICY_TOL:
        r, c = divmod(int(d.argmax()), 4096)
        bad.append(f"row {r} move {c} (plane {c // 64}, square {c % 64}): log-probability off by {float(d.max()):.3g} "
                   f"({int((d.amax(1) > POLICY_TOL).sum())} rows wrong)")
    dv = (v - torch.tanh(z)).abs()
    if float(dv.max()) > VALUE_TOL:
        bad.append(f"row {int(dv.argmax())}: value off by {float(dv.max()):.3g} (z = {float(z[int(dv.argmax())]):.6g}, "
                   f"{int((dv > VALUE_TOL).sum())} rows wrong)")
    return bad


def check(policy, value, rep, rows=None, what=""):
    bad = compare(policy, value, rep.logits, rep.z, rows)
    assert not bad, f"{what}: " + "; ".join(bad)


def outputs_of(logits, z):
    """What an exact kernel would return for (logits, z): float32 softmax and tanh."""
    return torch.softmax(logits, 1).to(torch.float32), torch.tanh(z).to(torch.float32)
