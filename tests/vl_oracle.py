"""Restatement of az_search_vl's semantics (leaf-parallel search with virtual loss, NOT in the reference; DESIGN.md section 5)
for the tests, written from the semantics, not from the CUDA code.  It keeps the reference's arithmetic (tree.rs:180-207) in
IEEE f32 and uses the oracle library for the chess rules (play_move with the game history plus the leaf's own path), the
legal-move order, Dirichlet noise and the synthetic evaluator.  With leaves_per_root = 1 it is orc.search (checked in
tests/test_search_vl_cpu.py).

    search_vl(root, evaluate, num_simulations, leaves_per_root, virtual_loss, history=None, noise_game=-1, noise_ply=0)

`evaluate(position) -> (policy [4096] f32, value)`; `stub(seed)` is the shared synthetic evaluator.  Returns dict(visits,
scores, depth, evaluations (the root's included), collisions, terminal_leaves)."""
import numpy as np

from helpers import orc

F = np.float32
ONGOING, DRAW, ILLEGAL = 0, 1, -1


def stub(seed):
    return lambda pos: orc.stub_eval(seed, pos)


class Node:
    """MCTree (tree.rs:25-34) over the node's distinct legal policy indices in move order (the reference iterates the legal
    indices with the under-promotion duplicates; a duplicate never wins its strict '>' comparison)."""

    def __init__(self, pos, history, policy):
        self.pos, self.history = pos, history        # history: every position counted so far, this one last
        _, ix = orc.legal_moves(pos)
        _, first = np.unique(ix, return_index=True)
        self.index = ix[np.sort(first)].astype(np.int64)
        self.P = policy[self.index].astype(F)
        L = len(self.index)
        self.N, self.W = np.zeros(L, F), np.zeros(L, F)
        self.V = np.zeros(L, np.int64)
        self.children = {}

    def depth(self):   # max_subtree_depth (tree.rs:258-269)
        return 1 + max(c.depth() for c in self.children.values()) if self.children else 0


def _noisy(policy, pos, params):
    """apply_dirichlet_noise (tree.rs:272-289) on the dense policy: one component per legal move, duplicates included."""
    seed, game, ply, alpha, eps = params
    _, ix = orc.legal_moves(pos)
    if len(ix) < 2:
        return policy
    noise = orc.dirichlet(seed, game, ply, alpha, len(ix))
    p = (policy.astype(F) * (F(1.0) - F(eps))).astype(F)
    for k, i in enumerate(ix):
        p[i] = F(p[i] + F(F(eps) * noise[k]))
    return p


def _gather(root, c_puct, lam):
    """One descent.  Returns the path [(node, edge)] of a leaf (V += 1 along it) or None for a collision."""
    path, t = [], root
    while True:
        v = t.V.astype(F)
        n = (t.N + v).astype(F)
        w = (t.W - (F(lam) * v).astype(F)).astype(F)
        total = F(F(int(t.N.sum()) + int(t.V.sum())) + F(1.0))     # sum of N' over the node's edges, plus 1: exact integers
        u = (((F(c_puct) * t.P).astype(F) * np.sqrt(total)).astype(F) / (F(1.0) + n)).astype(F)
        with np.errstate(divide="ignore", invalid="ignore"):
            q = np.where(n > 0, (w / n).astype(F), F(0.0)).astype(F)
        val = (q + u).astype(F)
        val = np.where(np.isnan(val), F(-np.inf), val)
        e = int(np.argmax(val)) if len(val) and val.max() > -np.inf else 0   # first maximum = strict '>' in move order
        path.append((t, e))
        if e in t.children:
            t = t.children[e]
            continue
        if t.V[e] > 0:
            return None
        for node, edge in path:
            node.V[edge] += 1
        return path


def search_vl(root, evaluate, num_simulations, leaves_per_root, virtual_loss=1.0, history=None, noise_game=-1, noise_ply=0,
              c_puct=3.0, alpha=0.3, eps=0.25, seed=42):
    if leaves_per_root < 1 or not virtual_loss >= 0.0:
        raise ValueError("leaves_per_root must be >= 1 and virtual_loss >= 0")
    root = np.ascontiguousarray(np.atleast_1d(root), orc.POSITION_DTYPE)[0]
    hist = [h for h in history] if history is not None and len(history) else [root]
    policy, _ = evaluate(root)
    if noise_game >= 0:
        policy = _noisy(policy, root, (seed, noise_game, noise_ply, alpha, eps))
    tree = Node(root, hist, policy)
    stats = dict(evaluations=1, collisions=0, terminal_leaves=0)
    done = 0
    while len(tree.index) and done < num_simulations:
        leaves = []
        for _ in range(min(leaves_per_root, num_simulations - done)):
            path = _gather(tree, c_puct, virtual_loss)
            if path is None:
                stats["collisions"] += 1
                break
            leaves.append(path)
        values = []
        for path in leaves:   # expand (tree.rs:209-237) after the whole gather
            parent, e = path[-1]
            child, r = orc.play_move(parent.pos, int(parent.index[e]), np.array(parent.history, orc.POSITION_DTYPE))
            assert r != ILLEGAL
            if r == ONGOING:
                pol, value = evaluate(child)
                stats["evaluations"] += 1
                parent.children[e] = Node(child, parent.history + [child], pol)
                values.append(F(value))
            else:
                stats["terminal_leaves"] += 1
                values.append(F(0.0) if r == DRAW else F(-1.0))
        for path, value in zip(leaves, values):   # backup in leaf order (tree.rs:197-206)
            for node, e in reversed(path):
                value = F(-value)
                node.V[e] -= 1
                node.W[e] = F(node.W[e] + value)
                node.N[e] = F(node.N[e] + F(1.0))
        done += len(leaves)
    visits = np.zeros(orc.ACTION_SPACE, F)
    scores = np.zeros(orc.ACTION_SPACE, F)
    visits[tree.index] = tree.N
    scores[tree.index] = tree.W
    return dict(visits=visits, scores=scores, depth=tree.depth(), **stats)
