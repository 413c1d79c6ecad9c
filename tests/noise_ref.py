"""Restatement of the Dirichlet root noise (DESIGN.md §4.6) on top of tests/pyref.py, for the parity tests of
tests/test_root_noise.py.

NoisyTree is pyref.Tree whose PUCT score at the root uses P' = (1 - eps) * P + eps * eta (f32, each operation rounded, eta in
child order); every other depth uses the stored prior, and use_subtree drops the noise.  search_vl restates the K-leaf search
with virtual loss (DESIGN.md §4.3) over pyref states; search (K = 1) and the chess search are pyref's / test_chess_search's.
"""
import numpy as np

import pyref
from oracle import pyoracle as O

F = np.float32


class NoisyTree(pyref.Tree):
    def __init__(self, state, c=2.0):
        super().__init__(state, c)
        self.eta, self.eps, self.omeps = None, F(0), F(1)

    def set_root_noise(self, eta, eps):
        """eta: one entry per root child; eps = 0 turns the noise off."""
        self.eps = F(eps)
        self.omeps = F(F(1) - F(eps))
        self.eta = [F(x) for x in eta] if eps != 0 else None

    def ucb(self, pid, cid):
        if pid != 0 or self.eta is None:
            return super().ucb(pid, cid)
        p, ch = self.arena[pid], self.arena[cid]
        prior = F(F(self.omeps * ch["prior"]) + F(self.eps * self.eta[cid - p["children"][0]]))
        q = F(0) if ch["N"] == 0 else F(F(F(-ch["W"]) / F(ch["N"]) + F(1)) / F(2))
        u = F(self.c * prior)
        u = F(u * np.sqrt(F(p["N"])))
        u = F(u / F(F(1) + F(ch["N"])))
        return F(q + u)

    def use_subtree(self, rid):
        super().use_subtree(rid)
        self.eta = None


def _terminal_value(st):
    return F(-1) if st.status == 2 else F(0)


def search_vl(trees, num_searches, K, evaluator):
    """K leaves per tree per step: a terminal leaf is backed up at once; otherwise every path node takes a virtual loss
    (N += 1, W += 1) and the leaf is queued, as a duplicate if it is already queued in this step.  After the evaluator the
    entries finish in selection order: a first occurrence expands, every entry rewrites W = (W - 1) + sign * v on its path."""
    done = 0
    while done < num_searches:
        k_this = min(K, num_searches - done)
        for t in trees:
            pend = []                                            # (leaf, index of the first occurrence or -1, path)
            for _ in range(k_this):
                nid, path = 0, [0]
                while t.arena[nid]["children"]:
                    nid = t.select(nid)
                    path.append(nid)
                st = t.arena[nid]["state"]
                if st.status != 0:
                    t.backprop(nid, _terminal_value(st))
                    continue
                dup = next((j for j, e in enumerate(pend) if e[1] < 0 and e[0] == nid), -1)
                for i in path:
                    t.arena[i]["N"] += 1
                    t.arena[i]["W"] = F(t.arena[i]["W"] + F(1))
                pend.append((nid, dup, path))
            values = {}
            for j, (leaf, dup, path) in enumerate(pend):
                if dup < 0:
                    st = t.arena[leaf]["state"]
                    probs, values[j] = evaluator(st)
                    t.expand(leaf, pyref.mask(st, probs))
                v = values[j if dup < 0 else dup]
                sign = F(1)
                for i in reversed(path):
                    t.arena[i]["W"] = F(F(t.arena[i]["W"] - F(1)) + F(sign * v))
                    sign = F(-sign)
        done += k_this


def synthetic_root(game, g, max_ply):
    """helpers.synthetic_root as (oracle State, pyref state): the same seeded playout applied to both."""
    while True:
        r = pyref.splitmix64(0x5EED0000 + g)
        plies = r % max_ply
        s = O.State()
        p = pyref.C4() if game == O.GAME_C4 else pyref.TTT()
        ok = True
        for _ in range(plies):
            va = O.valid_actions(game, s)
            r = pyref.splitmix64(r)
            a = va[r % len(va)]
            s = O.next_state(game, s, a)
            p = p.next_state(a)
            if s.status != O.ONGOING:
                ok = False
                break
        if ok:
            return s, p
        g += 1 << 32


def table(t):
    """Node records of a pyref tree as spb_node_stats reports them (a root's prior is 0; a leaf's first child is 0)."""
    return [dict(visit_count=n["N"], value_sum=float(n["W"]), prior=0.0 if n["prior"] is None else float(n["prior"]),
                 first_child=n["children"][0] if n["children"] else 0, n_children=len(n["children"])) for n in t.arena]


def root_children(t):
    ch = t.arena[0]["children"]
    return [t.arena[c]["action"] for c in ch], [t.arena[c]["N"] for c in ch], list(ch)
