"""Several circuits of ONE constraint system and proving key (create_proof's `circuits: &[C]`): the same fixed columns and copy
constraints, each circuit with its own witness, instance values and blinding scalars.  Test infrastructure for the multi-circuit
proof tests."""
import random

import pyref as P
from halo2_ref import FIXED, ADVICE, INSTANCE
from circuits import ToyCircuit, GatesOnlyCircuit, ThinCompressionShape

R = P.R_MOD


class ToyVariant(ToyCircuit):
    """ToyCircuit whose structure (selectors, fixed columns, copy constraints) is drawn from `seed` and whose values (witness,
    instances, blinds) from `value_seed`: variants with one seed and different value seeds share a proving key."""

    def __init__(self, k, seed=0, value_seed=0, two_phase=True, lookups=True, n_instance=4, extra_perm=True):
        base = ToyCircuit(k, seed=seed, two_phase=two_phase, lookups=lookups, n_instance=n_instance, extra_perm=extra_perm)
        self.k, self.n, self.two_phase, self.cs = base.k, base.n, two_phase, base.cs
        self.bf, self.usable, self.fixed_ints = base.bf, base.usable, base.fixed_ints
        n, usable, fixed = self.n, self.usable, self.fixed_ints
        rs = random.Random(seed * 7919 + 1)       # structure: copy constraints
        rv = random.Random(value_seed)           # values
        T = max(2, min(usable, 1 << max(1, k - 2)))
        q_mul, q_add, q_lk, q_lk2 = fixed[0], fixed[1], fixed[2], fixed[3]
        self.instances = [[rv.randrange(R) for _ in range(n_instance)]]
        A = [rv.randrange(R) for _ in range(n)]
        B = [rv.randrange(R) for _ in range(n)]
        C = [rv.randrange(R) for _ in range(n)]
        copies = []
        for i in range(usable):
            t = rs.random()
            if i > 2 and t < 0.25:
                j = rs.randrange(i)
                A[i] = C[j]; copies.append(((ADVICE, 0, i), (ADVICE, 2, j)))
            elif t < 0.35 and n_instance:
                j = rs.randrange(n_instance)
                A[i] = self.instances[0][j]; copies.append(((ADVICE, 0, i), (INSTANCE, 0, j)))
            elif t < 0.45:
                j = rs.randrange(usable)
                A[i] = fixed[7][j]; copies.append(((ADVICE, 0, i), (FIXED, 7, j)))
            if i > 0 and q_add[i - 1]:
                pass
            elif i > 2 and rs.random() < 0.2:
                j = rs.randrange(i)
                B[i] = B[j]; copies.append(((ADVICE, 1, i), (ADVICE, 1, j)))
            if q_mul[i]: C[i] = A[i] * B[i] % R
            if i > 0 and q_add[i - 1]: C[i] = (A[i - 1] + B[i]) % R
        # lookup columns: rows linked by a copy constraint hold the same table row (union-find over the structural pairs)
        parent = list(range(usable))

        def find(a):
            while parent[a] != a:
                parent[a] = parent[parent[a]]; a = parent[a]
            return a
        if extra_perm:
            for _ in range(max(1, usable // 8)):
                i, j = rs.randrange(usable), rs.randrange(usable)
                if i == j: continue
                parent[find(i)] = find(j)
                copies.append(((ADVICE, 3, i), (ADVICE, 3, j))); copies.append(((ADVICE, 4, i), (ADVICE, 4, j)))
        row_of = {}
        D, E = [0] * n, [0] * n
        for i in range(usable):
            r = find(i)
            if r not in row_of: row_of[r] = rv.randrange(T)
            D[i], E[i] = fixed[4][row_of[r]], fixed[5][row_of[r]]
        self.copies = copies
        self.cols0 = [A, B, C, D, E]
        self.rnd = rv
        self.blind_rows = {c: [rv.randrange(R) for _ in range(self.bf + 1)] for c in range(6)}
        cs = self.cs
        nsets = (len(cs.perm_columns) + (cs.degree() - 2) - 1) // (cs.degree() - 2)
        self.blinds_ints = {"z": [[rv.randrange(R) for _ in range(self.bf)] for _ in range(nsets)],
                            "phi": [[rv.randrange(R) for _ in range(self.bf)] for _ in cs.lookups],
                            "random_poly": [rv.randrange(R) for _ in range(n)]}
        self.transcript_repr = base.transcript_repr


class ThinVariant(ThinCompressionShape):
    """ThinCompressionShape with another witness on the SAME fixed columns and copy constraints: the gate rows keep their layout,
    the gate inputs and range-checked cells get new values (the copied cells follow their copies)."""

    def __init__(self, k, seed=0, value_seed=0, n_instance=6):
        base = ThinCompressionShape(k, seed=seed, n_instance=n_instance)
        self.__dict__.update(base.__dict__)
        rv = random.Random(value_seed)
        n, usable, fixed = self.n, self.usable, self.fixed_ints
        T = 1 << max(2, k - 2)
        self.instances = [[rv.randrange(R) for _ in range(n_instance)]]
        A = [rv.randrange(T) for _ in range(n)]
        pinned = {}          # advice row -> instance index / fixed row it is copied from
        for (lt, lc, lr), (rt, rc, rr) in base.copies:
            if rt == INSTANCE: pinned[lr] = ("inst", rr)
            elif rt == FIXED: pinned[lr] = ("fix", rr)
        r = 0
        while r < usable:
            if fixed[2][r]:
                A[r], A[r + 1], A[r + 2] = rv.randrange(R), rv.randrange(R), rv.randrange(R)
                if r in pinned:
                    kind, j = pinned[r]
                    A[r] = self.instances[0][j] if kind == "inst" else fixed[1][j]
                A[r + 3] = (A[r] + A[r + 1] * A[r + 2]) % R
                r += 4
            else:
                r += 1
        # advice-advice copies of the base witness held equal values; keep only those that still hold (both in one cycle class)
        self.copies = [cp for cp in base.copies if cp[1][0] != ADVICE]
        self.A = A
        self.blind = [rv.randrange(R) for _ in range(self.bf + 1)]
        self.blinds_ints = {"z": [[rv.randrange(R) for _ in range(self.bf)]], "phi": [[rv.randrange(R) for _ in range(self.bf)]],
                            "random_poly": [rv.randrange(R) for _ in range(n)]}


def variants(kind, k, count, seed=0, **kw):
    """`count` circuits sharing one constraint system, fixed columns and copy constraints"""
    if kind == "toy":
        return [ToyVariant(k, seed=seed, value_seed=1000 * seed + 17 * c + 1, **kw) for c in range(count)]
    if kind == "thin":
        # advice-advice copies depend on the witness: every variant uses the copies without them (the same for all)
        return [ThinVariant(k, seed=seed, value_seed=1000 * seed + 17 * c + 1, **kw) for c in range(count)]
    if kind == "gates":      # GatesOnlyCircuit's selector does not depend on the seed
        return [GatesOnlyCircuit(k, seed=1000 * seed + 17 * c + 1, **kw) for c in range(count)]
    raise ValueError(kind)
