"""CPU restatement of halo2_proofs' create_proof / verify_proof with SEVERAL circuits of one constraint system in one proof
(`circuits: &[C]`, `instances: &[&[&[Fr]]]`), on top of oracle/halo2_ref.py's single-circuit `Ref` (TEST INFRASTRUCTURE ONLY).

Follows halo2_proofs 1.1.0 = scroll-tech/halo2 v1.1 @ e5ddf67 plonk/prover.rs, plonk/verifier.rs and plonk/evaluation.rs, restated.
With C circuits, in transcript order:
  1. vk.transcript_repr, then the instance values circuit-major (KZG: QUERY_INSTANCE = false);
  2. per phase: every circuit's advice commitments of that phase (circuit-major), then the phase's challenges, shared by all;
  3. theta; every circuit's m commitments;  4. beta, gamma; every circuit's z commitments (the chain z_i[0] = last(z_{i-1}) runs
     within one circuit; every circuit's first set starts at 1);  5. every circuit's phi commitments;  6. one random polynomial, y;
  7. ONE quotient: evaluate_h keeps folding into the same accumulator across the circuits, so h = sum_c A_c y^(K (C - 1 - c));
  8. evaluations: every circuit's advice queries, the fixed queries, the random polynomial, sigma, every circuit's z, every
     circuit's lookups;  9. SHPLONK queries: per circuit [advice; z; lookups], then fixed, sigma, h, random.
With one circuit this is exactly Ref.create_proof / Ref.verify_proof (tests/test_oracle_prover_multi.py checks the bytes).
"""
import numpy as np

import pyref as P
import halo2_ref as H
from halo2_ref import FIXED, ADVICE, INSTANCE, R, rot


def create_proof_multi(ref, pk, transcript_repr, instances, synthesize, blinds, transcript=None):
    """instances: per circuit, a list (per instance column) of lists of ints.
    synthesize(circuit, phase, challenges) -> dict advice column -> (n,4) array (blinded), for that circuit and phase.
    blinds: 'z' [C][sets][bf] ints, 'phi' [C][lookups][bf] ints, 'random_poly' (n,4) array (one for the proof).
    Returns (proof bytes, debug dict)."""
    F, cs, dom, n, bf = ref.F, ref.cs, ref.dom, ref.cs.n, ref.bf
    C = len(instances)
    tr = transcript or H.Ref.Transcript(ref)
    tr.common_scalar(transcript_repr)
    inst_values = []
    for inst in instances:
        vals = []
        for col in inst:
            assert len(col) <= n - (bf + 1)
            for v in col: tr.common_scalar(v % R)
            a = np.zeros((n, 4), dtype=np.uint64)
            if col: a[: len(col)] = F.arr(col)
            vals.append(a)
        inst_values.append(vals)
    inst_polys = [[ref.lagrange_to_coeff(a) for a in vals] for vals in inst_values]
    adv_values = [[None] * cs.num_advice for _ in range(C)]
    challenges = {}
    for phase in range(cs.num_phases()):
        for c in range(C):
            cols = synthesize(c, phase, dict(challenges))
            for j in range(cs.num_advice):
                if cs.advice_phase[j] == phase:
                    adv_values[c][j] = np.ascontiguousarray(cols[j])
                    tr.write_point(ref.commit_lagrange(adv_values[c][j]))
        for ci, ph in enumerate(cs.challenge_phase):
            if ph == phase: challenges[ci] = tr.squeeze()
    theta = tr.squeeze()
    vals = [{FIXED: pk["fixed_values"], ADVICE: adv_values[c], INSTANCE: inst_values[c]} for c in range(C)]
    one = ref.w_arr(1)
    usable = n - bf - 1
    lk_data = []          # [circuit][lookup] = (inputs, table, m)
    for c in range(C):
        per = []
        for li, lk in enumerate(cs.lookups):
            fs = [ref.compress(inp, theta, vals[c], challenges, n, 1) for inp in lk.inputs]
            t = ref.compress(lk.table, theta, vals[c], challenges, n, 1)
            index = {r.tobytes(): i for i, r in enumerate(t[:usable])}    # the last duplicate table row wins
            m = [0] * n
            for f in fs:
                for r in f[:usable]:
                    key = r.tobytes()
                    if key not in index:
                        raise KeyError(f"circuit {c}, lookup {li}: an input row is not in the table")
                    m[index[key]] += 1
            per.append((fs, t, F.arr(m)))
        lk_data.append(per)
    for c in range(C):
        for (_, _, m_arr) in lk_data[c]: tr.write_point(ref.commit_lagrange(m_arr))
    beta = tr.squeeze(); gamma = tr.squeeze()
    pcols = cs.perm_columns
    omega_pows = F.powers(dom.omega, n)
    zs = []               # [circuit][set]
    for c in range(C):
        last_z, delta_pow, zc = one.copy(), 1, []
        for ci in range(0, len(pcols), ref.chunk):
            den = np.repeat(one[None], n, axis=0)
            num = np.repeat(one[None], n, axis=0)
            for j, (t_, i_) in enumerate(pcols[ci: ci + ref.chunk]):
                v = vals[c][t_][i_]
                den = F.mul(den, F.addc(F.add(v, F.scal(pk["sigma_values"][ci + j], beta)), gamma))
                num = F.mul(num, F.addc(F.add(v, F.scal(omega_pows, beta * delta_pow % R)), gamma))
                delta_pow = delta_pow * P.FR_DELTA % R
            zi = F.ints(F.mul(num, F.inv(den)))
            cur = F.ints(last_z[None])[0]
            zl = [cur]
            for row in range(1, n):
                cur = cur * zi[row - 1] % R
                zl.append(cur)
            z = F.arr(zl)
            z[n - bf:] = F.arr(blinds["z"][c][ci // ref.chunk])
            last_z = z[n - bf - 1].copy()
            zc.append(z)
        zs.append(zc)
    z_polys = [[ref.lagrange_to_coeff(z) for z in zc] for zc in zs]
    for zc in zs:
        for z in zc: tr.write_point(ref.commit_lagrange(z))
    phis = []             # [circuit][lookup]
    for c in range(C):
        pc = []
        for li, (fs, t, m_arr) in enumerate(lk_data[c]):
            acc = F.neg(F.mul(m_arr, F.inv(F.addc(t, beta))))
            for f in fs: acc = F.add(acc, F.inv(F.addc(f, beta)))
            ai = F.ints(acc)
            ph = [0]
            for row in range(1, n - bf): ph.append((ph[-1] + ai[row - 1]) % R)
            ph += [b % R for b in blinds["phi"][c][li]]
            pc.append(F.arr(ph))
        phis.append(pc)
    for pc in phis:
        for p_ in pc: tr.write_point(ref.commit_lagrange(p_))
    m_polys = [[ref.lagrange_to_coeff(d[2]) for d in per] for per in lk_data]
    phi_polys = [[ref.lagrange_to_coeff(p_) for p_ in pc] for pc in phis]
    random_poly = np.ascontiguousarray(blinds["random_poly"])
    tr.write_point(ref.commit(random_poly))
    y = tr.squeeze()
    adv_polys = [[ref.lagrange_to_coeff(a) for a in av] for av in adv_values]
    # ---- one quotient: every circuit's constraints continue the Horner chain in y
    N, E = dom.N, dom.E
    fixed_ext = [ref.coeff_to_extended(p_) for p_ in pk["fixed_polys"]]
    sig_ext = [ref.coeff_to_extended(p_) for p_ in pk["sigma_polys"]]
    l0 = ref.coeff_to_extended(pk["l0"]); llast = ref.coeff_to_extended(pk["l_last"]); lblind = ref.coeff_to_extended(pk["l_blind"])
    onesN = np.repeat(one[None], N, axis=0)
    lactive = F.sub(F.sub(onesN, llast), lblind)
    xs = F.scal(F.powers(dom.extended_omega, N), P.FR_ZETA)
    h = np.zeros((N, 4), dtype=np.uint64)

    def fold(term):
        nonlocal h
        h = F.add(F.scal(h, y), term)
    for c in range(C):
        ext = {FIXED: fixed_ext, ADVICE: [ref.coeff_to_extended(p_) for p_ in adv_polys[c]],
               INSTANCE: [ref.coeff_to_extended(p_) for p_ in inst_polys[c]]}
        for g in cs.gates: fold(ref.eval_expr(g, ext, challenges, N, E))
        if zs[c]:
            z_ext = [ref.coeff_to_extended(p_) for p_ in z_polys[c]]
            fold(F.mul(F.sub(onesN, z_ext[0]), l0))
            fold(F.mul(F.sub(F.mul(z_ext[-1], z_ext[-1]), z_ext[-1]), llast))
            for i in range(1, len(z_ext)): fold(F.mul(F.sub(z_ext[i], rot(z_ext[i - 1], -(bf + 1), E)), l0))
            delta_pow = 1
            for si, ze in enumerate(z_ext):
                left, right = rot(ze, 1, E), ze
                for j, (t_, i_) in enumerate(pcols[si * ref.chunk: (si + 1) * ref.chunk]):
                    v = ext[t_][i_]
                    left = F.mul(left, F.addc(F.add(v, F.scal(sig_ext[si * ref.chunk + j], beta)), gamma))
                    right = F.mul(right, F.addc(F.add(v, F.scal(xs, beta * delta_pow % R)), gamma))
                    delta_pow = delta_pow * P.FR_DELTA % R
                fold(F.mul(F.sub(left, right), lactive))
        for li, lk in enumerate(cs.lookups):
            phi_e = ref.coeff_to_extended(phi_polys[c][li]); m_e = ref.coeff_to_extended(m_polys[c][li])
            fsb = [F.addc(ref.compress(inp, theta, ext, challenges, N, E), beta) for inp in lk.inputs]
            tb = F.addc(ref.compress(lk.table, theta, ext, challenges, N, E), beta)
            prod = fsb[0]
            for f in fsb[1:]: prod = F.mul(prod, f)
            ssum = np.zeros((N, 4), dtype=np.uint64)
            for i in range(len(fsb)):
                pr = None
                for j in range(len(fsb)):
                    if j != i: pr = fsb[j] if pr is None else F.mul(pr, fsb[j])
                ssum = F.add(ssum, onesN if pr is None else pr)
            lhs = F.mul(F.mul(tb, prod), F.sub(rot(phi_e, 1, E), phi_e))
            rhs = F.sub(F.mul(tb, ssum), F.mul(m_e, prod))
            fold(F.mul(phi_e, l0)); fold(F.mul(phi_e, llast)); fold(F.mul(F.sub(lhs, rhs), lactive))
    tinv = F.inv(F.arr(dom.t_evaluations))
    h_coeffs = ref.extended_to_coeff(F.mul(h, tinv[np.arange(N) % E]))
    pieces = [np.ascontiguousarray(h_coeffs[i * n: (i + 1) * n]) for i in range(dom.qdeg)]
    for pc in pieces: tr.write_point(ref.commit(pc))
    x = tr.squeeze()
    xn = pow(x, n, R)
    x_next, x_last = dom.rotate_omega(x, 1), dom.rotate_omega(x, -(bf + 1))
    # ---- evaluations
    for c in range(C):
        for (j, r) in cs.advice_queries: tr.write_scalar(ref.eval_poly(adv_polys[c][j], dom.rotate_omega(x, r)))
    for (j, r) in cs.fixed_queries: tr.write_scalar(ref.eval_poly(pk["fixed_polys"][j], dom.rotate_omega(x, r)))
    tr.write_scalar(ref.eval_poly(random_poly, x))
    for sp in pk["sigma_polys"]: tr.write_scalar(ref.eval_poly(sp, x))
    for c in range(C):
        for i, zp in enumerate(z_polys[c]):
            tr.write_scalar(ref.eval_poly(zp, x)); tr.write_scalar(ref.eval_poly(zp, x_next))
            if i != len(z_polys[c]) - 1: tr.write_scalar(ref.eval_poly(zp, x_last))
    for c in range(C):
        for li in range(len(cs.lookups)):
            tr.write_scalar(ref.eval_poly(phi_polys[c][li], x)); tr.write_scalar(ref.eval_poly(phi_polys[c][li], x_next))
            tr.write_scalar(ref.eval_poly(m_polys[c][li], x))
    h_poly = np.zeros((n, 4), dtype=np.uint64)
    for pc in reversed(pieces): h_poly = F.add(F.scal(h_poly, xn), pc)
    # ---- multiopen queries: per circuit [advice; z; lookups], then fixed, sigma, h, random
    queries = []
    for c in range(C):
        for (j, r) in cs.advice_queries: queries.append((("adv", c, j), adv_polys[c][j], dom.rotate_omega(x, r)))
        for i, zp in enumerate(z_polys[c]):
            queries.append((("z", c, i), zp, x)); queries.append((("z", c, i), zp, x_next))
        for i in range(len(z_polys[c]) - 2, -1, -1): queries.append((("z", c, i), z_polys[c][i], x_last))
        for li in range(len(cs.lookups)):
            queries.append((("phi", c, li), phi_polys[c][li], x)); queries.append((("phi", c, li), phi_polys[c][li], x_next))
            queries.append((("m", c, li), m_polys[c][li], x))
    for (j, r) in cs.fixed_queries: queries.append((("fix", j), pk["fixed_polys"][j], dom.rotate_omega(x, r)))
    for i, sp in enumerate(pk["sigma_polys"]): queries.append((("sig", i), sp, x))
    queries.append((("h",), h_poly, x)); queries.append((("rand",), random_poly, x))
    ref.shplonk_prove(tr, queries)
    return bytes(tr.buf), dict(theta=theta, beta=beta, gamma=gamma, y=y, x=x, challenges=challenges, zs=zs, phis=phis)


def verify_proof_multi(ref, pk, transcript_repr, instances, proof, reader=None):
    """Checks ONE folded identity h(x) (x^n - 1) = sum_c A_c(x) y^(K (C - 1 - c)) over all circuits, then the SHPLONK opening
    (known-s trapdoor check, as Ref.verify_proof).  instances: per circuit, per instance column, lists of ints."""
    cs, dom, n, bf = ref.cs, ref.dom, ref.cs.n, ref.bf
    C = len(instances)
    rd = reader or H.Ref.Reader(ref, proof)
    rd.common_scalar(transcript_repr)
    for inst in instances:
        assert len(inst) == cs.num_instance
        for col in inst:
            for v in col: rd.common_scalar(v % R)
    adv_c = [[None] * cs.num_advice for _ in range(C)]
    challenges = {}
    for phase in range(cs.num_phases()):
        for c in range(C):
            for j in range(cs.num_advice):
                if cs.advice_phase[j] == phase: adv_c[c][j] = rd.read_point()
        for ci, ph in enumerate(cs.challenge_phase):
            if ph == phase: challenges[ci] = rd.squeeze()
    theta = rd.squeeze()
    nl = len(cs.lookups)
    m_c = [[rd.read_point() for _ in range(nl)] for _ in range(C)]
    beta = rd.squeeze(); gamma = rd.squeeze()
    nsets = (len(cs.perm_columns) + ref.chunk - 1) // ref.chunk
    z_c = [[rd.read_point() for _ in range(nsets)] for _ in range(C)]
    phi_c = [[rd.read_point() for _ in range(nl)] for _ in range(C)]
    rand_c = rd.read_point()
    y = rd.squeeze()
    h_c = [rd.read_point() for _ in range(dom.qdeg)]
    x = rd.squeeze()
    xn = pow(x, n, R)

    def lag(i):
        wi = pow(dom.omega, i % n, R)
        return (xn - 1) * wi % R * pow(n * (x - wi) % R, -1, R) % R
    ev = [{} for _ in range(C)]
    for c in range(C):
        for (j, r) in cs.instance_queries:
            ev[c][(INSTANCE, j, r)] = sum(v * lag(i - r) for i, v in enumerate(instances[c][j])) % R
    for c in range(C):
        for (j, r) in cs.advice_queries: ev[c][(ADVICE, j, r)] = rd.read_scalar()
    fix_ev = {(FIXED, j, r): rd.read_scalar() for (j, r) in cs.fixed_queries}
    for c in range(C): ev[c].update(fix_ev)
    rand_eval = rd.read_scalar()
    sig_ev = [rd.read_scalar() for _ in cs.perm_columns]
    z_ev = []
    for c in range(C):
        zc = []
        for i in range(nsets):
            a = rd.read_scalar(); b = rd.read_scalar()
            zc.append((a, b, rd.read_scalar() if i != nsets - 1 else None))
        z_ev.append(zc)
    lk_ev = [[(rd.read_scalar(), rd.read_scalar(), rd.read_scalar()) for _ in range(nl)] for _ in range(C)]
    l0 = lag(0); llast = lag(n - bf - 1); lblind = sum(lag(i) for i in range(n - bf, n)) % R
    lactive = (1 - llast - lblind) % R
    acc = 0

    def fold(t):
        nonlocal acc
        acc = (acc * y + t) % R
    for c in range(C):
        for g in cs.gates: fold(ref.eval_expr_at(g, ev[c], challenges))
        if nsets:
            fold(l0 * (1 - z_ev[c][0][0]) % R)
            zl = z_ev[c][-1][0]
            fold(llast * (zl * zl - zl) % R)
            for i in range(1, nsets): fold(l0 * (z_ev[c][i][0] - z_ev[c][i - 1][2]) % R)
            dp = 1
            for si in range(nsets):
                left, right = z_ev[c][si][1], z_ev[c][si][0]
                for j, (t_, i_) in enumerate(cs.perm_columns[si * ref.chunk: (si + 1) * ref.chunk]):
                    v = ev[c][(t_, i_, 0)]
                    left = left * (v + beta * sig_ev[si * ref.chunk + j] + gamma) % R
                    right = right * (v + beta * dp % R * x + gamma) % R
                    dp = dp * P.FR_DELTA % R
                fold(lactive * (left - right) % R)
        for li, lk in enumerate(cs.lookups):
            phi_x, phi_nx, m_x = lk_ev[c][li]

            def comp(exprs):
                a = 0
                for e in exprs: a = (a * theta + ref.eval_expr_at(e, ev[c], challenges)) % R
                return a
            fsb = [(comp(inp) + beta) % R for inp in lk.inputs]
            tb = (comp(lk.table) + beta) % R
            prod = 1
            for f in fsb: prod = prod * f % R
            ssum = 0
            for i in range(len(fsb)):
                pr = 1
                for j in range(len(fsb)):
                    if j != i: pr = pr * fsb[j] % R
                ssum = (ssum + pr) % R
            lhs = tb * prod % R * (phi_nx - phi_x) % R
            rhs = (tb * ssum - m_x * prod) % R
            fold(l0 * phi_x % R); fold(llast * phi_x % R); fold(lactive * (lhs - rhs) % R)
    expected_h = acc * pow(xn - 1, -1, R) % R
    hc = None
    for c_ in reversed(h_c): hc = P.g1_add(P.g1_mul(hc, xn) if hc else None, c_)
    x_next, x_last = dom.rotate_omega(x, 1), dom.rotate_omega(x, -(bf + 1))
    queries = []
    for c in range(C):
        for (j, r) in cs.advice_queries: queries.append((("adv", c, j), adv_c[c][j], dom.rotate_omega(x, r), ev[c][(ADVICE, j, r)]))
        for i in range(nsets):
            queries.append((("z", c, i), z_c[c][i], x, z_ev[c][i][0])); queries.append((("z", c, i), z_c[c][i], x_next, z_ev[c][i][1]))
        for i in range(nsets - 2, -1, -1): queries.append((("z", c, i), z_c[c][i], x_last, z_ev[c][i][2]))
        for li in range(nl):
            queries.append((("phi", c, li), phi_c[c][li], x, lk_ev[c][li][0])); queries.append((("phi", c, li), phi_c[c][li], x_next, lk_ev[c][li][1]))
            queries.append((("m", c, li), m_c[c][li], x, lk_ev[c][li][2]))
    pt = lambda c_: c_ if isinstance(c_, tuple) else ref.aff_to_pt(c_)    # vk commitments: affine limbs, or (x, y) points
    for (j, r) in cs.fixed_queries: queries.append((("fix", j), pt(pk["fixed_commitments"][j]), dom.rotate_omega(x, r), fix_ev[(FIXED, j, r)]))
    for i in range(len(cs.perm_columns)): queries.append((("sig", i), pt(pk["sigma_commitments"][i]), x, sig_ev[i]))
    queries.append((("h",), hc, x, expected_h)); queries.append((("rand",), rand_c, x, rand_eval))
    yv = rd.squeeze(); v = rd.squeeze()
    h1 = rd.read_point(); u = rd.squeeze(); h2 = rd.read_point()
    assert rd.pos == len(proof), "trailing bytes"
    evalmap = {(k_, p_): e_ for k_, _, p_, e_ in queries}
    rsets, super_pts = ref.intermediate_sets([(k_, c_, p_) for k_, c_, p_, _ in queries])
    outer = None; r_outer = 0; z0 = 0; z0_diff_inv = 0
    vpow = 1
    for i, (points, comms) in enumerate(rsets):
        zd = 1
        for p_ in super_pts:
            if p_ not in points: zd = zd * (u - p_) % R
        if i == 0:
            z0 = 1
            for p_ in points: z0 = z0 * (u - p_) % R
            z0_diff_inv = pow(zd, -1, R); zd = 1
        else:
            zd = zd * z0_diff_inv % R
        inner = None; r_inner = 0; ypow = 1
        for key, cpt in comms:
            r_ = ref.lagrange_interpolate(points, [evalmap[(key, p_)] for p_ in points])
            r_u = 0
            for cc in reversed(r_): r_u = (r_u * u + cc) % R
            r_inner = (r_inner + ypow * r_u) % R
            inner = P.g1_add(inner, P.g1_mul(cpt, ypow))
            ypow = ypow * yv % R
        outer = P.g1_add(outer, P.g1_mul(inner, vpow * zd % R))
        r_outer = (r_outer + vpow * r_inner % R * zd) % R
        vpow = vpow * v % R
    right = P.g1_add(outer, P.g1_mul(P.G1_GEN, (-r_outer) % R))
    right = P.g1_add(right, P.g1_mul(h1, (-z0) % R))
    right = P.g1_add(right, P.g1_mul(h2, u))
    return P.g1_mul(h2, ref.s) == right


def verify_ok(ref, pk, transcript_repr, instances, proof, reader=None):
    """verify_proof_multi, with a malformed proof (failed assertion while reading) counted as a rejection"""
    try:
        return verify_proof_multi(ref, pk, transcript_repr, instances, proof, reader=reader)
    except (AssertionError, ValueError, TypeError, KeyError, IndexError):
        return False
