"""CPU: the oracle's create_proof over several circuits of one proving key (halo2_multi.py).  With one circuit it writes exactly
the single-circuit oracle's bytes; with several, its verifier accepts the proof and rejects tampered ones."""
import pytest

import halo2_ref as H
import halo2_multi as M
from circuits import ToyCircuit, ThinCompressionShape, GatesOnlyCircuit
from multi_circuits import variants


def setup(tcs, srs_s=1234):
    """oracle, proving key, transcript_repr, per-circuit instances, synthesize(c, phase, ch) and blinds for circuits sharing a key"""
    tc0 = tcs[0]
    ref = H.Ref(tc0.cs, srs_s)
    F = ref.F
    pk = ref.keygen([F.arr(c) for c in tc0.fixed_ints], tc0.copies)
    blinds = {"z": [tc.blinds_ints["z"] for tc in tcs], "phi": [tc.blinds_ints["phi"] for tc in tcs],
              "random_poly": F.arr(tc0.blinds_ints["random_poly"])}
    synth = lambda c, phase, ch: {j: F.arr(v) for j, v in tcs[c].advice_ints(phase, ch).items()}
    return ref, pk, tc0.transcript_repr, [tc.instances for tc in tcs], synth, blinds


def prove(tcs, **kw):
    ref, pk, repr_, inst, synth, blinds = setup(tcs)
    proof, dbg = M.create_proof_multi(ref, pk, repr_, inst, synth, blinds, **kw)
    return ref, pk, repr_, inst, proof


@pytest.mark.parametrize("kind,k", [("toy", 5), ("toy", 6), ("thin", 6), ("gates", 5)])
def test_one_circuit_is_the_single_circuit_proof(kind, k):
    tc = {"toy": ToyCircuit, "thin": ThinCompressionShape, "gates": GatesOnlyCircuit}[kind](k, seed=50 + k)
    ref, pk, repr_, inst, synth, blinds = setup([tc])
    proof, _ = M.create_proof_multi(ref, pk, repr_, inst, synth, blinds)
    F = ref.F
    single, _ = ref.create_proof(pk, repr_, tc.instances, lambda ph, ch: {c: F.arr(v) for c, v in tc.advice_ints(ph, ch).items()},
                                 {"z": tc.blinds_ints["z"], "phi": tc.blinds_ints["phi"], "random_poly": blinds["random_poly"]})
    assert proof == single
    assert M.verify_proof_multi(ref, pk, repr_, inst, proof)
    assert ref.verify_proof(pk, repr_, tc.instances, proof)


@pytest.mark.parametrize("count", [2, 3])
def test_several_toy_circuits_verify(count):
    tcs = variants("toy", 5, count, seed=count)
    assert tcs[0].two_phase and tcs[0].cs.lookups and len(tcs[0].cs.perm_columns) == 8   # two phases, lookups, a second permutation set
    assert len({tuple(tc.instances[0]) for tc in tcs}) == count
    ref, pk, repr_, inst, proof = prove(tcs)
    assert M.verify_proof_multi(ref, pk, repr_, inst, proof)
    cs = tcs[0].cs
    nsets = (len(cs.perm_columns) + ref.chunk - 1) // ref.chunk
    npoints = count * (cs.num_advice + 2 * len(cs.lookups) + nsets) + 1 + ref.dom.qdeg + 2
    nevals = count * (len(cs.advice_queries) + 3 * nsets - 1 + 3 * len(cs.lookups)) + len(cs.fixed_queries) + 1 + len(cs.perm_columns)
    assert len(proof) == 32 * (npoints + nevals)


def test_several_circuits_rejections():
    tcs = variants("toy", 5, 2, seed=9)
    ref, pk, repr_, inst, proof = prove(tcs)
    assert M.verify_proof_multi(ref, pk, repr_, inst, proof)
    # circuit 1's first advice commitment follows circuit 0's five phase-0 commitments
    bad = bytearray(proof)
    bad[32 * 5 + 3] ^= 1
    assert not M.verify_ok(ref, pk, repr_, inst, bytes(bad))
    assert not M.verify_ok(ref, pk, repr_, [inst[1], inst[0]], proof)
    assert not M.verify_ok(ref, pk, repr_, inst[:1], proof)


def test_unsatisfied_lookup_in_one_circuit_raises():
    tcs = variants("toy", 5, 2, seed=4)
    bad = tcs[1]
    for i in range(bad.usable):
        if bad.fixed_ints[2][i]:
            bad.cols0[3][i] = 123456789
            break
    with pytest.raises(KeyError, match="circuit 1"):
        prove(tcs)
