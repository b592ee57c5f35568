"""GPU: create_proof over several circuits of one proving key (zkb_prove_begin_multi, plonk.create_proof_multi) writes the bytes of
the CPU oracle's multi-circuit prover (halo2_multi.py), and the oracle verifier accepts them."""
import numpy as np
import pytest

import halo2_ref as H
import halo2_multi as M
from multi_circuits import variants
from test_gpu_prover import to_product_cs, first_diff
from test_oracle_prover_multi import setup

pytestmark = pytest.mark.gpu


def gpu_args(tcs, ref, pkr):
    """(pk, transcript_repr, instances, synthesize, z_blinds, phi_blinds, random_poly) for plonk.create_proof_multi"""
    from zkb200 import plonk as Z
    F = ref.F
    tc0 = tcs[0]
    pk = Z.ProvingKey(to_product_cs(tc0.cs, ref.bf, ref.d), pkr["fixed_values"], pkr["sigma_values"], ref.g, ref.g_lagrange)

    def synth(c, phase, ch):
        chi = {i: F.ints(v[None])[0] for i, v in ch.items()}
        return {j: F.arr(v) for j, v in tcs[c].advice_ints(phase, chi).items()}
    zb = [F.arr(b) for tc in tcs for b in tc.blinds_ints["z"]]
    pb = [F.arr(b) for tc in tcs for b in tc.blinds_ints["phi"]]
    return (pk, F.arr([tc0.transcript_repr])[0], [[F.arr(c) for c in tc.instances] for tc in tcs], synth,
            np.concatenate(zb) if zb else None, np.concatenate(pb) if pb else None, F.arr(tc0.blinds_ints["random_poly"]))


CASES = [("toy", 6, 2), ("toy", 6, 3), ("toy", 8, 2), ("toy", 8, 3), ("thin", 7, 2), ("thin", 7, 3), ("gates", 5, 2), ("gates", 5, 3)]


@pytest.mark.parametrize("kind,k,count", CASES)
def test_multi_circuit_proof_matches_oracle(kind, k, count):
    from zkb200 import plonk as Z
    tcs = variants(kind, k, count, seed=k)
    ref, pkr, repr_, inst, synth_ref, blinds = setup(tcs)
    proof_ref, _ = M.create_proof_multi(ref, pkr, repr_, inst, synth_ref, blinds)
    proof = Z.create_proof_multi(*gpu_args(tcs, ref, pkr))
    assert len(proof) == len(proof_ref)
    assert first_diff(proof, proof_ref) is None, f"first differing 32-byte proof item: {first_diff(proof, proof_ref)}"
    assert M.verify_proof_multi(ref, pkr, repr_, inst, proof)


@pytest.mark.parametrize("transcript", ["poseidon", "evm", "callback"])
def test_multi_circuit_transcripts(transcript):
    import keccak_ref as K
    from zkb200 import plonk as Z
    tcs = variants("toy", 6, 2, seed=21)
    ref, pkr, repr_, inst, synth_ref, blinds = setup(tcs)
    F = ref.F
    args = gpu_args(tcs, ref, pkr)
    if transcript == "callback":
        class Mine:
            def __init__(self): self.t = H.Ref.Transcript(ref)
            def common_scalar(self, l): self.t.common_scalar(F.ints(l[None])[0])
            def write_scalar(self, l): self.t.write_scalar(F.ints(l[None])[0])
            def write_point(self, l): self.t.write_point(l)
            def squeeze_challenge(self): return F.arr([self.t.squeeze()])[0]
        mine = Mine()
        assert Z.create_proof_multi(*args, transcript=Z.CallbackTranscript(mine)) == b""
        proof, (proof_ref, _) = bytes(mine.t.buf), M.create_proof_multi(ref, pkr, repr_, inst, synth_ref, blinds)
        reader = None
    else:
        writer = H.Ref.PoseidonTranscript(ref) if transcript == "poseidon" else K.EvmTranscript(ref)
        proof_ref, _ = M.create_proof_multi(ref, pkr, repr_, inst, synth_ref, blinds, transcript=writer)
        proof = Z.create_proof_multi(*args, transcript=transcript)
        reader = H.Ref.PoseidonReader(proof) if transcript == "poseidon" else K.EvmTranscript(proof=proof)
    assert first_diff(proof, proof_ref) is None, f"first differing 32-byte proof item: {first_diff(proof, proof_ref)}"
    assert M.verify_proof_multi(ref, pkr, repr_, inst, proof, reader=reader)


def test_begin_multi_with_one_circuit_and_upload_ahead():
    """zkb_prove_begin_multi with C = 1 writes the bytes of zkb_prove_begin_ex; columns handed over ahead of their phase under their
    circuit-major index give the same proof"""
    from zkb200 import plonk as Z
    tcs = variants("toy", 7, 1, seed=5)
    ref, pkr, *_ = setup(tcs)
    pk, tr, inst, synth, zb, pb, rp = gpu_args(tcs, ref, pkr)
    single = Z.create_proof(pk, tr, inst[0], lambda ph, ch: synth(0, ph, ch), zb, pb, rp)
    assert Z.create_proof_multi(pk, tr, inst, synth, zb, pb, rp) == single
    tcs = variants("toy", 7, 3, seed=5)
    ref, pkr, *_ = setup(tcs)
    args = gpu_args(tcs, ref, pkr)
    assert Z.create_proof_multi(*args, upload_ahead=True) == Z.create_proof_multi(*args)


def test_zero_circuits_is_an_argument_error():
    import ctypes
    from zkb200 import plonk as Z
    tcs = variants("gates", 5, 1, seed=1)
    ref, pkr, *_ = setup(tcs)
    pk = gpu_args(tcs, ref, pkr)[0]
    tr = np.zeros(4, dtype=np.uint64)
    sess = ctypes.c_void_p()
    assert pk.ctx.lib.zkb_prove_begin_multi(pk.handle, 0, None, ctypes.c_void_p(tr.ctypes.data), 0, None, None, ctypes.byref(sess)) == -2


def test_unsatisfied_lookup_in_circuit_1_names_it():
    from zkb200 import plonk as Z, ZkbError
    tcs = variants("toy", 6, 2, seed=8)
    for i in range(tcs[1].usable):
        if tcs[1].fixed_ints[2][i]:
            tcs[1].cols0[3][i] = 123456789
            break
    ref, pkr, *_ = setup(tcs)
    with pytest.raises(ZkbError, match="circuit 1, lookup 0"):
        Z.create_proof_multi(*gpu_args(tcs, ref, pkr))


def test_keccak_standin_two_circuits_match_oracle():
    """the Keccak-shaped stand-in (56 rotations, 58 blinding factors, two-column tables, two phases) at k = 12, two circuits with
    the same fixed / sigma columns and different witnesses"""
    import standins
    from zkb200 import plonk as Z
    from zkb200.params import ParamsKZG
    from test_gpu_prover_wide import to_oracle_cs

    class ValueOps(standins.DeviceOps):   # another witness: the random values come from other seeds, the structure does not change
        def __init__(self, off): super().__init__(); self.off = off
        def rand(self, n, seed): return super().rand(n, seed + self.off)
    k = 12
    scs = [standins.keccak_shape(k, seed=k, scale=0.25, ops=ValueOps(off)) for off in (0, 99991)]
    h = scs[0].host
    assert all((h(a) == h(b)).all() for a, b in zip(scs[0].fixed + scs[0].sigma, scs[1].fixed + scs[1].sigma))
    assert not (h(scs[0].adv0[0]) == h(scs[1].adv0[0])).all()
    params = ParamsKZG.unsafe_setup_with_s(k, 4321)
    fixed, sigma = [h(t) for t in scs[0].fixed], [h(t) for t in scs[0].sigma]
    pk = Z.ProvingKey(scs[0].cs, fixed, sigma, srs=params.load())
    synth = lambda c, phase, ch: {j: h(t) for j, t in scs[c].synthesize_dev(phase, ch).items()}
    zb = np.concatenate([h(sc.z_blinds) for sc in scs]); pb = np.concatenate([h(sc.phi_blinds) for sc in scs])
    proof = Z.create_proof_multi(pk, h(scs[0].transcript_repr[None])[0], [[], []], synth, zb, pb, h(scs[0].random_poly))

    sc0 = scs[0]
    ref = H.Ref(to_oracle_cs(sc0.cs), 4321)
    F = ref.F
    n, bf = sc0.n, sc0.bf
    pkr = {"fixed_values": fixed, "fixed_polys": [ref.lagrange_to_coeff(v) for v in fixed], "sigma_values": sigma,
           "sigma_polys": [ref.lagrange_to_coeff(v) for v in sigma]}
    l0 = np.zeros((n, 4), dtype=np.uint64); l0[0] = ref.w_arr(1)
    lb = np.zeros((n, 4), dtype=np.uint64); lb[n - bf:] = ref.w_arr(1)
    ll = np.zeros((n, 4), dtype=np.uint64); ll[n - bf - 1] = ref.w_arr(1)
    pkr["l0"], pkr["l_last"], pkr["l_blind"] = [ref.lagrange_to_coeff(v) for v in (l0, ll, lb)]
    pkr["fixed_commitments"] = [ref.commit_lagrange(v) for v in fixed]
    pkr["sigma_commitments"] = [ref.commit_lagrange(v) for v in sigma]
    blinds = {"z": [[F.ints(h(sc.z_blinds)[i * bf:(i + 1) * bf]) for i in range(sc.nsets)] for sc in scs],
              "phi": [[F.ints(h(sc.phi_blinds)[i * bf:(i + 1) * bf]) for i in range(sc.L)] for sc in scs],
              "random_poly": h(sc0.random_poly)}
    trep = F.ints(h(sc0.transcript_repr[None]))[0]
    synth_ref = lambda c, phase, ch: {j: h(t) for j, t in scs[c].synthesize_dev(phase, {i: F.arr([v])[0] for i, v in ch.items()}).items()}
    proof_ref, _ = M.create_proof_multi(ref, pkr, trep, [[], []], synth_ref, blinds)
    assert first_diff(proof, proof_ref) is None, f"first differing 32-byte proof item: {first_diff(proof, proof_ref)}"
    assert M.verify_proof_multi(ref, pkr, trep, [[], []], proof)


def test_multi_gpu_multi_circuit_proof_identical():
    """the multi-GPU session (every rank's units dealt over all circuits) writes the single-GPU bytes of a 3-circuit proof"""
    from test_gpu_multi import _ngpu, _torchrun
    if _ngpu() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _torchrun("multi_gpu_proof_multi.py", [8, 3], 2)
    assert r["identical_proof_on_all_ranks"]
