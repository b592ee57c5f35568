"""Host mirror of the prover-facing surface of halo2_proofs::plonk (names follow the crate: `Expression`,
`ConstraintSystem`, `ProvingKey`, `create_proof`) on top of the C ABI's proving session (`zkb_pk_*`, `zkb_prove_*`).

The reference reaches this surface at circuit-benchmarks/src/super_circuit.rs:109-132 (`keygen_pk`, `create_proof`).
Here a constraint system is described by plain Python objects (the Rust shim would serialise halo2's own
`ConstraintSystem` the same way, see INTEGRATION.md) and flattened into the CSF blob documented in include/zkb200.h.
Nothing in this module computes field arithmetic on the CPU; it only marshals buffers.
"""
import ctypes
import struct
import numpy as np

from .lib import check, default_context

_vp = ctypes.c_void_p
CONST, FIXED, ADVICE, INSTANCE, CHALLENGE, NEG, ADD, MUL, SCALED = range(9)
CSF_MAGIC = 0x3146535A


class Expression:
    """plonk::Expression<Fr> (selectors already compiled into fixed columns)."""
    __slots__ = ("op", "a", "b")

    def __init__(self, op, a=None, b=None):
        self.op, self.a, self.b = op, a, b

    @staticmethod
    def Constant(limbs):               # limbs: 4 x u64 Montgomery
        return Expression(CONST, tuple(int(x) for x in limbs))

    @staticmethod
    def Fixed(col, rot=0): return Expression(FIXED, col, rot)
    @staticmethod
    def Advice(col, rot=0): return Expression(ADVICE, col, rot)
    @staticmethod
    def Instance(col, rot=0): return Expression(INSTANCE, col, rot)
    @staticmethod
    def Challenge(i): return Expression(CHALLENGE, i)
    def __neg__(self): return Expression(NEG, self)
    def __add__(self, o): return Expression(ADD, self, o)
    def __mul__(self, o): return Expression(MUL, self, o)
    def scaled(self, limbs): return Expression(SCALED, self, tuple(int(x) for x in limbs))


class ConstraintSystem:
    """The fields of plonk::ConstraintSystem the prover reads."""

    def __init__(self, k, num_fixed, num_advice, num_instance, advice_phase, challenge_phase, blinding_factors, degree):
        self.k, self.n = k, 1 << k
        self.num_fixed, self.num_advice, self.num_instance = num_fixed, num_advice, num_instance
        self.advice_phase, self.challenge_phase = list(advice_phase), list(challenge_phase)
        self.blinding_factors, self.degree = blinding_factors, degree
        self.gates, self.lookups, self.perm_columns = [], [], []      # lookups: (list of input-expression lists, table list)
        self.advice_queries, self.fixed_queries, self.instance_queries = [], [], []

    def num_phases(self):
        return max(self.advice_phase + self.challenge_phase + [0]) + 1

    def to_csf(self):
        nodes, consts, memo, cmemo = [], [], {}, {}

        def cidx(limbs):
            if limbs not in cmemo:
                cmemo[limbs] = len(consts)
                consts.append(limbs)
            return cmemo[limbs]

        def visit(e):
            key = id(e)
            if key in memo: return memo[key]
            if e.op == CONST: nd = (CONST, cidx(e.a), 0)
            elif e.op in (FIXED, ADVICE, INSTANCE): nd = (e.op, e.a, e.b & 0xFFFFFFFF)
            elif e.op == CHALLENGE: nd = (CHALLENGE, e.a, 0)
            elif e.op == NEG: nd = (NEG, visit(e.a), 0)
            elif e.op in (ADD, MUL): nd = (e.op, visit(e.a), visit(e.b))
            elif e.op == SCALED: nd = (SCALED, visit(e.a), cidx(e.b))
            else: raise ValueError(e.op)
            nodes.append(nd)
            memo[key] = len(nodes) - 1
            return memo[key]
        gates = [visit(g) for g in self.gates]
        lks = []
        for inputs, table in self.lookups:
            lks.append(([[visit(e) for e in inp] for inp in inputs], [visit(e) for e in table]))
        w = [CSF_MAGIC, self.k, self.num_fixed, self.num_advice, self.num_instance, len(self.challenge_phase), self.blinding_factors, self.degree,
             self.num_phases(), len(nodes), len(consts), len(gates), len(lks), len(self.perm_columns), len(self.advice_queries),
             len(self.fixed_queries), len(self.instance_queries), 0]
        w += self.advice_phase + self.challenge_phase
        for nd in nodes: w += list(nd)
        for c in consts:
            for limb in c: w += [limb & 0xFFFFFFFF, limb >> 32]
        w += gates
        for inputs, table in lks:
            w += [len(inputs), len(table)]
            for inp in inputs: w += inp
            w += table
        for (t, i) in self.perm_columns: w += [t, i]
        for q in (self.advice_queries, self.fixed_queries, self.instance_queries):
            for (c, r) in q: w += [c, r & 0xFFFFFFFF]
        return np.array(w, dtype=np.uint32)


def validate_csf(blob):
    """host-only structural check of a CSF blob (raises ZkbError)."""
    from .lib import load_library
    b = np.ascontiguousarray(blob, dtype=np.uint32)
    check(load_library().zkb_csf_validate(_vp(b.ctypes.data), b.size))


def _ptr_array(arrs):
    """host numpy arrays, device buffers (objects with a `device_ptr` attribute) or None -> (keepalive list, void** as c_void_p array)."""
    keep, ptrs = [], []
    for a in arrs:
        if a is None:
            keep.append(None); ptrs.append(None)
        elif hasattr(a, "device_ptr"):
            keep.append(a); ptrs.append(int(a.device_ptr))
        else:
            c = np.ascontiguousarray(a)
            keep.append(c); ptrs.append(c.ctypes.data)
    tbl = (ctypes.c_void_p * max(1, len(keep)))(*ptrs)
    return keep, tbl


class DeviceColumn:
    """a witness column that already lives in HBM (torch tensor or raw pointer): zkb_prove_advice_phase copies it device-to-device"""
    def __init__(self, tensor):
        self.tensor = tensor
        self.device_ptr = tensor.data_ptr()
        self.shape = tuple(tensor.shape)
        self.dtype = np.dtype(np.uint64)


class ProvingKey:
    """plonk::ProvingKey<G1Affine> material resident on the GPU (keygen itself stays with the caller: SURVEY 8f row 3)."""

    def __init__(self, cs, fixed_values, sigma_values, g=None, g_lagrange=None, ctx=None, srs=None, copies=None):
        """Either (g, g_lagrange) host arrays [legacy: the pk uploads its own SRS] or srs = params.Srs handle (shared).
        copies != None: keygen path (zkb_keygen_pk) -- sigma_values is ignored and the permutation is assembled from the copy
        constraints [(left perm column, left row, right perm column, right row), ...]."""
        self.ctx = ctx or (srs.ctx if srs is not None else default_context())
        self.cs = cs
        self.srs = srs
        n = cs.n
        blob = cs.to_csf()
        kf, ftbl = _ptr_array(fixed_values)
        h = _vp()
        if copies is not None:
            assert srs is not None
            cp = np.ascontiguousarray(np.asarray(copies, dtype=np.uint32).reshape(-1, 4))
            check(self.ctx.lib.zkb_keygen_pk(self.ctx.handle, _vp(blob.ctypes.data), blob.size, ctypes.cast(ftbl, _vp), _vp(cp.ctypes.data), cp.shape[0],
                                             srs.handle, ctypes.byref(h)))
        elif srs is not None:
            ks, stbl = _ptr_array(sigma_values)
            check(self.ctx.lib.zkb_pk_create_with_srs(self.ctx.handle, _vp(blob.ctypes.data), blob.size, ctypes.cast(ftbl, _vp), ctypes.cast(stbl, _vp),
                                                      srs.handle, ctypes.byref(h)))
        else:
            assert g.shape == (n, 8) and g_lagrange.shape == (n, 8)
            ks, stbl = _ptr_array(sigma_values)
            g = np.ascontiguousarray(g); gl = np.ascontiguousarray(g_lagrange)
            check(self.ctx.lib.zkb_pk_create(self.ctx.handle, _vp(blob.ctypes.data), blob.size, ctypes.cast(ftbl, _vp), ctypes.cast(stbl, _vp),
                                             _vp(g.ctypes.data), _vp(gl.ctypes.data), ctypes.byref(h)))
        self.handle = h

    def sigma_values(self, column):
        out = np.empty((self.cs.n, 4), dtype=np.uint64)
        check(self.ctx.lib.zkb_pk_sigma_read(self.handle, int(column), _vp(out.ctypes.data)))
        return out

    def vk_bytes(self):
        """VerifyingKey::to_bytes(SerdeFormat::Processed): fixed + permutation commitments computed on the GPU."""
        n = ctypes.c_uint64(0)
        check(self.ctx.lib.zkb_pk_vk_bytes(self.handle, None, 0, ctypes.byref(n)))
        out = (ctypes.c_uint8 * n.value)()
        check(self.ctx.lib.zkb_pk_vk_bytes(self.handle, ctypes.cast(out, _vp), n.value, ctypes.byref(n)))
        return bytes(out)

    def close(self):
        if self.handle:
            self.ctx.lib.zkb_pk_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try: self.close()
        except Exception: pass


TRANSCRIPTS = {"blake2b": 0, "poseidon": 1, "evm": 2}

_CB_SCALAR = ctypes.CFUNCTYPE(ctypes.c_int32, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64))


class _TranscriptVtable(ctypes.Structure):
    _fields_ = [("user", ctypes.c_void_p), ("common_scalar", _CB_SCALAR), ("write_scalar", _CB_SCALAR), ("write_point", _CB_SCALAR),
                ("squeeze_challenge", _CB_SCALAR)]


class CallbackTranscript:
    """zkb_transcript_vtable around a caller-side transcript object (the stand-in for create_proof's generic `T: TranscriptWrite`, which
    the Rust shim forwards the same way).  `obj` implements common_scalar(limbs), write_scalar(limbs), write_point(limbs8) and
    squeeze_challenge() -> 4 Montgomery limbs; limbs are numpy uint64 arrays in halo2curves' in-memory layout."""

    def __init__(self, obj):
        self.obj = obj
        self.error = None

        def wrap(fn, n_in):
            def cb(_user, ptr):
                try:
                    fn(np.ctypeslib.as_array(ptr, shape=(n_in,)).copy())
                    return 0
                except Exception as e:   # never let a Python exception unwind through C
                    self.error = e
                    return 1
            return _CB_SCALAR(cb)

        def squeeze(_user, ptr):
            try:
                out = np.ascontiguousarray(obj.squeeze_challenge(), dtype=np.uint64)
                for i in range(4): ptr[i] = int(out[i])
                return 0
            except Exception as e:
                self.error = e
                return 1
        self._keep = (wrap(obj.common_scalar, 4), wrap(obj.write_scalar, 4), wrap(obj.write_point, 8), _CB_SCALAR(squeeze))
        self.vt = _TranscriptVtable(None, *self._keep)


def create_proof(pk, transcript_repr, instances, synthesize, z_blinds, phi_blinds, random_poly, transcript="blake2b", upload_ahead=False):
    """Mirror of plonk::create_proof for one circuit; transcript = "blake2b" (Blake2bWrite, the reference's benches) or "poseidon"
    (snark-verifier-sdk's PoseidonTranscript, what gen_snark_shplonk uses) or "evm" (snark-verifier's EvmTranscript over Keccak-256,
    what gen_evm_proof_shplonk uses; proof items uncompressed big-endian) or a CallbackTranscript around the caller's own transcript
    object (create_proof's generic `T`): then the returned bytes are empty and the proof is whatever that object wrote.

    transcript_repr: uint64[4] (Montgomery Fr).   instances: list of uint64 (len, 4) arrays (one per instance column).
    synthesize(phase, challenges) -> dict {advice column: uint64 (n,4) array, already blinded} for that phase's columns,
      where challenges is a dict {index: uint64[4]} of the challenges available so far (Circuit::synthesize stand-in).
    z_blinds (n_sets*bf, 4), phi_blinds (n_lookups*bf, 4), random_poly (n, 4): uint64 Montgomery arrays.
    Returns the proof bytes."""
    lib = pk.ctx.lib
    tr = np.ascontiguousarray(np.asarray(transcript_repr, dtype=np.uint64).reshape(4))
    ki, itbl = _ptr_array(instances)
    lens = (ctypes.c_uint32 * max(1, len(instances)))(*[a.shape[0] for a in instances])
    sess = _vp()
    if isinstance(transcript, CallbackTranscript):   # the caller's own transcript object: proof bytes are written on its side
        check(lib.zkb_prove_begin_cb(pk.handle, ctypes.cast(ctypes.pointer(transcript.vt), _vp), _vp(tr.ctypes.data), ctypes.cast(itbl, _vp),
                                     ctypes.cast(lens, _vp), ctypes.byref(sess)))
    else:
        check(lib.zkb_prove_begin_ex(pk.handle, TRANSCRIPTS[transcript], _vp(tr.ctypes.data), ctypes.cast(itbl, _vp), ctypes.cast(lens, _vp), ctypes.byref(sess)))
    return _prove(pk, sess, 1, lambda c, phase, ch: synthesize(phase, ch), z_blinds, phi_blinds, random_poly, upload_ahead)


def create_proof_multi(pk, transcript_repr, instances, synthesize, z_blinds, phi_blinds, random_poly, transcript="blake2b", upload_ahead=False):
    """Mirror of plonk::create_proof with several circuits (`circuits: &[C]`, `instances: &[&[&[Fr]]]`): ONE proof of C circuits of
    the same constraint system.  They share the challenges, one quotient and one SHPLONK opening (zkb_prove_begin_multi).

    instances: one list per circuit of uint64 (len, 4) arrays (one per instance column).
    synthesize(circuit, phase, challenges) -> dict {advice column: uint64 (n,4) array, already blinded} for circuit `circuit`.
    z_blinds (C*n_sets*bf, 4) and phi_blinds (C*n_lookups*bf, 4): circuit-major; random_poly (n, 4): one for the proof.
    transcript and upload_ahead as in create_proof.  Returns the proof bytes (empty with a CallbackTranscript)."""
    cs, lib = pk.cs, pk.ctx.lib
    nc = len(instances)
    for inst in instances:
        assert len(inst) == cs.num_instance, "every circuit passes one array per instance column"
    tr = np.ascontiguousarray(np.asarray(transcript_repr, dtype=np.uint64).reshape(4))
    flat = [a for inst in instances for a in inst]
    ki, itbl = _ptr_array(flat)
    lens = (ctypes.c_uint32 * max(1, len(flat)))(*[a.shape[0] for a in flat])
    cb = isinstance(transcript, CallbackTranscript)
    vt = ctypes.cast(ctypes.pointer(transcript.vt), _vp) if cb else None
    sess = _vp()
    check(lib.zkb_prove_begin_multi(pk.handle, 3 if cb else TRANSCRIPTS[transcript], vt, _vp(tr.ctypes.data), nc, ctypes.cast(itbl, _vp),
                                    ctypes.cast(lens, _vp), ctypes.byref(sess)))
    return _prove(pk, sess, nc, synthesize, z_blinds, phi_blinds, random_poly, upload_ahead)


def _prove(pk, sess, nc, synthesize, z_blinds, phi_blinds, random_poly, upload_ahead):
    """the advice phases and zkb_prove_finish of a begun session of nc circuits; destroys the session"""
    cs, lib = pk.cs, pk.ctx.lib
    na = cs.num_advice
    try:
        nch = len(cs.challenge_phase)
        ch_buf = np.zeros((max(1, nch), 4), dtype=np.uint64)
        challenges = {}
        for phase in range(cs.num_phases()):
            arrs = []      # circuit-major: circuit c's column j at c * na + j
            for circ in range(nc):
                cols = synthesize(circ, phase, dict(challenges))
                arrs += [cols.get(c) if cs.advice_phase[c] == phase else None for c in range(na)]
            for i, a in enumerate(arrs):
                if cs.advice_phase[i % na] == phase:
                    assert a is not None and a.shape == (cs.n, 4) and a.dtype == np.uint64
            if upload_ahead:   # column by column ahead of the phase call (zkb_prove_upload_advice), then NULL pointers in the phase call
                idx = [c for c, a in enumerate(arrs) if a is not None]
                keep_up, utbl = _ptr_array([arrs[c] for c in idx])      # keep_up holds the (contiguous) buffers alive until the phase call returns
                for t, c in enumerate(idx):
                    check(lib.zkb_prove_upload_advice(sess, c, _vp(utbl[t])))
                arrs = [None] * len(arrs)
            ka, atbl = _ptr_array(arrs)
            check(lib.zkb_prove_advice_phase(sess, phase, ctypes.cast(atbl, _vp), _vp(ch_buf.ctypes.data)))
            for i, ph in enumerate(cs.challenge_phase):
                if ph == phase: challenges[i] = ch_buf[i].copy()
        zb = np.ascontiguousarray(z_blinds) if z_blinds is not None and len(z_blinds) else None
        pb = np.ascontiguousarray(phi_blinds) if phi_blinds is not None and len(phi_blinds) else None
        rp = np.ascontiguousarray(random_poly)
        plen = ctypes.c_uint64(0)
        # first call runs the proof and reports its length (bytes stay in the session); second call copies them out
        check(lib.zkb_prove_finish(sess, _vp(zb.ctypes.data) if zb is not None else None, _vp(pb.ctypes.data) if pb is not None else None,
                                   _vp(rp.ctypes.data), None, 0, ctypes.byref(plen)))
        out = (ctypes.c_uint8 * max(1, plen.value))()
        check(lib.zkb_prove_finish(sess, None, None, None, ctypes.cast(out, _vp), plen.value, ctypes.byref(plen)))
        return bytes(out[: plen.value])
    finally:
        lib.zkb_session_destroy(sess)
