"""ctypes binding of libzkb200.so (the C ABI declared in include/zkb200.h).

There is no CPU fallback: if the shared library is missing, or no sm_100 device is present, every compute entry
point raises ZkbError.  Build with `python -c "import __graft_entry__ as g; g.build()"` or `make -C zkevm-circuits_b200/csrc`.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libzkb200.so")

_u64p = ctypes.POINTER(ctypes.c_uint64)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_vp = ctypes.c_void_p


class ZkbError(RuntimeError):
    pass


# name -> (restype, argtypes); must list every symbol include/zkb200.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    "zkb_init": (ctypes.c_int32, [ctypes.c_int32, ctypes.POINTER(_vp)]),
    "zkb_destroy": (ctypes.c_int32, [_vp]),
    "zkb_last_error": (ctypes.c_char_p, []),
    "zkb_version": (ctypes.c_uint32, []),
    "zkb_launch_count": (ctypes.c_uint64, [_vp]),
    "zkb_sync": (ctypes.c_int32, [_vp]),
    "zkb_prof_enable": (ctypes.c_int32, [_vp, ctypes.c_int32]),
    "zkb_prof_read": (ctypes.c_int32, [_vp, ctypes.c_int32, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double), ctypes.c_int32]),
    "zkb_stream": (_vp, [_vp]),
    "zkb_malloc": (ctypes.c_int32, [_vp, ctypes.c_uint64, ctypes.POINTER(_vp)]),
    "zkb_free": (ctypes.c_int32, [_vp, _vp]),
    "zkb_h2d": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64]),
    "zkb_d2h": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64]),
    "zkb_ntt_fr_host": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_int32]),
    "zkb_ntt_fr_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_int32, _vp]),
    "zkb_ntt_fr_batch_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp, ctypes.c_int32, _vp]),
    "zkb_fr_root_of_unity": (ctypes.c_int32, [ctypes.c_uint32, _vp, _vp]),
    "zkb_msm_g1_host": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_msm_g1_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64, _vp, _vp, _vp, _vp]),
    "zkb_msm_g1_batch_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_msm_last_adds": (ctypes.c_uint64, [_vp]),
    "zkb_msm_last_levels": (ctypes.c_uint32, [_vp]),
    "zkb_srs_load": (ctypes.c_int32, [_vp, ctypes.c_uint32, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_srs_load_dev": (ctypes.c_int32, [_vp, ctypes.c_uint32, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_srs_destroy": (ctypes.c_int32, [_vp]),
    "zkb_srs_k": (ctypes.c_uint32, [_vp]),
    "zkb_srs_downsize": (ctypes.c_int32, [_vp, ctypes.c_uint32, ctypes.POINTER(_vp)]),
    "zkb_srs_read": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp]),
    "zkb_srs_commit_dev": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_srs_commit_host": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_srs_commit_batch_dev": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp, ctypes.c_uint32, ctypes.c_uint64, _vp, _vp]),
    "zkb_g1_fixed_base_mul_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_field_binop_dev": (ctypes.c_int32, [_vp, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _vp, ctypes.c_uint64, _vp]),
    "zkb_field_unop_dev": (ctypes.c_int32, [_vp, ctypes.c_int32, ctypes.c_int32, _vp, _vp, ctypes.c_uint64, _vp]),
    "zkb_fr_batch_invert_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64, _vp]),
    "zkb_fr_powers_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_poly_eval_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_fr_prefix_product_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_fr_prefix_sum_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_kate_division_dev": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_ntt_cross_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint64, _vp, _vp]),
    "zkb_g1_sum_affine_host": (ctypes.c_int32, [_vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_ntt_fr_sharded_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_int32, _vp]),
    "zkb_msm_g1_sharded_dev": (ctypes.c_int32, [_vp, _vp, _vp, ctypes.c_uint64, _vp, _vp, _vp]),
    "zkb_comm_unique_id": (ctypes.c_int32, [_vp]),
    "zkb_comm_init": (ctypes.c_int32, [_vp, _vp, ctypes.c_int32, ctypes.c_int32]),
    "zkb_comm_destroy": (ctypes.c_int32, [_vp]),
    "zkb_pk_create": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_pk_create_with_srs": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_keygen_pk": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, _vp, _vp, ctypes.c_uint64, _vp, ctypes.POINTER(_vp)]),
    "zkb_pk_sigma_read": (ctypes.c_int32, [_vp, ctypes.c_uint32, _vp]),
    "zkb_pk_destroy": (ctypes.c_int32, [_vp]),
    "zkb_pk_vk_bytes": (ctypes.c_int32, [_vp, _vp, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64)]),
    "zkb_csf_validate": (ctypes.c_int32, [_vp, ctypes.c_uint64]),
    "zkb_prove_begin": (ctypes.c_int32, [_vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_prove_begin_ex": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_prove_begin_cb": (ctypes.c_int32, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_prove_begin_multi": (ctypes.c_int32, [_vp, ctypes.c_int32, _vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.POINTER(_vp)]),
    "zkb_poseidon_hash_host": (ctypes.c_int32, [_vp, ctypes.c_uint64, _vp]),
    "zkb_blake2b_challenge_host": (ctypes.c_int32, [_vp, ctypes.c_uint64, _vp]),
    "zkb_keccak256_host": (ctypes.c_int32, [_vp, ctypes.c_uint64, _vp]),
    "zkb_transcript_script_host": (ctypes.c_int32, [ctypes.c_int32, _vp, ctypes.c_uint64, _vp, _vp, ctypes.c_uint64, _vp, _vp]),
    "zkb_prove_advice_phase": (ctypes.c_int32, [_vp, ctypes.c_uint32, _vp, _vp]),
    "zkb_prove_upload_advice": (ctypes.c_int32, [_vp, ctypes.c_uint32, _vp]),
    "zkb_prove_finish": (ctypes.c_int32, [_vp, _vp, _vp, _vp, _vp, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64)]),
    "zkb_session_destroy": (ctypes.c_int32, [_vp]),
}

_lib = None


def load_library():
    """Load libzkb200.so and attach signatures.  Raises ZkbError when the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ZkbError(f"{LIB_PATH} is missing: build the CUDA extension first (__graft_entry__.build()); "
                       "zkb200 has no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load_library().zkb_last_error()
        raise ZkbError(f"libzkb200 error {rc}: {msg.decode() if msg else ''}")


class Context:
    """One per GPU (per process rank).  Mirrors the process-global, mutex-guarded prover state the reference keeps
    (prover/src/test/inner.rs:20-30)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = _vp()
        check(self.lib.zkb_init(int(device), ctypes.byref(h)))
        self.handle = h
        self.device = int(device)

    def close(self):
        if self.handle:
            self.lib.zkb_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def init_comm(self, group=None):
        """Create this rank's NCCL communicator (multi-GPU create_proof): rank 0's unique id is broadcast with torch.distributed."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        buf = (ctypes.c_uint8 * 128)()
        if rank == 0:
            check(self.lib.zkb_comm_unique_id(ctypes.cast(buf, _vp)))
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        t = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
        dist.broadcast(t, src=0, group=group)
        raw = bytes(t.cpu().tolist())
        buf2 = (ctypes.c_uint8 * 128).from_buffer_copy(raw)
        check(self.lib.zkb_comm_init(self.handle, ctypes.cast(buf2, _vp), rank, world))
        return rank, world

    def prof_enable(self, on=True):
        check(self.lib.zkb_prof_enable(self.handle, 1 if on else 0))

    def prof_read(self, cls, reset=False):
        """-> (launches, total ms) of kernel class cls (0 ntt_tile, 1 msm_acc_chunk, 2 expr) since the last reset."""
        n, ms = ctypes.c_uint64(0), ctypes.c_double(0)
        check(self.lib.zkb_prof_read(self.handle, int(cls), ctypes.byref(n), ctypes.byref(ms), 1 if reset else 0))
        return int(n.value), float(ms.value)

    @property
    def launch_count(self):
        return int(self.lib.zkb_launch_count(self.handle))

    def sync(self):
        check(self.lib.zkb_sync(self.handle))


_default = {}


def default_context(device=None):
    import torch
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]
