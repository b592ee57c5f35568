"""Host-side logic of bench.py that needs no GPU: the algorithmic-bytes accounting of a proof (SURVEY.md 8d row #3: the figures
DESIGN.md section 7 quotes), the isolated CPU-proof child process of the reference arm, and the oracle's explicit thread control."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_proof_accounting_of_the_k20_shape():
    import bench
    shape = {"k": 20, "advice_columns": 128, "lookup_arguments": 16, "permutation_columns": 49, "fixed_columns": 11, "instance_columns": 1, "cs_degree": 9}
    a = bench.proof_accounting(shape, None)
    n = 1 << 20
    assert a["msm_acc_chunk_kernel"]["alg_bytes"] == 178 * n * 96                      # 128 advice + 16 m + 7 z + 16 phi + 1 + 8 h + 2
    assert a["ntt_tile_kernel"]["alg_bytes"] == 64 * n * (167 + 168 * 8 + 8)            # iNTTs + coset NTTs + the extended iNTT (8 n)
    assert a["expr_kernel"]["alg_bytes"] == 8 * (232 * 32 * n + 32 * n)
    assert round(a["msm_acc_chunk_kernel"]["alg_bytes"] / 1e9, 1) == 17.9 and round(a["ntt_tile_kernel"]["alg_bytes"] / 1e9, 1) == 101.9


def test_cpu_proof_child_runs_in_its_own_process():
    env = dict(os.environ, OMP_NUM_THREADS="2", CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cpu-proof-child", "8", "1"], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    rec = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert rec["k"] == 8 and len(rec["times"]) == 1 and rec["times"][0] > 0 and rec["cores"] >= 1


def test_dump_outputs_and_steps_argument(tmp_path):
    import numpy as np
    import bench
    proofs = {"proof_device_witness": bytes(range(256)) * 3, "proof_host_witness": b"\x00\xff\x07"}
    bench.dump_outputs(str(tmp_path / "out"), proofs)
    for name, proof in proofs.items():
        a = np.load(tmp_path / "out" / f"{name}.npy")
        assert a.dtype == np.float64 and bytes(a.astype(np.uint8)) == proof
    assert bench.positive_int("3") == 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_oracle_thread_count_is_explicit():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_lib
    orc = oracle_lib.load()
    before = orc.num_threads()
    assert orc.set_num_threads(2) == 2        # what bench.py does under torchrun, where OMP_NUM_THREADS=1 is inherited
    assert orc.set_num_threads(before) == before
