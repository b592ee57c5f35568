"""torchrun --nproc-per-node N scripts/multi_gpu_proof_multi.py K C
One proof of C circuits of one proving key (plonk.create_proof_multi) on every rank with the multi-GPU session (columns, lookups and
permutation sets of all circuits dealt across the ranks, coset parts of the one quotient dealt) must emit exactly the single-GPU
proof; prints one JSON line on rank 0."""
import os, sys, json, hashlib
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, torch.distributed as dist


def run(k, count):
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    import zkb200
    from zkb200 import plonk as Z
    from multi_circuits import variants
    from test_oracle_prover_multi import setup
    from test_gpu_prover import to_product_cs
    tcs = variants("toy", k, count, seed=k)
    ref, pkr, *_ = setup(tcs)
    F = ref.F

    def synth(c, phase, ch):
        chi = {i: F.ints(v[None])[0] for i, v in ch.items()}
        return {j: F.arr(v) for j, v in tcs[c].advice_ints(phase, chi).items()}
    import numpy as np
    args = (F.arr([tcs[0].transcript_repr])[0], [[F.arr(c) for c in tc.instances] for tc in tcs], synth,
            np.concatenate([F.arr(b) for tc in tcs for b in tc.blinds_ints["z"]]), np.concatenate([F.arr(b) for tc in tcs for b in tc.blinds_ints["phi"]]),
            F.arr(tcs[0].blinds_ints["random_poly"]))
    zcs = to_product_cs(tcs[0].cs, ref.bf, ref.d)
    ctx1 = zkb200.Context(local)
    pk1 = Z.ProvingKey(zcs, pkr["fixed_values"], pkr["sigma_values"], ref.g, ref.g_lagrange, ctx=ctx1)
    proof1 = Z.create_proof_multi(pk1, *args)
    pk1.close()
    ctxn = zkb200.Context(local)
    ctxn.init_comm()
    pkn = Z.ProvingKey(zcs, pkr["fixed_values"], pkr["sigma_values"], ref.g, ref.g_lagrange, ctx=ctxn)
    proofn = Z.create_proof_multi(pkn, *args)
    same = torch.tensor([int(proofn == proof1)], device="cuda"); dist.all_reduce(same, op=dist.ReduceOp.MIN)
    pkn.close(); ctxn.close(); ctx1.close()
    if rank == 0:
        return {"k": k, "circuits": count, "world": dist.get_world_size(), "identical_proof_on_all_ranks": bool(same.item()),
                "proof_sha256": hashlib.sha256(proofn).hexdigest()[:16]}
    return None


def main():
    k, count = int(sys.argv[1]), int(sys.argv[2])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = run(k, count)
    if res is not None:
        print(json.dumps(res))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
