"""python scripts/multi_circuit_bench.py [--k 17] [--circuits 1,2,4] [--warmup 1] [--steps 3]
C circuits of the Keccak-shaped stand-in (tests/standins.py: one proving key, C witnesses) proved two ways on one GPU: C separate
create_proof calls, and ONE create_proof_multi proof of all C.  Prints one JSON line per C with the median seconds of each, the
per-circuit ratio, and `verified` = the oracle verifier accepts the batched proof.  The card's name, power limit and SM clock are
read in the same run and printed with the numbers."""
import argparse, json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k", type=int, default=17)
    ap.add_argument("--circuits", default="1,2,4")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    import standins
    import halo2_ref as H
    import halo2_multi as M
    import pyref as P
    from test_gpu_prover_wide import to_oracle_cs
    from zkb200 import plonk as Z
    from zkb200.params import ParamsKZG

    class ValueOps(standins.DeviceOps):   # circuit c's witness: the same structure, random values from other seeds
        def __init__(self, off): super().__init__(); self.off = off
        def rand(self, n, seed): return super().rand(n, seed + self.off)
    k, s = args.k, 4321
    counts = [int(c) for c in args.circuits.split(",")]
    scs = [standins.keccak_shape(k, seed=3, ops=ValueOps(99991 * c)) for c in range(max(counts))]
    sc0, h = scs[0], scs[0].host
    params = ParamsKZG.unsafe_setup_with_s(k, s)
    pk = Z.ProvingKey(sc0.cs, [h(t) for t in sc0.fixed], [h(t) for t in sc0.sigma], srs=params.load())
    tr = h(sc0.transcript_repr[None])[0]

    def synth(c, phase, ch):
        return {j: h(t) for j, t in scs[c].synthesize_dev(phase, ch).items()}
    zb = [h(sc.z_blinds) for sc in scs]; pb = [h(sc.phi_blinds) for sc in scs]; rp = h(sc0.random_poly)

    def separate(C):
        return [Z.create_proof(pk, tr, [], lambda ph, ch, c=c: synth(c, ph, ch), zb[c], pb[c], rp) for c in range(C)]

    def batched(C):
        return Z.create_proof_multi(pk, tr, [[]] * C, synth, np.concatenate(zb[:C]), np.concatenate(pb[:C]), rp)

    def timed(fn, C):
        for _ in range(args.warmup): fn(C)
        ts, out = [], None
        for _ in range(args.steps):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            out = fn(C)
            torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
        return statistics.median(ts), ts, out
    # oracle verifier: vk commitments from the device, checked against the SRS trapdoor inside the verifier's final equation
    ref = H.Ref(to_oracle_cs(sc0.cs), s, build_srs=False)
    vk = pk.vk_bytes()
    pts = [P.g1_decompress(vk[8 + 32 * i: 40 + 32 * i]) for i in range((len(vk) - 8) // 32)]
    nf = sc0.cs.num_fixed
    pkr = {"fixed_commitments": pts[:nf], "sigma_commitments": pts[nf:]}
    info = gpu_info()
    for C in counts:
        t_sep, ts_sep, _ = timed(separate, C)
        t_bat, ts_bat, proof = timed(batched, C)
        ok = M.verify_ok(ref, pkr, ref.F.ints(tr[None])[0], [[]] * C, proof)
        print(json.dumps({"workload": f"keccak_shape k={k}", "circuits": C, "separate_seconds": t_sep, "batched_seconds": t_bat,
                          "separate_per_circuit": t_sep / C, "batched_per_circuit": t_bat / C, "batched_over_separate": t_bat / t_sep,
                          "separate_steps": ts_sep, "batched_steps": ts_bat, "proof_bytes": len(proof), "verified": bool(ok),
                          "warmup": args.warmup, "steps": args.steps, "gpu": info}), flush=True)


if __name__ == "__main__":
    main()
