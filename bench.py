#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 Halo2/KZG proving path.

BASELINE.json's metric has three terms: "SuperCircuit k=20 proof-gen sec + MSM G1-adds/s + NTT Fr-butterflies/s @1/2/4/8 B200".
The JSON line's `metric`/`value` is the FIRST term: wall-clock seconds of one create_proof (halo2 KZG + SHPLONK, Blake2b transcript)
of the SuperCircuit-shaped k = 20 stand-in (tests/standins.py: 3 phases, 128 advice columns, 640 condition*constraint gates, 16
lookup arguments = 48 input sets, 49 permutation columns incl. the instance column; the real circuit cannot be synthesised without
Rust, SURVEY.md 8d #4).  A "step" is one proof.  The other two terms are carried in `extras` with their own roofline / e2e /
cpu_baseline objects: `ntt_2^24_round_trip` (configs[1]) and `msm_2^20` (configs[0]); `proof_keccak_shape_k17` is configs[2].

  value   proof seconds with the witness columns already resident in HBM (device pointers through the same C-ABI session)
  e2e     the same with HOST (pinned) witness buffers: every advice column is copied H2D inside the timed region, the proof bytes
          come back D2H -- this is what a Rust caller gets
  N > 1   ONE proof spread over the N ranks (strong scaling): commitment batches, lookup arguments and the quotient's coset parts
          are dealt across the GPUs and exchanged over NCCL; extras carry the domain-sharded NTT (fused peer-memory exchange vs the
          NCCL baseline), the point-range sharded 2^26 MSM (configs[4]) and the cross-rank parity flags.  A mismatch fails the run.
  --impl reference   the CPU restatement of halo2's create_proof (oracle/halo2_ref.py over oracle/libzkoracle.so, OpenMP on all host
          cores; the Rust crate cannot be built here) on a BOUNDED sample of the same shape (smaller k), scaled linearly in the rows.

Every proof timed here is checked AFTER the timed region by the pinned oracle verifier (`verified`), never inside it.

  --dump-outputs DIR   after the timed steps, the proof bytes of the last timed step of each witness placement as
          DIR/proof_device_witness.npy and DIR/proof_host_witness.npy (float64, one element per byte; inputs are seeded, so two
          builds given the same arguments can be compared output for output)
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K_PROOF = 20
ADVICE = 128
METRIC = "SuperCircuit-shaped k=20 create_proof seconds (halo2 KZG/SHPLONK, Blake2b transcript)"
UNIT = "s"
LOG_N = 24
N_PTS = 1 << LOG_N
BUTTERFLIES_PER_DIR = (N_PTS // 2) * LOG_N          # 201,326,592  (SURVEY.md 8d)
ALG_BYTES_PER_DIR = 2 * 32 * N_PTS                  # 1,073,741,824 B: read + write each element once per transform
MSM_LOG_N = 20
SRS_S = 1234                                        # zkevm-circuits/src/super_circuit/test.rs:74 uses the same toy trapdoor


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def config_dict(world):
    return {"workload": f"create_proof of the SuperCircuit-shaped stand-in at k={K_PROOF}, {ADVICE} advice columns (BASELINE configs[3]); "
                        "N>1: the same single proof spread over N GPUs",
            "k": K_PROOF, "advice_columns": ADVICE, "transcript": "blake2b",
            "l2": "working set (GBs of columns per stage) >> 126 MB L2: no flush needed", "n_gpus": world}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe in B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu"

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                if float(f[8]) < 50:       # keep only samples taken under load (GPU utilisation >= 50 %)
                    continue
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------- CPU side (oracle)
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def load_oracle(threads=None):
    """the CPU oracle with an EXPLICIT OpenMP thread count (torchrun exports OMP_NUM_THREADS=1 to its workers), so that the CPU arm does
    not depend on the launcher"""
    threads = threads or min(host_threads(), CPU_THREADS_CAP)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_lib
    orc = oracle_lib.load()
    orc.set_num_threads(threads)     # the OpenMP runtime may already have been initialised with the launcher's value
    return orc


def oracle_proof_seconds(k, advice, reps=1):
    """seconds of the oracle's restated create_proof on the same shape at degree k (CPU witness, CPU SRS: nothing of the product runs)"""
    import numpy as np
    import halo2_ref as H
    import standins
    from test_gpu_prover_wide import to_oracle_cs
    sc = standins.super_shape(k, advice=advice, seed=5, ops=standins.OracleOps())
    cs = to_oracle_cs(sc.cs)
    ref = H.Ref(cs, SRS_S)
    F, h, n, bf = ref.F, sc.host, sc.n, sc.bf
    fixed = [h(t) for t in sc.fixed]
    sigma = [h(t) for t in sc.sigma]
    pkr = {"fixed_values": fixed, "fixed_polys": [ref.lagrange_to_coeff(v) for v in fixed], "sigma_values": sigma,
           "sigma_polys": [ref.lagrange_to_coeff(v) for v in sigma]}
    l0 = np.zeros((n, 4), dtype=np.uint64); l0[0] = ref.w_arr(1)
    lb = np.zeros((n, 4), dtype=np.uint64); lb[n - bf:] = ref.w_arr(1)
    ll = np.zeros((n, 4), dtype=np.uint64); ll[n - bf - 1] = ref.w_arr(1)
    pkr["l0"], pkr["l_last"], pkr["l_blind"] = [ref.lagrange_to_coeff(v) for v in (l0, ll, lb)]
    zb, pb = h(sc.z_blinds), h(sc.phi_blinds)
    blinds = {"z": [F.ints(zb[i * bf:(i + 1) * bf]) for i in range(sc.nsets)], "phi": [F.ints(pb[i * bf:(i + 1) * bf]) for i in range(sc.L)],
              "random_poly": h(sc.random_poly)}
    trep = F.ints(h(sc.transcript_repr[None]))[0]
    inst = [F.ints(h(t)) for t in sc.instances]
    cols = {}

    def synth(phase, ch):
        chm = {i: F.arr([v])[0] for i, v in ch.items()}
        return {c: h(t) for c, t in sc.synthesize_dev(phase, chm).items()}
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        proof, _ = ref.create_proof(pkr, trep, inst, synth, blinds)
        times.append(time.perf_counter() - t0)
    return times, sc.shape


def cpu_primitive_model(shape):
    """Lower bound of a CPU create_proof from MEASURED oracle primitives (all host threads): one best_multiexp and one best_fft of the
    circuit's size, multiplied by the number of commitments / transforms halo2's create_proof performs for this shape (SURVEY 8a).
    Quotient evaluation, scans, lookups' hash maps and witness generation are NOT included."""
    import numpy as np
    orc = load_oracle()
    k, A, L, P = shape["k"], shape["advice_columns"], shape["lookup_arguments"], shape["permutation_columns"]
    nf, ni, d = shape["fixed_columns"], shape["instance_columns"], shape["cs_degree"]
    n = 1 << k
    nsets = (P + (d - 2) - 1) // (d - 2)
    rng = np.random.default_rng(5)

    def rand_fr(m):
        a = rng.integers(0, 1 << 64, size=(m, 4), dtype=np.uint64)
        a[:, 3] = rng.integers(0, 0x30644E72E131A029, size=m, dtype=np.uint64)
        return a
    small = orc.g1_fixed_base_mul(orc.g1_generator(), rand_fr(1 << 12))
    bases = np.tile(small, (n >> 12, 1)) if n >= (1 << 12) else small[:n]
    s = rand_fr(n)
    orc.best_multiexp(s[:1 << 10], bases[:1 << 10])

    def best_of(fn, reps=3):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        return min(ts)
    t_msm = best_of(lambda: orc.best_multiexp(s, bases), 2)
    w = orc.fr_omega(k)
    a = rand_fr(n)
    t_fft = best_of(lambda: orc.best_fft(a, w, k))
    ek = k + 3
    t_ext = t_fft * ((1 << ek) * ek) / (n * k)
    commits = A + 2 * L + nsets + 1 + (d - 1) + 2
    iffts = A + 2 * L + nsets + ni
    ext_ffts = A + nf + ni + P + nsets + 2 * L + 4 + 1
    return {"seconds_lower_bound": commits * t_msm + iffts * t_fft + ext_ffts * t_ext, "msm_seconds": t_msm, "fft_seconds": t_fft,
            "extended_fft_seconds_scaled": t_ext, "commitments": commits, "iffts": iffts, "extended_ffts": ext_ffts, "cores": orc.num_threads(),
            "note": "measured oracle MSM / FFT x halo2's operation counts; excludes quotient evaluation, scans, lookups and witness generation"}


CPU_THREADS_CAP = 32     # every CPU leg: the GPU boxes report 128 hardware threads but share them with the other jobs of the pod; with
                         # 64-128 OpenMP threads the same oracle call varied 5-25x between boxes (r01 VERDICT), with 32 it is stable
PROOF_CPU_THREADS = 32   # the oracle prover's small-array stages get SLOWER with more threads (fork/join + spinning on boxes whose
                         # cgroup grants fewer CPUs than sched_getaffinity reports: 25 s at 64 threads, 380-660 s at 128 on this pool)


def _cpu_proof_child(k, steps):
    """runs in a fresh interpreter (no CUDA context, no inherited OpenMP pool): prints one JSON line"""
    orc = load_oracle(min(host_threads(), PROOF_CPU_THREADS))
    times, shape = oracle_proof_seconds(k, ADVICE, reps=steps)
    print(json.dumps({"k": k, "times": times, "cores": orc.num_threads()}), flush=True)


def cpu_proof_sample(budget_s, steps):
    """oracle create_proof on a bounded sample of the same shape, in a SUBPROCESS with a hard timeout: calibrate on k = 11, then the
    largest k <= 15 whose `steps` proofs fit the budget; -> (k_sample, [seconds per proof], threads)"""
    env = dict(os.environ, OMP_NUM_THREADS=str(min(host_threads(), PROOF_CPU_THREADS)), OMP_WAIT_POLICY="passive", CUDA_VISIBLE_DEVICES="")

    def child(k, reps, timeout):
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-proof-child", str(k), str(reps)], env=env, capture_output=True, text=True,
                             timeout=timeout)
        lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
        if not lines:
            raise RuntimeError("cpu proof child failed: " + out.stderr[-400:])
        return json.loads(lines[-1])
    r = child(11, 1, max(60.0, 4 * budget_s))
    t11 = r["times"][0]
    k_s = 11
    while k_s < 15 and t11 * (1 << (k_s + 1 - 11)) * steps <= budget_s:
        k_s += 1
    if k_s > 11:
        try:
            r = child(k_s, steps, max(120.0, 3 * budget_s))
        except subprocess.TimeoutExpired:
            k_s = 11
    return k_s, r["times"], r["cores"]


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    k_s, times, cores = cpu_proof_sample(150.0, steps)
    scale = 1 << (K_PROOF - k_s)
    sec = sorted(times)[len(times) // 2] * scale
    cfg = config_dict(args.gpus)
    cfg["reference_steps_cap"] = f"{len(times)} timed oracle proofs (cap 3; no warm-up needed on the CPU), asked for --steps {args.steps} --warmup {args.warmup}"
    line = {"impl": "reference", "metric": METRIC, "value": sec, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "warmup": 0,
            "ms_per_step": sec * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u256 (4x u64 Montgomery limbs, BN254 Fr/Fq)", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": sec, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"oracle create_proof (restated halo2 prover, OpenMP field/NTT/MSM kernels) of the same shape at k={k_s}: "
                                       f"median {sorted(times)[len(times) // 2]:.2f} s, scaled x{scale} (linear in rows; the n log n parts make this an underestimate)"},
            "e2e": {"value": sec, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    try:   # context: what the C/OpenMP primitives alone would cost at the full size (the Python-orchestrated prover above is far slower)
        shape = {"k": K_PROOF, "advice_columns": ADVICE, "lookup_arguments": 16, "permutation_columns": 49, "fixed_columns": 11, "instance_columns": 1, "cs_degree": 9}
        line["cpu_baseline"]["primitive_model"] = cpu_primitive_model(shape)
    except Exception as e:
        line["cpu_baseline"]["primitive_model_error"] = repr(e)
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- GPU side
class Pinned:
    """device tensor -> numpy view of a PINNED host copy (what a shim-allocated advice column would be)"""
    def __init__(self):
        self.keep = []

    def __call__(self, t):
        import numpy as np
        import torch
        p = torch.empty(t.shape, dtype=t.dtype).pin_memory()
        p.copy_(t)
        self.keep.append(p)
        return p.numpy().view(np.uint64)


def proof_accounting(shape, launches_by_class):
    """algorithmic bytes of one proof per kernel class (SURVEY.md 8d row #3): MSM = sum over commitments of n*96; NTT = 64 B per
    element per transform (read + write once); quotient interpreter = every referenced column once per coset part + the output."""
    k, A, L, P = shape["k"], shape["advice_columns"], shape["lookup_arguments"], shape["permutation_columns"]
    nf, ni, d = shape["fixed_columns"], shape["instance_columns"], shape["cs_degree"]
    n = 1 << k
    E = 8 if d == 9 else 4
    nsets = (P + (d - 2) - 1) // (d - 2)
    commitments = A + L + nsets + L + 1 + (d - 1) + 2
    intt = A + L + nsets + L
    coset_cols = A + ni + nsets + 2 * L                      # fixed / sigma / l_i / X come from the pk's coset cache
    ntt_bytes = 64 * n * intt + 64 * n * coset_cols * E + 64 * n * E
    quot_cols = nf + A + ni + P + nsets + 2 * L + 4
    expr_bytes = E * (quot_cols * 32 * n + 32 * n)
    return {"msm_acc_chunk_kernel": {"alg_bytes": commitments * n * 96, "units": f"{commitments} commitments x 2^{k} x 96 B"},
            "ntt_tile_kernel": {"alg_bytes": ntt_bytes, "units": f"{intt} iNTT(2^{k}) + {coset_cols}x{E} coset NTT(2^{k}) + 1 iNTT(2^{k + 3})"},
            "expr_kernel": {"alg_bytes": expr_bytes, "units": f"{E} coset parts x ({quot_cols} columns read once + 1 written) x 2^{k} x 32 B (lookup / permutation "
                                                              "value-domain programs not counted)"}}


def verify_with_oracle(sc, vk_bytes, proof, inst_host, fixed_host, sigma_host):
    """the checker leg: oracle verifier on a proof the GPU produced (outside every timed region).  vk_bytes = pk.vk_bytes(), fetched
    by the caller on EVERY rank (with a communicator that call is a collective)"""
    load_oracle()
    from test_gpu_standins import verify_gpu_proof
    ok, rejected, checked = verify_gpu_proof(sc, vk_bytes, proof, inst_host, SRS_S, fixed_host, sigma_host)
    return {"verified": bool(ok), "tampered_rejected": bool(rejected), "vk_commitments_checked_by_trapdoor": checked,
            "verifier": "oracle/halo2_ref.py verify_proof (pinned by the reference's own k=25 proof, tests/test_fixture_proof.py)"}


def build_case(kind, k, advice, pin):
    import torch
    import standins
    from zkb200 import plonk as Z
    from zkb200.params import ParamsKZG
    t0 = time.perf_counter()
    sc = standins.super_shape(k, advice=advice, seed=5) if kind == "super" else standins.keccak_shape(k, seed=3)
    params = ParamsKZG.unsafe_setup_with_s(k, SRS_S)
    srs = params.load()
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    fixed = [pin(t) for t in sc.fixed]
    sigma = [pin(t) for t in sc.sigma]
    t0 = time.perf_counter()
    pk = Z.ProvingKey(sc.cs, fixed, sigma, srs=srs)
    t_pk = time.perf_counter() - t0
    return sc, pk, fixed, sigma, {"setup_seconds": t_setup, "pk_build_seconds": t_pk}


def make_provers(sc, pk, pin):
    """-> (prove_host, prove_dev, inst_host): create_proof closures with pinned-host / device-resident witness columns"""
    import numpy as np
    import torch
    from zkb200 import plonk as Z
    cols0_dev = sc.synthesize_dev(0, {})
    cols0_host = {c: pin(t) for c, t in cols0_dev.items()}
    cols0_devcols = {c: Z.DeviceColumn(t) for c, t in cols0_dev.items()}
    later = {}    # pinned staging of the challenge-dependent columns (allocated once; Rust would own such buffers)
    zb, pb, rp, tr = pin(sc.z_blinds), pin(sc.phi_blinds), pin(sc.random_poly), pin(sc.transcript_repr[None])[0]
    inst = [pin(t) for t in sc.instances]

    def prove(host):
        def synth(phase, ch):
            if phase == 0:
                return cols0_host if host else cols0_devcols
            cols = sc.synthesize_dev(phase, ch)          # later phases depend on the challenge: produced inside the step, like Rust would
            if not host:
                return {c: Z.DeviceColumn(t) for c, t in cols.items()}
            out = {}
            for c, t in cols.items():
                if c not in later:
                    later[c] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
                later[c].copy_(t)
                out[c] = later[c].numpy().view(np.uint64)
            return out
        return Z.create_proof(pk, tr, inst, synth, zb, pb, rp)
    return (lambda: prove(True)), (lambda: prove(False)), inst


def dump_outputs(out_dir, proofs):
    """--dump-outputs: each proof as <out_dir>/<name>.npy, one float64 per byte (exact)"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, proof in proofs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float64))


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def time_steps(fn, warmup, steps, barrier):
    for _ in range(warmup):
        fn()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fn()
    barrier()
    return (time.perf_counter() - t0) / steps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's proofs as DIR/<name>.npy")
    ap.add_argument("--cpu-proof-child", nargs=2, type=int, default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_proof_child:
        return _cpu_proof_child(*args.cpu_proof_child)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the proofs of the GPU path (--impl ours)")
        return run_reference(args)

    import numpy as np
    import torch
    rank, local_rank, world = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import zkb200
    from zkb200 import arithmetic as A
    ctx = zkb200.default_context(local_rank)
    if world > 1:
        ctx.init_comm()
    W = max(3, args.warmup)
    K = args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    pin = Pinned()
    extras = {}
    failures = []
    # ------------------------------------------------------------------ headline: k = 20 proof
    sc, pk, fixed_h, sigma_h, setup = build_case("super", K_PROOF, ADVICE, pin)
    prove_host, prove_dev, inst_h = make_provers(sc, pk, pin)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx.prof_enable(False)
    sec_dev, proof_dev = time_steps(prove_dev, W, K, barrier)
    sec_dev = max_over_ranks(sec_dev)
    launches0 = ctx.launch_count
    sec_e2e, proof = time_steps(prove_host, 1, K, barrier)
    sec_e2e = max_over_ranks(sec_e2e)
    launches = (ctx.launch_count - launches0) // K
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"proof_device_witness": proof_dev, "proof_host_witness": proof})
    # per-kernel-class device time of ONE more proof (event pairs on the launching stream; outside the timed region because the
    # extra event records would perturb it)
    ctx.prof_enable(True)
    ctx.prof_read(0, reset=True)
    t0 = time.perf_counter(); prove_dev(); torch.cuda.synchronize(); sec_prof = time.perf_counter() - t0
    names = ["ntt_tile_kernel", "msm_acc_chunk_kernel", "expr_kernel"]
    prof = {nm: ctx.prof_read(i) for i, nm in enumerate(names)}
    ctx.prof_enable(False)
    acct = proof_accounting(sc.shape, prof)
    sc_shape_degree = sc.shape["cs_degree"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs_sustained", peaks.get("hbm_gbs", 6650.0)))
    kernels = {}
    for nm in names:
        cnt, ms = prof[nm]
        if cnt == 0:
            continue
        per_launch_bytes = acct[nm]["alg_bytes"] / cnt
        kernels[nm] = {"launches_per_proof": cnt, "ms_per_proof": ms, "share_of_proof": ms * 1e-3 / sec_prof, "avg_launch_ms": ms / cnt,
                       "alg_bytes_per_proof": acct[nm]["alg_bytes"], "alg_units": acct[nm]["units"],
                       "achieved_gbs": per_launch_bytes / (ms / cnt * 1e-3) / 1e9}
    dom = max(kernels, key=lambda nm: kernels[nm]["ms_per_proof"])
    # dram bytes per launch of the dominant kernel from the committed ncu --set full capture of this command (profiles/), if present
    traffic, traffic_note = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_proof_k20_traffic.json")))
        per = tj.get(dom, {}).get("dram_bytes_per_launch")
        if per and dom == "expr_kernel":
            # the ncu capture is one QUOTIENT launch (one coset part); the class also holds the small value-domain programs (lookup
            # compression, permutation / grand-sum terms), so express it per average launch of the class like `achieved`
            parts = 8 if sc_shape_degree == 9 else 4
            traffic = parts * per / kernels[dom]["launches_per_proof"]
            traffic_note = (f"{parts} quotient launches x {per / 1e9:.1f} GB (ncu --set full, profiles/r02_expr_kernel_k20_ncu.txt) / "
                            f"{kernels[dom]['launches_per_proof']} launches of the class; algorithmic = {acct[dom]['alg_bytes'] / parts / 1e9:.1f} GB per quotient launch: the "
                            "interpreter re-reads a column at every use and its local-memory register file competes for L2 (DESIGN.md 3.4)")
        elif per:
            traffic = per
            traffic_note = "dram bytes of one launch (ncu --set full, profiles/)"
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["achieved_gbs"] / peak,
                "peak_source": "MEASURED_PEAKS.json (sustained copy bandwidth: the kernel runs inside a long step)" if peaks else "fallback 6650 GB/s",
                "traffic": traffic, "traffic_note": traffic_note,
                "note": "dominant kernel of the proof by measured device time; all three hot kernels are bound by the integer-multiply pipe "
                        "(254-bit Montgomery arithmetic), not by HBM: see DESIGN.md section 2 and profiles/r02_microbench_pipes.txt",
                "kernels": kernels}
    vk_bytes = pk.vk_bytes()      # collective when world > 1: every rank calls it
    verdict = verify_with_oracle(sc, vk_bytes, proof, inst_h, fixed_h, sigma_h) if rank == 0 else None
    if rank == 0 and not (verdict["verified"] and verdict["tampered_rejected"]):
        failures.append("k=20 proof rejected by the oracle verifier")
    if world > 1:
        # every rank must hold the same proof bytes
        import hashlib
        hsh = torch.tensor(list(hashlib.sha256(proof).digest()), dtype=torch.int64, device="cuda")
        lo, hi = hsh.clone(), hsh.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(torch.equal(lo, hi))
        extras["identical_proof_on_all_ranks"] = same
        if not same:
            failures.append("proof bytes differ between ranks")
    h2d = sc.shape["advice_columns"] * (1 << K_PROOF) * 32 + (1 << K_PROOF) * 32
    shape = dict(sc.shape)
    shape.update(setup)
    extras["proof_super_shape_k20"] = {"shape": shape, "proof_bytes": len(proof), "seconds_device_resident_witness": sec_dev, "seconds_host_witness": sec_e2e,
                                       "kernel_launches": launches, **(verdict or {})}
    pk.close()
    del sc, pk, prove_host, prove_dev
    pin.keep.clear()
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ extras
    if not args.no_extras and world == 1:
        try:
            extras["ntt_2^24_round_trip"] = bench_ntt(ctx, A, peak, peaks, args)
        except Exception as e:
            extras["ntt_error"] = repr(e)
        try:
            extras["msm_2^20"] = bench_msm(ctx, A, peak, args)
        except Exception as e:
            extras["msm_error"] = repr(e)
        try:
            sck, pkk, fk, sk, setk = build_case("keccak", 17, 0, pin)
            ph, pd, ik = make_provers(sck, pkk, pin)
            sd, _ = time_steps(pd, 2, 3, barrier)
            se, prf = time_steps(ph, 1, 3, barrier)
            v = verify_with_oracle(sck, pkk.vk_bytes(), prf, ik, fk, sk)
            if not (v["verified"] and v["tampered_rejected"]):
                failures.append("k=17 proof rejected by the oracle verifier")
            extras["proof_keccak_shape_k17"] = {"shape": {**sck.shape, **setk}, "proof_bytes": len(prf), "seconds_device_resident_witness": sd,
                                                "seconds_host_witness": se, **v}
            pkk.close()
            del sck, pkk, ph, pd
            pin.keep.clear()
            torch.cuda.empty_cache()
        except Exception as e:
            extras["proof_keccak_error"] = repr(e)
    if not args.no_extras and world > 1:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        try:
            import multi_gpu_check
            res = multi_gpu_check.run(sizes=(22, 24, 26), msm_log=20, ctx=ctx)
            extras["sharded_paths"] = res
            if not res.get("all_ranks_ok", False):
                failures.append("sharded NTT / MSM mismatch")
            extras["msm_2^26_sharded"] = bench_msm_sharded(ctx, A, world, rank)
        except Exception as e:
            extras["sharded_error"] = repr(e)
            failures.append("sharded paths raised " + repr(e))

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            k_s, times, cores = cpu_proof_sample(25.0, 1)
            scale = 1 << (K_PROOF - k_s)
            cpu_baseline = {"value": times[0] * scale, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"one oracle create_proof (restated halo2 prover over the OpenMP C oracle) of the same shape at k={k_s}: {times[0]:.2f} s, "
                                      f"scaled x{scale} (linear in rows: an underestimate of the CPU time)"}
            cpu_baseline["primitive_model"] = cpu_primitive_model(shape)
        except Exception as e:
            cpu_baseline = {"error": repr(e)}

    if rank == 0:
        line = {"metric": METRIC, "value": sec_dev, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": sec_dev * 1e3,
                "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
                "dtype": "u256 (8x u32 Montgomery limbs, BN254 Fr/Fq)", "data": "synthetic (seeded satisfying witness of the stand-in; see tests/standins.py)",
                "config": config_dict(world),
                "e2e": {"value": sec_e2e, "unit": UNIT, "ms_per_step": sec_e2e * 1e3, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": len(proof)},
                "gpu_launches": launches * K, "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks, "extras": extras}
        if failures:
            line["failures"] = failures
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if failures:
        sys.exit(1)


def bench_ntt(ctx, A, peak, peaks, args):
    """BASELINE configs[1]: 2^24 Fr NTT forward + inverse round trip, data resident in HBM; e2e through the host-pointer entry point"""
    import numpy as np
    import torch
    w, wi = A.root_of_unity(LOG_N)
    n_can = torch.tensor([[N_PTS, 0, 0, 0]], dtype=torch.int64, device="cuda")
    ninv = A.field_unop_dev(A.FR, A.UOP_INV, A.field_unop_dev(A.FR, A.UOP_TO_MONT, n_can)).cpu().numpy().view(np.uint64)[0]
    data = A.random_fr_dev(N_PTS, 1000)
    orig = data.clone()

    def step_dev():
        A.best_fft_dev(data, w, LOG_N)
        A.best_fft_dev(data, wi, LOG_N, scale=ninv)
    for _ in range(3):
        step_dev()
    torch.cuda.synchronize()
    assert torch.equal(data, orig), "round trip does not restore the input"
    K = 20
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        step_dev()
    e1.record()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count - l0
    ms_step = ms_total / K
    host = torch.empty((N_PTS, 4), dtype=torch.int64).pin_memory()
    host.copy_(orig)

    def step_e2e():
        A.best_fft_pinned(host, w, LOG_N)
        A.best_fft_pinned(host, wi, LOG_N, scale=ninv)
    step_e2e()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        step_e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / 3
    assert torch.equal(host, orig.cpu()), "e2e round trip does not restore the input"
    passes = launches // (2 * K)
    avg_launch_s = ms_total * 1e-3 / launches
    burst = float(peaks.get("hbm_gbs", peak))
    achieved = (ALG_BYTES_PER_DIR / passes) / avg_launch_s / 1e9
    out = {"butterflies_per_s": 2 * BUTTERFLIES_PER_DIR / (ms_step * 1e-3), "ms_per_round_trip": ms_step, "gpu_launches": launches,
           "e2e": {"butterflies_per_s": 2 * BUTTERFLIES_PER_DIR / (e2e_ms * 1e-3), "ms_per_round_trip": e2e_ms, "h2d_bytes_per_step": 2 * 32 * N_PTS,
                   "d2h_bytes_per_step": 2 * 32 * N_PTS},
           "roofline": {"bound": "hbm", "kernel": "ntt_tile_kernel", "launches_per_transform": passes, "achieved": achieved, "peak": burst, "unit": "GB/s",
                        "frac": achieved / burst, "alg_bytes_per_launch": ALG_BYTES_PER_DIR / passes,
                        "traffic": 1213.4e6,
                        "traffic_note": "dram read+write per launch, mean of the three passes of a transform (ncu --set full, profiles/r02_ntt_tile_v5_ncu.txt: "
                                        "1586 / 1026 / 1031 MB; pass 1 also reads the 537 MB boundary-twiddle table)"}}
    if not args.no_cpu_baseline:
        orc = load_oracle()
        a = orig.cpu().numpy().view(np.uint64).copy()
        orc.best_fft(a[: 1 << 16].copy(), orc.fr_omega(16), 16)
        t0 = time.perf_counter()
        f = orc.best_fft(a, w, LOG_N)
        orc.best_fft(f, wi, LOG_N)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 2 * BUTTERFLIES_PER_DIR / dt, "unit": "butterflies/s", "cores": orc.num_threads(), "kind": "port",
                               "sample": "one full 2^24 fwd+inv round trip, oracle best_fft (OpenMP, threads spread over the sockets)", "seconds": dt}
    return out


def bench_msm(ctx, A, peak, args):
    """BASELINE configs[0]: 2^20-point G1 MSM; plain entry point (bases as given) and the SRS handle (ParamsKZG::commit: window-shifted
    copies of the fixed bases precomputed at load time, one bucket set, no Horner)"""
    import numpy as np
    import torch
    from zkb200.params import ParamsKZG, g1_generator
    n = 1 << MSM_LOG_N
    bases = A.g1_fixed_base_mul_dev(g1_generator(), A.random_fr_dev(n, 7))
    scal = A.random_fr_dev(n, 77)

    def timed(fn, reps=5):
        for _ in range(2):
            r = fn()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(reps):
            r = fn()
        m1.record()
        torch.cuda.synchronize()
        return m0.elapsed_time(m1) / reps, r
    ms_plain, r = timed(lambda: A.best_multiexp_dev(scal, bases))
    adds_plain = A.msm_last_adds(ctx)
    srs = ParamsKZG(MSM_LOG_N, bases, bases).load()
    ms_srs, r2 = timed(lambda: srs.commit(scal))
    adds_srs = A.msm_last_adds(ctx)
    assert r2.compressed == r.compressed, "SRS-handle commitment differs from the plain MSM"
    ctx.prof_enable(True)
    ctx.prof_read(1, reset=True)
    A.best_multiexp_dev(scal, bases)
    cnt, ms_acc = ctx.prof_read(1, reset=True)
    ctx.prof_enable(False)
    out = {"ms": ms_plain, "g1_adds": adds_plain, "g1_adds_per_s": adds_plain / (ms_plain * 1e-3),
           "srs_commit": {"ms": ms_srs, "g1_adds": adds_srs, "g1_adds_per_s": adds_srs / (ms_srs * 1e-3),
                          "note": "zkb_srs_commit_dev: what create_proof uses (fixed SRS bases, shifted copies built once at zkb_srs_load)"},
           "commitment": r.compressed.hex(),
           "roofline": {"bound": "hbm", "kernel": "msm_acc_chunk_kernel", "achieved": n * 96 / (ms_acc / max(cnt, 1) * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": n * 96 / (ms_acc / max(cnt, 1) * 1e-3) / 1e9 / peak, "alg_bytes_per_launch": n * 96, "avg_launch_ms": ms_acc / max(cnt, 1),
                        "traffic": None, "note": "bucket accumulation is bound by the integer-multiply pipe (87.6 % fmaheavy, profiles/r02_msm_kernels_ncu.txt)"}}
    if not args.no_cpu_baseline:
        orc = load_oracle()
        hs, hb = scal.cpu().numpy().view(np.uint64), bases.cpu().numpy().view(np.uint64)
        orc.best_multiexp(hs[:1 << 12], hb[:1 << 12])
        t0 = time.perf_counter()
        rr = orc.best_multiexp(hs, hb)
        dt = time.perf_counter() - t0
        same = bytes(orc.g1_compress(orc.g1_to_affine(rr))) == r.compressed
        out["cpu_baseline"] = {"value": adds_plain / dt, "unit": "G1-adds/s (the GPU's add count / CPU seconds)", "cores": orc.num_threads(), "kind": "port",
                               "sample": "one full 2^20 oracle best_multiexp (halo2's window rule, OpenMP chunks)", "seconds": dt, "bit_exact_vs_gpu": bool(same)}
    return out


def bench_msm_sharded(ctx, A, world, rank):
    """BASELINE configs[4]: 2^26-point MSM sharded by point range over the ranks (2^26 / world points per GPU, bases generated on the
    device), partial sums all-gathered (64 B per rank).  Checked against the sum of the per-rank partials recomputed slice by slice."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from zkb200 import parallel
    from zkb200.params import g1_generator
    total_log = 26
    n_loc = (1 << total_log) // world
    bases = A.g1_fixed_base_mul_dev(g1_generator(), A.random_fr_dev(n_loc, 9000 + rank))
    scal = A.random_fr_dev(n_loc, 9100 + rank)
    best = None
    for _ in range(3):
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        aff, comp = parallel.msm_sharded_dev(scal, bases, ctx=ctx)
        e1.record(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda"); dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        best = float(ms.item()) if best is None else min(best, float(ms.item()))
    adds = A.msm_last_adds(ctx)
    t = torch.tensor([adds], dtype=torch.int64, device="cuda"); dist.all_reduce(t)
    # cross-check: the local partial recomputed in 8 slices (different window sizes / bucket sets) and combined by all-gather on the host side
    parts = []
    sl = n_loc // 8
    for i in range(8):
        parts.append(A.best_multiexp_dev(scal[i * sl:(i + 1) * sl], bases[i * sl:(i + 1) * sl]).affine)
    loc_aff, _ = parallel.g1_sum_affine(np.stack(parts))
    aff2, comp2 = parallel.combine_msm_partials(loc_aff, device="cuda")
    ok = comp2 == comp
    return {"points": 1 << total_log, "points_per_gpu": n_loc, "ms": best, "g1_adds": int(t.item()), "g1_adds_per_s": int(t.item()) / (best * 1e-3),
            "alg_bytes": (1 << total_log) * 96, "matches_sliced_recomputation": bool(ok), "commitment": comp.hex()}


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the source tree may be read-only: nothing (not even __pycache__) is written there
    main()
