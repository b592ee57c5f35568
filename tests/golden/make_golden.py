"""Extract golden vectors for the hot path from the reference's own fixture.

Run against a checkout of scroll-tech/zkevm-circuits:  python tests/golden/make_golden.py <zkevm-circuits checkout>
Source: aggregator/data/batch-task.json -> chunk_proofs[0]  (used by the reference's tests at
aggregator/src/tests/aggregation.rs:160,244).  It is a genuine SHPLONK proof of the k=25 thin
compression circuit together with its vk and snark-verifier Protocol.  We keep only what pins the
encodings/constants of the MSM/NTT path (SURVEY.md 8c): Montgomery limb form, domain generators,
G1 compression, proof layout, evaluation order, transcript_repr and PARAMS_G2_SECRET_POWER.
"""
import base64, json, os, re, sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    d = json.load(open(f"{ref}/aggregator/data/batch-task.json"))
    c = d["chunk_proofs"][0]
    pr = json.loads(base64.b64decode(c["protocol"]))
    out = {
        "source": "aggregator/data/batch-task.json chunk_proofs[0]",
        "git_version": c["git_version"],
        "proof_hex": base64.b64decode(c["proof"]).hex(),
        "vk_hex": base64.b64decode(c["vk"]).hex(),
        "instances_hex": base64.b64decode(c["instances"]).hex(),
        "domain": pr["domain"],
        "preprocessed": pr["preprocessed"],
        "num_instance": pr["num_instance"],
        "num_witness": pr["num_witness"],
        "num_challenge": pr["num_challenge"],
        "evaluations": pr["evaluations"],
        "queries": pr["queries"],
        "quotient_num_chunk": pr["quotient"]["num_chunk"],
        "transcript_initial_state": pr["transcript_initial_state"],
        # snark-verifier's own spelling of the quotient numerator (expression tree over polys p0..p12, challenges, Lagrange
        # polynomials): tests/test_fixture_proof.py evaluates it at the proof's point and compares with the oracle's formulas
        "quotient_numerator": pr["quotient"]["numerator"],
    }
    # Montgomery-form constants appearing inside the quotient numerator: 1, DELTA, DELTA^2
    consts = []
    def walk(e):
        if isinstance(e, dict):
            for k, v in e.items():
                if k == "Constant" and v not in consts:
                    consts.append(v)
                else:
                    walk(v)
        elif isinstance(e, list):
            for v in e:
                walk(v)
    walk(pr["quotient"]["numerator"])
    out["numerator_constants_mont_limbs"] = consts
    src = open(f"{ref}/prover/src/utils.rs").read()
    m = re.search(r'PARAMS_G2_SECRET_POWER: &str = "(.*)";', src)
    out["params_g2_secret_power"] = m.group(1)
    with open(os.path.join(HERE, "thin_chunk_proof.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", os.path.join(HERE, "thin_chunk_proof.json"))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_golden.py <zkevm-circuits checkout>")
    main(sys.argv[1])
