"""Cost model of the verification hot path -- the single source of the unit counts behind `roofline` in bench.py
(SURVEY.md §8(d) "canonical algorithmic cost model v1") and of the judge's re-computation.

Work unit  W = one 32x32->64-bit unsigned multiply (one IMAD.WIDE.U32).  Additions / carries are not counted.
The CANONICAL counts are those of textbook algorithms (schoolbook Fp6, Jacobian formulas, binary NAF subgroup
check, 4-bit windows): they are algorithm-independent "how much arithmetic does one verification stand for" figures,
so a leaner implementation legitimately shows an algorithmic fraction above its physical one.  The EXECUTED counts
are what the shipped kernels really multiply (counted by the test-only counter of the host build of the device
headers, tests/test_device_formulas_hostsim.py::test_executed_multiply_counts_match_design_doc pins them to this
file); the instruction-level figures of an ncu capture live in profiles/r2_ncu_constants.json together with the hash
of the library they were taken from.

Reference call stacks: Signature::verify src/signature.rs:181-205, hash_message :274-306, verify_batch
src/batch.rs:31-130."""
import hashlib
import json
import os

ROOT = os.path.dirname(os.path.abspath(__file__))

# ---- canonical model v1 (SURVEY.md §8(d) table) --------------------------------------------------------------------
W_FP_MUL, W_FP_SQR = 4, 3
W_FP6_MUL = 36 * W_FP_MUL                       # 144: schoolbook, x7 folds are shifts
W_FP6_SQR = 6 * W_FP_SQR + 15 * W_FP_MUL        # 78
W_JAC_DBL = 1 * W_FP6_MUL + 8 * W_FP6_SQR       # 768   dbl-2007-bl, a = 1
W_JAC_MADD = 7 * W_FP6_MUL + 4 * W_FP6_SQR      # 1320  madd-2007-bl
W_JAC_ADD = 11 * W_FP6_MUL + 5 * W_FP6_SQR      # 1974  add-2007-bl
RESCUE_ROUNDS = 7
W_PERMUTATION = RESCUE_ROUNDS * (12 * (2 * W_FP_SQR + 2 * W_FP_MUL) + 12 * (63 * W_FP_SQR + 9 * W_FP_MUL) + 2 * 144 * W_FP_MUL)  # 28 140
W_SUBGROUP_CHECK = 254 * W_JAC_DBL + 90 * W_JAC_MADD                         # 313 872: binary NAF of q (weight 91)
W_DOUBLE_BASE = (1 * W_JAC_DBL + 6 * W_JAC_ADD) + 252 * W_JAC_DBL + 64 * W_JAC_ADD + 64 * W_JAC_MADD   # 416 964
W_X_COMPARE = W_FP6_SQR + W_FP6_MUL                                          # 222
W_DECOMPRESS = 384 * W_FP6_SQR + 96 * W_FP6_MUL                              # 43 776: Fp6 square root
W_ZQ_MULS = 300                                                              # two 256-bit products mod q


def permutations_for(msg_len: int) -> int:
    """Rescue permutations of hash_message: 13 fixed elements + ceil(L / 7) message elements, rate 8; a partial last
    block costs one more permutation (padding element), a full one does not (src/signature.rs:284-301)."""
    elems = 13 + -(-msg_len // 7)
    return -(-elems // 8)


def w_per_hash(msg_len: int) -> int:
    return permutations_for(msg_len) * W_PERMUTATION


def w_per_verify(msg_len: int) -> int:
    """Canonical W of one Signature::verify: 787 338 for an 8-byte message."""
    return w_per_hash(msg_len) + W_SUBGROUP_CHECK + W_DOUBLE_BASE + W_X_COMPARE


def msm_plan(npoints: int, c_override: int = 0):
    """The window width the host planner picks (csrc/batch.cuh: msm_make_plan) -> (c, K, B)."""
    best, plan = None, None
    for c in range(4, 17):
        K = (256 + c - 1) // c
        B = 1 << (c - 1)
        cost = npoints * K + 3.0 * K * B
        if best is None or cost < best:
            best, plan = cost, (c, K, B)
    if 4 <= c_override <= 16:
        c = c_override
        plan = (c, (256 + c - 1) // c, 1 << (c - 1))
    return plan


def w_per_batch_signature(n: int, msg_len: int, plan=None) -> float:
    """Canonical W per signature of verify_batch over n signatures with the Pippenger plan (c, K, B) actually used
    (default: the planner's choice for 2n points): hash + decompression + two Z_q products + 2 K mixed additions
    (one per window and point) + the bucket reduction (2 B full additions per window) and the Horner tail (c doublings +
    one addition per window) and the final fixed-base product amortised over the batch."""
    c, K, B = plan or msm_plan(2 * n)
    per_sig = w_per_hash(msg_len) + W_DECOMPRESS + W_ZQ_MULS + 2 * K * W_JAC_MADD
    per_batch = K * 2 * B * W_JAC_ADD + K * (c * W_JAC_DBL + W_JAC_ADD) + 20 * W_JAC_MADD + W_X_COMPARE
    return per_sig + per_batch / max(n, 1)


# ---- executed by the shipped kernels (host-build counter; pinned by the CPU test named above) ------------------------
W_EXECUTED_FAST_L8 = 335892       # k_verify_fast, 8-byte message: products of the (X, Y, w) path incl. 2 permutations
W_EXECUTED_EXACT_L8 = 529896      # k_verify (exact Jacobian path)
W_EXECUTED_REG_L8 = 80219         # k_verify_reg (registered key, 8-byte message): 2 permutations + table additions
W_EXECUTED_PER_PERMUTATION = 28000


def w_executed_fast(msg_len: int) -> int:
    return W_EXECUTED_FAST_L8 + (permutations_for(msg_len) - 2) * W_EXECUTED_PER_PERMUTATION


# ---- algorithmic HBM bytes (irrelevant for this path, reported for completeness) -------------------------------------
def hbm_bytes_per_verify(msg_len: int) -> int:
    return 81 + 96 + 1 + msg_len + 8 + 1   # signature, key, identity flag, message, offset, verdict


# ---- peaks -----------------------------------------------------------------------------------------------------------
def nominal_peak_w_per_s(sm_count: int = 148, sm_mhz: float = 1965.0) -> float:
    """32 IMAD.WIDE per clock per SM (measured: 29.4, profiles/r1_imad_probe.log)."""
    return sm_count * 32 * sm_mhz * 1e6


# ---- constants taken from an ncu capture, tied to the library they were measured on -----------------------------------
def library_sha256(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def ncu_constants():
    """profiles/r2_ncu_constants.json: {"library_sha256", "source_sha256", "k_verify_fast": {"log2n": {"dram_bytes": ..,
    "inst_per_warp": .., "wide_inst_per_warp": ..}}}; None when no capture has been committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_constants.json")) as f:
            return json.load(f)
    except Exception:
        return None


def source_sha256() -> str:
    """Hash of the CUDA sources the library is built from (the .so itself differs between builds by embedded paths)."""
    d = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    h = hashlib.sha256()
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(d, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    for name in ("cheetah_params.h", "fp_sqrt_tables.h"):
        with open(os.path.join(ROOT, "include", name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()


if __name__ == "__main__":
    print(json.dumps({"w_per_verify_L8": w_per_verify(8), "w_per_verify_L80": w_per_verify(80), "w_per_hash_L8": w_per_hash(8),
                      "w_per_batch_signature_2^16_L8": w_per_batch_signature(1 << 16, 8), "plan_2^17_points": msm_plan(1 << 17),
                      "w_per_batch_signature_2^21_L8": w_per_batch_signature(1 << 21, 8), "plan_2^22_points": msm_plan(1 << 22),
                      "w_executed_fast_L8": w_executed_fast(8), "w_executed_reg_L8": W_EXECUTED_REG_L8, "source_sha256": source_sha256()}, indent=1))
