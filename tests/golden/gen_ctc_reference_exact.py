"""Generates tests/golden/ctc_reference_exact.npz: what the REFERENCE ITSELF computes on the inputs of the bit-exact
tests in tests/test_oracle.py, so that those tests compare the C restatement (oracle/ctc_oracle.c) with the
reference without needing it.  The reference is oracle/_ref = the unmodified ctc_fast.pyx and
ctc_fast_blankforce.pyx compiled by oracle/build_ref.py, called through oracle.ctc_oracle.ref_ctc_loss*.

Per case the file holds nll (float64), skip, the SHA-256 of the whole float64 gradient (recipes.grad_digest) and a
fixed sample of its values (recipes.grad_sample); the blank-forced cases add the best-path hypothesis.

Run from the repo root:  python tests/golden/gen_ctc_reference_exact.py      (needs the reference sources that
oracle/build_ref.py compiles)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import recipes  # noqa: E402
from oracle import build_ref, ctc_oracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def _digest(grad):
    return np.frombuffer(recipes.grad_digest(grad), dtype=np.uint8)


def _case(out, key, nll, grad, skip):
    out[key + "/nll"] = np.float64(nll)
    out[key + "/skip"] = np.bool_(skip)
    out[key + "/digest"] = _digest(grad)
    out[key + "/sample"] = recipes.grad_sample(grad)


def main():
    build_ref.build()
    assert ctc_oracle.ref_module() is not None and ctc_oracle.ref_module("ctc_fast_blankforce") is not None, \
        "oracle/_ref could not be built"
    out = {}
    for name in recipes.ALL_CTC:
        probs, seq = recipes.ctc_case(name)
        _case(out, "ctc/" + name, *ctc_oracle.ref_ctc_loss(np.asfortranarray(probs.astype(np.float64)), seq))
    for name in recipes.ALL_BF:
        probs, seq = recipes.bf_case(name)
        p64 = np.asfortranarray(probs.astype(np.float64))
        _case(out, "bf/" + name, *ctc_oracle.ref_ctc_loss_blankforce(p64, seq))
        out["bf/%s/hyp" % name] = np.array(ctc_oracle.ref_module("ctc_fast_blankforce").decode_best_path(p64),
                                           dtype=np.int32)
    hyp, align = ctc_oracle.ref_module().decode_best_path(recipes.best_path_probs())
    out["best_path/hyp"], out["best_path/align"] = np.array(hyp, dtype=np.int32), np.array(align, dtype=np.int32)
    out["bf_zero_probability/skip"] = np.bool_(ctc_oracle.ref_ctc_loss_blankforce(*recipes.bf_zero_probability_case())[2])

    for key, cases, fn in (("random", recipes.random_ctc_cases(), ctc_oracle.ref_ctc_loss),
                           ("random_bf", recipes.random_bf_cases(), ctc_oracle.ref_ctc_loss_blankforce)):
        nlls, skips, digests = [], [], []
        for _, _, _, p, seq in cases:
            nll, grad, skip = fn(p, seq)
            nlls.append(nll); skips.append(skip); digests.append(_digest(grad))
        out[key + "/nll"] = np.array(nlls, dtype=np.float64)
        out[key + "/skip"] = np.array(skips, dtype=bool)
        out[key + "/digest"] = np.stack(digests)
        print("%-10s %d cases, %d skipped" % (key, len(nlls), int(np.sum(skips))))
    np.savez_compressed(os.path.join(HERE, "ctc_reference_exact.npz"), **out)


if __name__ == "__main__":
    main()
