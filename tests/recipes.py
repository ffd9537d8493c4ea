"""Deterministic input recipes shared by the golden generator and the tests.

All follow the reference's own eyeball tests (seed 33, legacy np.random streams):
  time_trials : /root/reference/ctc/time_trials.py:13-25  (K=40, |l|=125, T=1200, peaked probs)
  ctc_py      : /root/reference/ctc/ctc.py:143-152        (K=62, |l|=54, T=453, logits ~ N(0,1))
  c1          : BASELINE.json configs[0]                  (T=200, K=62, |l|=30)
  rnnetcpu    : /root/reference/ctc_fast/debug-utils/rnnetcpu.py:181-193 (D=20,T=10,K=6,H=30,N=3,tl=2)
"""
import hashlib

import numpy as np


def softmax_cols(x):
    x = x - x.max(axis=0)
    e = np.exp(x)
    return e / e.sum(axis=0)


def time_trials():
    np.random.seed(33)
    numPhones, seqLen, uttLen = 40, 125, 1200
    seq = np.floor(np.random.rand(seqLen) * numPhones).astype(np.int32)
    params = np.random.randn(numPhones, uttLen)
    params[seq, np.arange(seqLen)] = 3
    params[0, seqLen:] = 3
    params = np.exp(params)
    params = params / np.sum(params, axis=0)
    return params, seq


def ctc_py():
    np.random.seed(33)
    numPhones, seqLen, uttLen = 62, 54, 453
    seq = np.floor(np.random.rand(seqLen, 1) * numPhones).astype(np.int32).reshape(-1)
    logits = np.random.randn(numPhones, uttLen)
    return logits, seq


def synth_ctc(T, K, nlab, seed=33):
    """Sweep-style case: logits ~ N(0,1), labels uniform over non-blank (ctc/gradcheck.py:68-69)."""
    rng = np.random.RandomState(seed + 1000003 * T + 1009 * K + nlab)
    logits = rng.randn(K, T)
    seq = (1 + np.floor(rng.rand(nlab) * (K - 1))).astype(np.int32)
    return logits, seq


CTC_CASES = {
    # name: (T, K, |l|)
    "c1": (200, 62, 30),
    "sweep_100_10_32": (100, 32, 10),
    "sweep_500_100_62": (500, 62, 100),
    "sweep_500_300_128_infeasible_len": (100, 128, 300),
    "wsj_800_100_32": (800, 32, 100),
    "swbd_1500_150_35": (1500, 35, 150),
    "long_2000_300_128": (2000, 128, 300),
    "repeat_heavy": (64, 8, 31),
    "single_label": (5, 4, 1),
    "T_equals_L": (12, 9, 12),
    "T_equals_L_feasible": (12, 16, 12),
}


def ctc_case(name):
    """Returns (probs float32 K x T, seq int32).  probs are float32-rounded softmax outputs, which is
    what the reference's CTC receives from the GPU (brnnet.py:170-175)."""
    if name == "time_trials":
        p, s = time_trials()
        return p.astype(np.float32), s
    if name == "ctc_py":
        l, s = ctc_py()
        return softmax_cols(l).astype(np.float32), s
    T, K, nlab = CTC_CASES[name]
    logits, seq = synth_ctc(T, K, nlab)
    if name == "repeat_heavy":
        seq = (1 + (np.arange(nlab) // 3) % (K - 1)).astype(np.int32)   # runs of repeated labels
    if name == "T_equals_L_feasible":
        seq = (1 + np.arange(nlab)).astype(np.int32)                    # all distinct: exactly one path
    return softmax_cols(logits).astype(np.float32), seq


ALL_CTC = ["time_trials", "ctc_py"] + list(CTC_CASES)


def golden_stride(K, T):
    """Golden gradients of the big cases are stored for every 8th frame only (fixtures stay small)."""
    return 1 if K * T <= 50000 else 8


def grad_digest(grad):
    """SHA-256 of a float64 gradient in Fortran order, with -0.0 folded into 0.0 and every NaN into one bit
    pattern: two gradients have the same digest exactly when np.array_equal(a, b, equal_nan=True) holds."""
    g = np.asfortranarray(grad, dtype=np.float64) + 0.0
    g[np.isnan(g)] = np.nan
    return hashlib.sha256(g.tobytes(order="F")).digest()


def grad_sample(grad, n=256):
    """A fixed, seeded sample of n entries of a gradient (all of it when it is smaller), Fortran order."""
    flat = np.asarray(grad, dtype=np.float64).ravel(order="F")
    if flat.size <= n:
        return flat.copy()
    return flat[np.sort(np.random.RandomState(0).choice(flat.size, n, replace=False))]


def random_ctc_cases():
    """300 random (K, T, |l|) cases incl. T = 1, T = |l|, T < |l|, heavy label repetition and peaked
    distributions: yields (K, T, |l|, probs float64 K x T Fortran order, seq int32)."""
    rng = np.random.RandomState(2024)
    for _ in range(300):
        K = int(rng.randint(2, 40))
        T = int(rng.choice([1, 2, 3, 5, 8, 17, 40, 90]))
        nlab = int(rng.randint(1, max(2, min(T + 3, 25))))
        scale = float(rng.choice([0.5, 1.0, 4.0, 12.0]))
        probs = softmax_cols(rng.randn(K, T) * scale).astype(np.float32).astype(np.float64)
        if rng.rand() < 0.3:
            seq = np.full(nlab, 1 + rng.randint(K - 1), dtype=np.int32)           # one label repeated
        else:
            seq = (1 + rng.randint(0, K - 1, size=nlab)).astype(np.int32)
        yield K, T, nlab, np.asfortranarray(probs), seq


def random_bf_cases():
    """200 random blank-forced cases: yields (K, T, len(seq), probs float64 K x T Fortran order, seq int32)."""
    rng = np.random.RandomState(77)
    for _ in range(200):
        K = int(rng.randint(2, 30))
        T = int(rng.choice([1, 2, 4, 9, 33, 70]))
        L = int(rng.randint(1, 20))
        probs = softmax_cols(rng.randn(K, T) * float(rng.choice([1.0, 5.0]))).astype(np.float32).astype(np.float64)
        seq = rng.randint(0, K, size=L).astype(np.int32)
        if rng.rand() < 0.7:
            seq[::2] = 0                                                           # the usual interleaved blanks
        yield K, T, L, np.asfortranarray(probs), seq


def best_path_probs():
    """One-hot K=10 x T=9 probabilities along a path whose labels 1 and 8 the reference drops (ctc_fast.pyx:176-179)."""
    probs = np.zeros((10, 9))
    probs[[0, 3, 3, 0, 3, 1, 5, 5, 8], np.arange(9)] = 1.0
    return np.asfortranarray(probs)


def bf_zero_probability_case():
    """bf_small with an all-zero frame: a zero frame normaliser (ctc_fast_blankforce.pyx:108-110)."""
    probs, seq = bf_case("bf_small")
    p64 = np.asfortranarray(probs.astype(np.float64))
    p64[:, 4] = 0.0
    return p64, seq


def rnnetcpu():
    """Data, labels and an oracle-initialised parameter stack for the reference's CPU BRNN self-test."""
    np.random.seed(33)
    data = np.random.randn(20, 10)
    labels = np.arange(3).astype(np.int32)
    return dict(inputDim=20, outputDim=6, layerSize=30, numLayers=3, temporalLayer=2, maxBatch=10), data, labels


def synth_batch(inputDim, outputDim, lens, nlabs, seed=33):
    """Features randn(D,T) float32 (rnnetcpu.py:189), labels uniform over non-blank."""
    rng = np.random.RandomState(seed)
    datas = [rng.randn(inputDim, T).astype(np.float32) for T in lens]
    labels = [(1 + np.floor(rng.rand(n) * (outputDim - 1))).astype(np.int32) for n in nlabs]
    return datas, labels


# ---- blank-forced CTC (ctc_fast_blankforce.pyx): the sequence carries its blanks ---------------------
BF_CASES = {
    # name: (T, K, number of non-blank labels)
    "bf_c1": (200, 62, 30),
    "bf_small": (10, 6, 3),
    "bf_wsj": (800, 32, 100),
    "bf_long": (1500, 35, 300),
    "bf_T_less_than_L": (8, 10, 6),          # no exception in the reference: absum == 0 -> grad = probs
    "bf_no_leading_blank": (50, 20, 10),     # seq[0] != 0 exercises the row-0 quirk (:49)
    "bf_one_state": (7, 5, 0),
    "bf_peaked": (400, 40, 60),
}


def bf_case(name):
    """Returns (probs float32 K x T, seq int32 with blanks interleaved: 0 l1 0 l2 ... 0)."""
    T, K, nlab = BF_CASES[name]
    logits, lab = synth_ctc(T, K, nlab, seed=77)
    if name == "bf_peaked":
        logits = logits * 4.0
    seq = np.zeros(2 * nlab + 1, dtype=np.int32)
    seq[1::2] = lab
    if name == "bf_no_leading_blank":
        seq = seq[1:].copy()
    return softmax_cols(logits).astype(np.float32), seq


ALL_BF = list(BF_CASES)


RNN_VARIANTS = (("uni", dict(temporalLayer=2, unidirectional=True)), ("dnn", dict(temporalLayer=-1)))


def rnn_variant_batch():
    return synth_batch(13, 11, [30, 41, 12, 41], [7, 11, 3, 15], seed=11)


def rnn_variant_net(cls, tag, **extra):
    """The uni-directional (nnets/rnnet.py) / feed-forward (nnets/nnet.py) golden nets: D=13, K=11, H=64, N=3."""
    kw = dict(RNN_VARIANTS)[tag]
    np.random.seed(9)
    nn = cls(13, 11, 64, 3, 41, **dict(kw, **extra))
    nn.initParams()
    return nn


def rnn_variant_perturb(stack, tag):
    """Host-side edits of the freshly initialised stack (list of [w, b] arrays) that the golden nets carry."""
    for w, b in stack[:3]:
        b += 0.05
    if tag == "uni":
        stack[1][1] += 4.0          # some units reach the 20.0 clip (rnnet.py:32,113-116)
        stack[-1][0] *= 1.2
