"""CPU tests: the oracle restatements against the reference's golden vectors (tests/golden, produced by
the unmodified ctc_fast.pyx), and bit for bit against what the reference itself computed on the same inputs
(tests/golden/ctc_reference_exact.npz, from tests/golden/gen_ctc_reference_exact.py)."""
import numpy as np
import pytest

import recipes
from oracle import ctc_oracle, brnn_oracle

REL = 1e-12


def _run(name):
    probs, seq = recipes.ctc_case(name)
    return probs, seq, ctc_oracle.ctc_loss(np.asfortranarray(probs.astype(np.float64)), seq)


def _assert_grad_is_reference(grad, golden_ref, key):
    """Bit-exact: the recorded sample of the reference's gradient value for value, and all of it by digest."""
    np.testing.assert_array_equal(recipes.grad_sample(grad), golden_ref[key + "/sample"])
    assert recipes.grad_digest(grad) == golden_ref[key + "/digest"].tobytes(), key


@pytest.mark.parametrize("name", recipes.ALL_CTC)
def test_c_restatement_matches_golden(name, golden_ctc):
    probs, seq, (nll, grad, skip) = _run(name)
    assert bool(golden_ctc[name + "/skip"]) == skip
    if skip:
        assert not grad.any()
        return
    g_nll = float(golden_ctc[name + "/nll"])
    if np.isinf(g_nll):
        assert np.isinf(nll)
    else:
        assert abs(nll - g_nll) <= REL * abs(g_nll)
    st = recipes.golden_stride(*probs.shape)
    np.testing.assert_allclose(grad[:, ::st], golden_ctc[name + "/grad"], rtol=0, atol=2e-7)  # stored as f32
    assert abs(np.linalg.norm(grad) - float(golden_ctc[name + "/gradnorm"])) <= 1e-10


def test_known_answer_time_trials():
    """ctc/time_trials.py:13-25 recipe on float64 probs -> the value recorded in BASELINE.md."""
    params, seq = recipes.time_trials()
    nll, grad, skip = ctc_oracle.ctc_loss(np.asfortranarray(params), seq)
    assert not skip
    assert abs(nll - 1710.233966660) < 1e-6
    assert abs(np.linalg.norm(grad) - 26.721212367) < 1e-6
    assert np.abs(grad.sum(axis=0)).max() < 1e-12      # gradient columns sum to zero


@pytest.mark.parametrize("name", recipes.ALL_CTC)
def test_c_restatement_matches_reference_live(name, golden_ref):
    probs, seq, (nll, grad, skip) = _run(name)
    key = "ctc/" + name
    r_nll, r_skip = float(golden_ref[key + "/nll"]), bool(golden_ref[key + "/skip"])
    assert skip == r_skip
    if not skip:
        assert (nll == r_nll) or (np.isinf(nll) and np.isinf(r_nll))
        _assert_grad_is_reference(grad, golden_ref, key)          # bit-exact: same operation order in float64


def test_reference_contract_errors():
    p, s = recipes.ctc_case("c1")
    with pytest.raises(ValueError):
        ctc_oracle.ctc_loss(np.ascontiguousarray(p.astype(np.float64)), s)   # C-ordered: reference raises too


def test_best_path_restatement(golden_ref):
    hyp, align = ctc_oracle.decode_best_path(recipes.best_path_probs())
    assert hyp == [3, 3, 5] and align == [2, 4, 7]
    assert (golden_ref["best_path/hyp"].tolist(), golden_ref["best_path/align"].tolist()) == (hyp, align)


def test_brnn_restatement_matches_golden(golden_brnn):
    cfg, data, labels = recipes.rnnetcpu()
    np.random.seed(33); np.random.randn(20, 10)
    nn = brnn_oracle.NNet(cfg["inputDim"], cfg["outputDim"], cfg["layerSize"], cfg["numLayers"], cfg["maxBatch"],
                          temporalLayer=cfg["temporalLayer"], dtype=np.float64)
    nn.initParams()
    for i, (w, b) in enumerate(nn.stack):
        assert np.array_equal(w.astype(np.float32), golden_brnn["rnnetcpu/w%d" % i])   # same draw order
    cost, grad, skip = nn.costAndGrad(data.astype(np.float32), labels)
    assert not skip and abs(cost - float(golden_brnn["rnnetcpu/cost"])) < 1e-9
    for i, (dw, db) in enumerate(grad):
        np.testing.assert_allclose(dw, golden_brnn["rnnetcpu/dw%d" % i], rtol=1e-9, atol=1e-12)


# ---- the BRNN restatement pinned to the reference's own NumPy BRNN (debug-utils/rnnetcpu.py) -----------------
RNNETCPU_CASES = ["selftest", "tl1_of_2", "tl3_of_5", "no_temporal", "long_T"]


@pytest.mark.parametrize("name", RNNETCPU_CASES)
def test_brnn_restatement_pinned_to_reference_rnnetcpu(name, golden_rnnetcpu):
    """tests/golden/rnnetcpu_ref.npz holds inputs and outputs of the REFERENCE's rnnetcpu.RNNet.costAndGrad
    (rnnetcpu.py:54-150), produced by tests/golden/gen_rnnetcpu_ref.py from the file as it lies in
    /root/reference (print/xrange/tabs converted mechanically, CTC = the unmodified ctc_fast.pyx).  The
    restatement, configured as that file computes -- float64 weights as drawn, no 20.0 clip (rnnetcpu.py:82-90),
    no float32 hand-offs, no L2 -- must reproduce cost and every gradient to 1e-12."""
    g = golden_rnnetcpu
    seed, D, T, K, H, N, tl = (int(x) for x in g[name + "/cfg"])
    nn = brnn_oracle.NNet(D, K, H, N, T, temporalLayer=tl, dtype=np.float64, round_f32=False)
    np.random.seed(seed); np.random.randn(D, T)                     # same global stream position as the reference
    nn.initParams()
    assert len(nn.stack) == int(g[name + "/nstack"])
    for i, (w, b) in enumerate(nn.stack):                           # same shapes and np.random draw order ...
        assert np.array_equal(w, g["%s/w%d" % (name, i)].astype(np.float32).astype(np.float64))
        w[...] = g["%s/w%d" % (name, i)]                            # ... then the reference's un-rounded float64 values
        b[...] = g["%s/b%d" % (name, i)]
    nn.maxAct = np.inf                                              # rnnetcpu.py has no clip
    cost, grad, skip = nn.costAndGrad(g[name + "/data"], g[name + "/labels"])
    assert not skip
    ref = float(g[name + "/cost"])
    assert abs(cost - ref) <= 1e-12 * abs(ref), (cost, ref)
    for i, (dw, db) in enumerate(grad):
        rdw = g["%s/dw%d" % (name, i)]
        assert np.abs(dw - rdw).max() <= 1e-12 * max(1.0, np.abs(rdw).max()), i
        if i <= N:
            rdb = g["%s/db%d" % (name, i)]
            assert np.abs(db - rdb).max() <= 1e-12 * max(1.0, np.abs(rdb).max()), i


def test_reference_selftest_known_answer(golden_rnnetcpu):
    """`COST 12.023458823` is what the reference's own `python rnnetcpu.py` prints (rnnetcpu.py:180-193)."""
    assert abs(float(golden_rnnetcpu["selftest/cost"]) - 12.023458823) < 5e-10


def test_brnn_restatement_gradcheck():
    """Finite-difference check of the restatement itself (tolerance of the reference's own check,
    |analytic - numeric| <= 1e-4: rnnetcpu.py:165, ctc/gradcheck.py:40)."""
    rng = np.random.RandomState(3)
    np.random.seed(3)
    nn = brnn_oracle.NNet(7, 5, 12, 3, 9, temporalLayer=2, dtype=np.float64, round_f32=False)
    nn.initParams()
    data = rng.randn(7, 9)
    labels = np.array([1, 2, 2, 4], dtype=np.int32)
    cost, grad, _ = nn.costAndGrad(data, labels)
    grad = [[dw.copy(), db.copy()] for dw, db in grad]
    eps = 1e-6
    for pi, (w, b) in enumerate(nn.stack):
        for _ in range(6):
            i, j = rng.randint(w.shape[0]), rng.randint(w.shape[1])
            w[i, j] += eps; cp = nn.costAndGrad(data, labels)[0]
            w[i, j] -= 2 * eps; cm = nn.costAndGrad(data, labels)[0]
            w[i, j] += eps
            assert abs(grad[pi][0][i, j] - (cp - cm) / (2 * eps)) < 1e-4


def test_brnn_float32_mode_close_to_float64():
    datas, labelss = recipes.synth_batch(13, 11, [20, 17], [5, 4], seed=1)
    outs = []
    for dt in (np.float64, np.float32):
        np.random.seed(5)
        nn = brnn_oracle.NNet(13, 11, 32, 2, 20, temporalLayer=1, dtype=dt)
        nn.initParams()
        costs, grad, skips = nn.costAndGradBatch(datas, labelss)
        outs.append((costs, np.concatenate([g[0].ravel() for g in grad]).astype(np.float64)))
    assert np.allclose(outs[0][0], outs[1][0], rtol=1e-4)
    assert np.linalg.norm(outs[0][1] - outs[1][1]) / np.linalg.norm(outs[0][1]) < 1e-4


# ---- blank-forced CTC (ctc_fast_blankforce.pyx) and the uni-directional / feed-forward nets ------------
@pytest.mark.parametrize("name", recipes.ALL_BF)
def test_blankforce_restatement_matches_golden(name, golden_bf):
    probs, seq = recipes.bf_case(name)
    nll, grad, skip = ctc_oracle.ctc_loss_blankforce(np.asfortranarray(probs.astype(np.float64)), seq)
    assert bool(golden_bf[name + "/skip"]) == skip and not skip
    g_nll = float(golden_bf[name + "/nll"])
    assert abs(nll - g_nll) <= REL * abs(g_nll)
    st = recipes.golden_stride(*probs.shape)
    np.testing.assert_allclose(grad[:, ::st], golden_bf[name + "/grad"], rtol=0, atol=2e-7)
    assert abs(np.linalg.norm(grad) - float(golden_bf[name + "/gradnorm"])) <= 1e-10


@pytest.mark.parametrize("name", recipes.ALL_BF)
def test_blankforce_restatement_matches_reference_live(name, golden_ref):
    probs, seq = recipes.bf_case(name)
    p64 = np.asfortranarray(probs.astype(np.float64))
    nll, grad, skip = ctc_oracle.ctc_loss_blankforce(p64, seq)
    key = "bf/" + name
    assert skip == bool(golden_ref[key + "/skip"]) and nll == float(golden_ref[key + "/nll"])
    _assert_grad_is_reference(grad, golden_ref, key)                                # bit-exact
    hyp = ctc_oracle.decode_best_path_blankforce(p64)
    assert hyp == golden_ref[key + "/hyp"].tolist()


def test_blankforce_zero_probability_skips(golden_ref):
    """A zero frame normaliser is the reference's ZeroDivisionError -> skip (ctc_fast_blankforce.pyx:108-110)."""
    _, _, skip = ctc_oracle.ctc_loss_blankforce(*recipes.bf_zero_probability_case())
    assert skip
    assert bool(golden_ref["bf_zero_probability/skip"])


@pytest.mark.parametrize("kw", [dict(temporalLayer=2, unidirectional=True), dict(temporalLayer=-1)])
def test_rnn_variants_gradcheck(kw):
    """rnnet.py / nnet.py restatements: analytic vs central differences, the reference's own 1e-4 bound."""
    rng = np.random.RandomState(4)
    np.random.seed(4)
    nn = brnn_oracle.NNet(7, 5, 12, 3, 9, dtype=np.float64, round_f32=False, **kw)
    nn.initParams()
    assert len(nn.stack) == 4 + (1 if kw.get("unidirectional") else 0)          # rnnet.py:38-65 / nnet.py:22-23
    data = rng.randn(7, 9)
    labels = np.array([1, 2, 2, 4], dtype=np.int32)
    cost, grad, _ = nn.costAndGrad(data, labels)
    grad = [[dw.copy(), db.copy()] for dw, db in grad]
    eps = 1e-6
    for pi, (w, b) in enumerate(nn.stack):
        for _ in range(6):
            i, j = rng.randint(w.shape[0]), rng.randint(w.shape[1])
            w[i, j] += eps; cp = nn.costAndGrad(data, labels)[0]
            w[i, j] -= 2 * eps; cm = nn.costAndGrad(data, labels)[0]
            w[i, j] += eps
            assert abs(grad[pi][0][i, j] - (cp - cm) / (2 * eps)) < 1e-4


def test_rnn_variants_match_golden(golden_rnn):
    datas, labelss = recipes.rnn_variant_batch()
    for tag, _ in recipes.RNN_VARIANTS:
        nn = recipes.rnn_variant_net(brnn_oracle.NNet, tag, dtype=np.float64)
        recipes.rnn_variant_perturb(nn.stack, tag)
        for i, (w, b) in enumerate(nn.stack):
            assert np.array_equal(w.astype(np.float32), golden_rnn["%s/w%d" % (tag, i)])
        costs, grad, skips = nn.costAndGradBatch(datas, labelss)
        np.testing.assert_allclose(costs, golden_rnn[tag + "/costs"], rtol=1e-9)
        for i, (dw, db) in enumerate(grad):
            np.testing.assert_allclose(dw, golden_rnn["%s/dw%d" % (tag, i)], rtol=1e-9, atol=1e-12)
    assert int(golden_rnn["uni/clip_hits"]) > 0


# ---- randomised pinning of the restatements against the compiled reference modules ---------------------------
def test_c_restatement_equals_reference_on_random_shapes(golden_ref):
    """recipes.random_ctc_cases (T = 1, T = |l|, T < |l|, heavy label repetition, peaked distributions): the C
    restatement must agree with the unmodified ctc_fast.pyx bit for bit (same float64 operation order), skip flags
    included."""
    r_nlls, r_skips, r_digests = golden_ref["random/nll"], golden_ref["random/skip"], golden_ref["random/digest"]
    n_skip = n_inf = 0
    for case, (K, T, nlab, p, seq) in enumerate(recipes.random_ctc_cases()):
        nll, grad, skip = ctc_oracle.ctc_loss(p, seq)
        r_nll, r_skip = float(r_nlls[case]), bool(r_skips[case])
        assert skip == r_skip, (case, K, T, nlab)
        n_skip += skip
        if skip:
            continue
        if np.isinf(r_nll):
            n_inf += 1
            assert np.isinf(nll)
        else:
            assert nll == r_nll, (case, K, T, nlab, nll, r_nll)
        assert recipes.grad_digest(grad) == r_digests[case].tobytes(), (case, K, T, nlab)
    assert case == len(r_nlls) - 1
    assert n_skip > 0 and n_inf > 0          # the sample did reach the failure and the T < |l| paths


def test_blankforce_restatement_equals_reference_on_random_shapes(golden_ref):
    r_nlls, r_skips, r_digests = golden_ref["random_bf/nll"], golden_ref["random_bf/skip"], golden_ref["random_bf/digest"]
    for case, (K, T, L, p, seq) in enumerate(recipes.random_bf_cases()):
        nll, grad, skip = ctc_oracle.ctc_loss_blankforce(p, seq)
        r_nll, r_skip = float(r_nlls[case]), bool(r_skips[case])
        assert skip == r_skip, (case, K, T, L)
        if not skip:
            assert (nll == r_nll) or (np.isnan(nll) and np.isnan(r_nll)) or (np.isinf(nll) and np.isinf(r_nll)), (case, nll, r_nll)
            assert recipes.grad_digest(grad) == r_digests[case].tobytes(), (case, K, T, L)
    assert case == len(r_nlls) - 1
