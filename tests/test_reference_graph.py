"""CPU: the simulator graphs as the REFERENCE'S OWN code wires them (rl4rs/nets/*.py run through oracle/tf_eager_stub.py,
vectors committed by tests/golden/make_nets_golden.py and tests/golden/make_reference_golden.py) against (i) the NumPy
oracles the GPU tests compare with and (ii) the variable-scope plans of the TF1 checkpoint reader.  Pins wiring and scope
order, not the third-party layer arithmetic (see the stub's header)."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_nets_golden as mk                                   # noqa: E402

from golden_util import REFERENCE_DIR, check_fingerprint, digest, golden_names, load_fingerprint   # noqa: E402
from oracle.dien_np import DienOracle                           # noqa: E402
from oracle.dnn_np import DnnOracle                             # noqa: E402
from oracle.lstm_np import LstmOracle                           # noqa: E402
from oracle.widedeep_np import WideDeepOracle                   # noqa: E402
from rl4rs_b200.utils import tf_checkpoint as tfc               # noqa: E402

ORACLES = {"dien": DienOracle, "dnn": DnnOracle, "widedeep": WideDeepOracle, "lstm": LstmOracle}
RECORDS = os.path.join(REFERENCE_DIR, "records.npz")
PLANS = {"dien": tfc.dien_layer_plan, "dnn": tfc.dnn_layer_plan, "widedeep": tfc.widedeep_layer_plan, "lstm": tfc.lstm_layer_plan}


@pytest.fixture(scope="module")
def golden():
    g = np.load(os.path.join(os.path.dirname(mk.__file__), "nets", "reference_graph.npz"))
    return g, json.loads(str(g["meta"]))


@pytest.mark.parametrize("case", sorted(mk.CASES))
def test_oracle_reproduces_what_the_reference_graph_code_computes(golden, case):
    g, _ = golden
    algo = mk.CASES[case][0]
    w, _ = mk.checkpoint_of(case)
    obs, probs = ORACLES[algo](w, np.float64).forward(g["seq"], g["dense"], g["cat"])
    ref_obs, ref_probs = g[case + "_obs"], g[case + "_probs"]
    assert obs.shape == ref_obs.shape and probs.shape == ref_probs.shape == (len(g["cat"]), 2)
    np.testing.assert_allclose(obs, ref_obs, rtol=0, atol=1e-11 * max(1.0, np.abs(ref_obs).max()))
    np.testing.assert_allclose(probs, ref_probs, rtol=0, atol=1e-12)
    # the f32 oracle (what the CUDA path is held to at 1e-4) sits at f32 rounding of the same vectors
    o32, p32 = ORACLES[algo](w, np.float32).forward(g["seq"], g["dense"], g["cat"])
    rms = np.sqrt((ref_obs ** 2).mean(-1, keepdims=True))
    assert (np.abs(o32 - ref_obs) / np.maximum(np.abs(ref_obs), rms)).max() < 3e-5
    assert np.abs(p32 - ref_probs).max() < 1e-5


@pytest.mark.parametrize("case", sorted(mk.CASES))
def test_checkpoint_plan_follows_the_reference_creation_order(golden, case):
    """Keras names layers in construction order; the scopes the reader expects (INTEGRATION.md section 5) must be the
    ones the reference's code brings into existence, in that order, with those shapes."""
    _, meta = golden
    algo = mk.CASES[case][0]
    created = [(s, tuple(sh)) for s, _, sh in meta[case]["variables"]]
    plan = [(scope, tuple(shape)) for _, scope, shape in PLANS[algo](mk.SMALL)]
    if algo == "dnn":                                            # the reader skips the embedding that feeds nothing
        assert ("embedding_1", (600, 128)) in created
        created.remove(("embedding_1", (600, 128)))
    dedupe = lambda seq: [x for i, x in enumerate(seq) if i == 0 or x != seq[i - 1]]
    assert dedupe([s for s, _ in created]) == dedupe([s for s, _ in plan])
    assert sorted(created) == sorted(plan)                       # every scope owns exactly the planned shapes
    names = {n for _, n, _ in meta[case]["variables"]}
    expect = getattr(tfc, mk.CASES[case][3])(mk.SMALL)
    assert set(expect.values()) <= names
    layers = meta[case]["layers"]
    assert sum("simulator_obs" in l for l in layers) == 1 and sum("simulator_reward" in l for l in layers) == 1


def test_checkpoint_file_feeds_the_reference_graph(golden, tmp_path):
    """n1 end to end: W-table -> Saver-format bundle on disk -> TensorBundleReader -> the reference's graph code.  The
    reference's graph turned the tensors read back from the file into dien_stress_obs; the committed digest of those
    tensors (tests/golden/make_reference_golden.py) holds today's writer and reader to them."""
    w, _ = mk.checkpoint_of("dien_stress")
    rd = tfc.TensorBundleReader(tfc.save_dien_checkpoint(str(tmp_path / "sim"), w, mk.SMALL))
    ck = {name: rd.get_tensor(name) for name in rd.variables()}
    want = expected_nets()["checkpoint_file_tensors"]
    assert sorted(ck) == sorted(want)
    for name in sorted(ck):
        assert digest(ck[name]) == want[name], name


@pytest.mark.parametrize("case", sorted(mk.CASES))
def test_committed_vectors_are_what_the_reference_code_computes_now(golden, case):
    """The vectors were computed by the reference's graph from mk.checkpoint_of(case) and the committed feature rows;
    tests/golden/make_reference_golden.py re-ran that graph, found the vectors and scopes unchanged, and stored a digest
    of each checkpoint tensor.  Today's checkpoint_of must still give those tensors."""
    g, meta = golden
    _, ck = mk.checkpoint_of(case)
    want = expected_nets()["checkpoints"][case]
    assert sorted(ck) == sorted(want)
    for name in sorted(ck):
        assert digest(ck[name]) == want[name], (case, name)
    assert sorted(n for _, n, _ in meta[case]["variables"]) == sorted(ck)


def expected_nets():
    with open(os.path.join(REFERENCE_DIR, "expected.json")) as f:
        return json.load(f)["nets"]


def test_the_check_has_teeth(golden):
    """A mis-wired weight set (the two embedding tables swapped) must not reproduce the vectors."""
    g, _ = golden
    w, _ = mk.checkpoint_of("dien_stress")
    w = dict(w, emb_cat=w["emb_seq"], emb_seq=w["emb_cat"])
    obs, _ = DienOracle(w, np.float64).forward(g["seq"], g["dense"], g["cat"])
    assert np.abs(obs - g["dien_stress_obs"]).max() > 1e-3


@pytest.mark.parametrize("name", golden_names())
def test_the_references_own_stack_reproduces_the_fixtures(name):
    """The fixtures the CUDA path is held to were made with the TensorFlow half of RecSimBase.__init__ bypassed.  Here the
    reference builds ITSELF -- RecEnvBase -> (Seq)SlateRecEnv.__init__ -> RecSimBase.__init__ -> rl4rs/nets/dien.py ->
    tf.train.Saver().restore of a checkpoint written by our n1 writer -> keras.backend.function -> obs_fn / forward --
    over the layer stand-ins, replays the fixture's actions, and must land on the fixture: integers exactly, observations
    and rewards at f32 rounding (the stand-ins compute in f64 and hand back float32 like keras.backend.function).  What
    that stack recorded is stored in tests/golden/reference/records.npz (tests/golden/make_reference_golden.py)."""
    from golden_util import Golden
    g = Golden(name)
    check_fingerprint(g.arr, load_fingerprint(RECORDS, "fixture_stack/" + name), rtol=3e-5, what=name + " (full stack)")


@pytest.mark.parametrize("algo,seq", [("dnn", False), ("widedeep", True), ("lstm", False)])
def test_the_references_own_stack_with_the_other_simulators(algo, seq):
    """config['algo'] dispatch (slate.py:239-242) through the reference's own constructors for the other three graphs of
    rl4rs/nets/: a short logged-policy episode of the self-constructed reference env against the oracle env the GPU tests
    use for that simulator (tests/test_gpu_dnn.py).  What the reference recorded is stored in
    tests/golden/reference/records.npz (tests/golden/make_reference_golden.py)."""
    from oracle.env_np import OracleEnv
    from rl4rs_b200.utils.datautil import FeatureUtil
    from test_oracle_vs_reference_random import roll_oracle
    cfg, cat, records, w = other_simulator_inputs(algo, seq)
    ora = OracleEnv(cfg, FeatureUtil.parse_log(records, 64), cat, ORACLES[algo](w, np.float32), seq=seq)
    rec = roll_oracle(ora, cfg, lambda env, ep, t, off: off, 1)
    check_fingerprint(rec, load_fingerprint(RECORDS, "simulator/" + algo), rtol=3e-5, what="%s simulator" % algo)
    assert rec["step_obs"].shape[-1] == (3072 if algo == "widedeep" else 256) and (rec["reward"] > 0).any()


def other_simulator_inputs(algo, seq):
    """(cfg, catalog, log records, weights) of the short logged-policy episode for simulator `algo`."""
    import make_golden
    from rl4rs_b200 import synth
    B = 4
    cfg = dict(make_golden.BASE_CFG, batch_size=B, cache_size=B, is_eval=True, support_rllib_mask=True, algo=algo,
               category_hash_size=600, max_steps=27 if seq else 9)
    cat = synth.make_catalog()
    log = synth.make_log(12, pages=4 if seq else 1, catalog=cat, hash_size=600, keep_hist=True)
    records = synth.render_records(log, cat)
    maker = {"dnn": synth.make_dnn_weights, "widedeep": synth.make_widedeep_weights, "lstm": synth.make_lstm_weights}[algo]
    return cfg, cat, records, maker(cfg, stress=2.0, bias_noise=0.2)


def test_rllib_policy_models_of_the_reference_against_the_torch_twins():
    """a22 / n4: rl4rs/nets/rllib/rllib_rawstate_model.py's TFModelWithRawState (its own Keras graph over nets/utils.py)
    and rllib_mask_model.py's MyMaskActionsModel.forward (the action masking), run from the reference tree over the
    stand-ins, against rl4rs_b200/policy.py -- the twins the kernels k_policy_act / k_policy_grad are themselves held to.
    What the reference's models returned is stored in tests/golden/reference/records.npz
    (tests/golden/make_reference_golden.py)."""
    c = rllib_case()
    z = np.load(RECORDS)
    out = {k[len("rllib/"):]: z[k] for k in z.files if k.startswith("rllib/")}
    scopes = [str(x) for x in out["scopes"]]
    assert not out["unused"].size
    assert [s_ for i, s_ in enumerate(scopes) if i == 0 or s_ != scopes[i - 1]] == \
        ["embedding", "dense", "dense_1", "embedding_1", "dense_2", "fc_out", "value_out"]       # Keras creation order
    np.testing.assert_allclose(out["logits"], c["logits"].numpy(), rtol=0, atol=2e-5)
    np.testing.assert_allclose(out["value"], c["value"].numpy(), rtol=0, atol=2e-5)
    # the masking itself, by the reference's forward(): fed the twin's unmasked logits as the action_embed_model output
    np.testing.assert_array_equal(out["masked"], c["masked"].numpy())
    # and for the 256-d observation policy of the benchmark configs
    got = out["masked256"]
    np.testing.assert_array_equal(got, c["want256"].numpy())
    assert (got[c["mask"] == 0] < -1e38).all()


def rllib_case():
    """The raw-state policy twin with perturbed weights, its checkpoint under the reference model's scope names, six
    random raw-state rows and action masks, and what the twins compute on them."""
    import torch
    from rl4rs_b200.policy import MaskedPolicy, RawStatePolicy
    cfg = {"category_hash_size": 600, "emb_size": 128, "hidden_units": 128, "category_feature_num": 21,
           "dense_feature_num": 432, "seq_num": 2, "maxlen": 64, "batch_size": 6}
    rs = np.random.RandomState(0)
    R, A = 6, 284
    mask = (rs.rand(R, A) < 0.4).astype(np.float32)
    mask[:, 7] = 1.0
    # raw-state policy: embeddings -> pools -> dense tower -> context 256 -> logits / value
    pol = RawStatePolicy(A, "cpu", seed=3, config=cfg)
    with torch.no_grad():
        pol.flat.add_(0.05 * torch.randn(pol.flat.shape, generator=torch.Generator().manual_seed(1)))
    p = {k: v.detach().numpy() for k, v in pol.params().items()}
    ck = {"embedding/embeddings": p["emb_cat"], "dense/kernel": p["dw1"], "dense/bias": p["db1"], "dense_1/kernel": p["dw2"],
          "dense_1/bias": p["db2"], "embedding_1/embeddings": p["emb_seq"], "dense_2/kernel": p["wc"], "dense_2/bias": p["bc"],
          "fc_out/kernel": p["w2"], "fc_out/bias": p["b2"], "value_out/kernel": p["wv"], "value_out/bias": p["bv"]}
    cat, dense, seq = rs.randint(0, 600, (R, 21)), rs.normal(0, 2, (R, 432)).astype(np.float32), rs.randint(0, 284, (R, 2, 64))
    obs = pol.pack({"category_feature": torch.as_tensor(cat), "dense_feature": torch.as_tensor(dense), "sequence_feature": torch.as_tensor(seq)})
    with torch.no_grad():
        logits, value = pol.forward(obs, torch.ones(R, A))
        masked, _ = pol.forward(obs, torch.as_tensor(mask))
    mp = MaskedPolicy(A, "cpu", seed=5)
    o256 = torch.as_tensor(rs.normal(0, 1, (R, 256)).astype(np.float32))
    with torch.no_grad():
        raw, _ = mp.forward(o256, torch.ones(R, A))
        want256, _ = mp.forward(o256, torch.as_tensor(mask))
    return {"cfg": cfg, "A": A, "mask": mask, "ck": ck, "cat": cat, "dense": dense, "seq": seq, "obs": obs,
            "logits": logits, "value": value, "masked": masked, "o256": o256, "raw": raw, "want256": want256}
