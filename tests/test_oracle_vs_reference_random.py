"""CPU: the oracle env (oracle/env_np.py) and the product's host layer against what the reference's OWN code computed on
RANDOM scenarios -- env kind, episode length, mask mode, continuous / one-hot actions, raw-state observations, sampling
mode, batch size, and per-step actions (logged, random, repeated, out-of-layer) are drawn from a seed.  The reference was
rolled through oracle/ref_harness.py exactly like the committed fixtures were, and its results are stored under
tests/golden/reference/ (tests/golden/make_reference_golden.py): everything it exposes per step must equal what the
oracle computes (integers and feature rows bit-exact).  The ten committed fixtures pin ten hand-picked corners; this
sweeps the product of the flags."""
import gzip
import json
import os
import shutil
import sys

import numpy as np
import pytest

from golden_util import REFERENCE_DIR, check_fingerprint, digest, load_fingerprint
from oracle.dnn_np import DnnOracle
from oracle.env_np import OracleEnv
from rl4rs_b200 import synth
from rl4rs_b200.utils.datautil import FeatureUtil

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))

RECORDS = os.path.join(REFERENCE_DIR, "records.npz")


def expected(section):
    with open(os.path.join(REFERENCE_DIR, "expected.json")) as f:
        return json.load(f)[section]


def draw_scenario(seed):
    rs = np.random.RandomState(1000 + seed)
    seq = bool(rs.rand() < 0.5)
    B = int(rs.randint(2, 7))
    cfg = {"epoch": 1, "maxlen": 64, "action_size": 284, "class_num": 2, "dense_feature_num": 432,
           "category_feature_num": 21, "category_hash_size": 5000, "seq_num": 2, "emb_size": 128, "page_items": 9,
           "hidden_units": 128, "action_emb_size": 32, "batch_size": B, "algo": "dnn",     # the cheap network: the env half is under test
           "max_steps": int(rs.choice([9, 18, 27, 36])) if seq else 9}
    mode = rs.choice(["plain", "rllib", "d3rl", "both"])
    if mode in ("rllib", "both"):
        cfg["support_rllib_mask"] = True
    if mode in ("d3rl", "both"):
        cfg["support_d3rl_mask"] = True
    if rs.rand() < 0.35:
        cfg["support_conti_env"] = True
        if rs.rand() < 0.3:
            cfg["support_onehot_action"] = True
    if rs.rand() < 0.25:
        cfg["rawstate_as_obs"] = True
    if rs.rand() < 0.4:
        cfg["simulator_info_fetch"] = True
    train_mode = bool(rs.rand() < 0.4)
    cfg["is_eval"] = not train_mode
    cfg["cache_size"] = int(rs.randint(B, 3 * B + 1)) if train_mode else B
    n_rows = int(rs.randint(cfg["cache_size"], 3 * cfg["cache_size"] + 2))     # small logs wrap around (base.py:85-88)
    episodes = int(rs.randint(1, 4))
    return cfg, seq, n_rows, episodes, int(rs.randint(1 << 30)), train_mode


def action_source(cfg, seed):
    rs = np.random.RandomState(seed)
    B = cfg["batch_size"]
    emb = cfg["action_size"] if cfg.get("support_onehot_action") else 32

    def pick(env, ep, t, off):
        if cfg.get("support_conti_env"):
            a = rs.uniform(-1, 1, (B, emb))
            a[rs.rand(B) < 0.15] = 0.0                              # all-zero rows: every score ties
            keep = rs.rand(B) < 0.3
            a[keep] = np.asarray(off, dtype=np.float64)[keep]       # the logged item's own embedding
            return a
        off = np.asarray(off)
        r = rs.rand(B)
        rand = rs.randint(0, cfg["action_size"], B)                 # often outside the layer, or a repeat
        prev = env.samples.prev_actions[:, max(t - 1, 0)]
        return np.where(r < 0.6, off, np.where(r < 0.85, rand, prev)).astype(np.int64)
    return pick


def scenario(seed):
    """The inputs of random scenario `seed`: (cfg, seq, records, catalog, weights, episodes, action seed, numpy seed)."""
    cfg, seq, n_rows, episodes, aseed, train_mode = draw_scenario(seed)
    cat = synth.make_catalog()
    log = synth.make_log(n_rows, pages=4 if seq else 1, catalog=cat, hash_size=5000, corrupt_frac=0.25, keep_hist=True,
                         seed=synth.LOG_SEED + seed)
    records = synth.render_records(log, cat)
    w = synth.make_dnn_weights(cfg, stress=2.0, bias_noise=0.2)
    return cfg, seq, records, cat, w, episodes, aseed, (77 + seed if train_mode else None)


def roll_oracle(env, cfg, actions_fn, n_episodes):
    """Everything the oracle env exposes per step, recorded like make_golden.run_reference records the reference env
    (which hands out click_p at the end of a Slate episode only)."""
    rec = {}

    def put(key, val):
        rec.setdefault(key, []).append(np.asarray(val))

    for ep in range(n_episodes):
        for k, v in env.reset().items():
            put("reset_" + k, v)
        put("reset_user", np.asarray([int(u) for u in env.samples.user], dtype=np.int64))
        for t in range(cfg["max_steps"]):
            off_a = np.asarray(env.offline_action)
            put("offline_action", off_a)
            a = actions_fn(env, ep, t, off_a)
            put("action_in", np.asarray(a))
            obs, reward, done, info = env.step(a)
            seqs, dense, cat = env.samples.features()
            assert dense.dtype == np.float32 and cat.dtype == np.int32 and seqs.dtype == np.int32
            put("seq", seqs); put("dense", dense); put("cat", cat)
            for k, v in obs.items():
                put("step_" + k, v)
            put("reward", np.asarray(reward, dtype=np.float64))
            put("done", np.asarray(done, dtype=np.int64))
            put("offline_reward", np.asarray(env.offline_reward, dtype=np.float64))
            put("prev_actions", env.samples.prev_actions.copy())
            put("violation", env.samples.get_violation())
            if cfg.get("simulator_info_fetch") and t == cfg["max_steps"] - 1 and not env.seq:
                put("click_p", np.stack([i["click_p"] for i in info]))     # the reference's SeqSlateRecEnv has none
    return {k: np.stack(v) for k, v in rec.items()}


@pytest.mark.parametrize("seed", range(32))
def test_oracle_env_equals_the_reference_env_on_a_random_scenario(seed):
    cfg, seq, records, cat, w, episodes, aseed, np_seed = scenario(seed)
    if np_seed is not None:
        np.random.seed(np_seed)
    env = OracleEnv(dict(cfg), FeatureUtil.parse_log(records, 64), cat, DnnOracle(w, np.float32), seq=seq)
    rec = roll_oracle(env, cfg, action_source(cfg, aseed), episodes)
    check_fingerprint(rec, load_fingerprint(RECORDS, "random/%d" % seed), what="random scenario %d" % seed)
    # ... and the product's own env classes (gym layer, sampler, obs / reward formatting) over the engine stand-in
    import rl4rs_b200.engine as engine_mod
    from oracle_engine import OracleEngine
    from test_host_layer_cpu import make_env, replay_through_host_layer
    real = engine_mod.Engine
    engine_mod.Engine = OracleEngine
    try:
        fmt = ("list", "numpy", "torch")[seed % 3]
        if np_seed is not None:
            np.random.seed(np_seed)
        host_env = make_env(dict(cfg), seq, cat, FeatureUtil.parse_log(records, 64), w, output_format=fmt)
        replay_through_host_layer(host_env, cfg, rec, episodes, "random scenario %d (host layer, %s)" % (seed, fmt), fmt)
    finally:
        engine_mod.Engine = real


INGEST_HEADER = ("timestamp@session_id@sequence_id@exposed_items@user_feedback@user_seqfeature@user_protrait@item_feature"
                 "@behavior_policy_id")


def ragged_sessions(seed):
    """A session table of 3-9 sessions with 1-4 surviving pages each, header first, newline-terminated."""
    rs = np.random.RandomState(500 + seed)
    n_sess = int(rs.randint(3, 10))
    cat = synth.make_catalog()
    recs = synth.render_records(synth.make_log(4 * n_sess, pages=1, catalog=cat, keep_hist=True, seed=900 + seed), cat)
    ragged = [INGEST_HEADER]
    for s in range(n_sess):
        base = recs[4 * s].split("@")
        for p in range(int(rs.randint(1, 5))):               # 1..4 pages of this session survive
            f = recs[4 * s + p].split("@")
            ragged.append("@".join([str(1000 * s + p), base[1], str(p + 1), f[3], f[4], base[5], base[6], f[7], base[8]]))
    ragged.append("")
    return n_sess, ragged


def augmented_table(aug):
    """The slate2trajectory input made of a data_augment output."""
    return [INGEST_HEADER] + aug[1:] + [""] if aug[0] == INGEST_HEADER else [INGEST_HEADER] + aug + [""]


@pytest.mark.parametrize("seed", range(8))
def test_ingest_equals_the_reference_preprocessing_on_random_sessions(seed):
    """n3: rl4rs_b200/utils/ingest.py against what the reference's own script/data_preprocess.py (run as its own CLI, like
    tests/golden/make_ingest_golden.py does) wrote for random session tables: `data_augment` pads sessions of 1-4 pages
    to 4 with the GLOBAL numpy RNG, `slate2trajectory` joins 4-page sessions and drops the last one."""
    from rl4rs_b200.utils import ingest
    want = expected("ingest")[str(seed)]
    n_sess, ragged = ragged_sessions(seed)
    np.random.seed(40 + seed)
    got_aug = ingest.data_augment(ragged)
    assert len(got_aug) == want["augment_lines"] and digest_lines(got_aug) == want["augment"]
    got_traj = ingest.slate2trajectory(augmented_table(got_aug))
    assert len(got_traj) == want["trajectory_lines"] and digest_lines(got_traj) == want["trajectory"]
    assert 1 <= len(got_traj) < n_sess                       # the script drops the last session (and any it merges)


def digest_lines(lines):
    return digest(np.frombuffer("\n".join(lines).encode(), dtype=np.uint8))


def test_trainer_defaults_are_the_reference_scripts_hyper_parameters():
    """a23: the RLlib config dicts of script/modelfree_train.py (PPO :179-217, A2C :248-268, common :390-415), as read
    out of the script's own source with `ast` (the literal entries; tests/golden/make_reference_golden.py), against the
    defaults rl4rs_b200/trainer.py trains with."""
    from rl4rs_b200 import trainer
    ref = expected("trainer_defaults")
    branches = ref["branches"]
    assert set(branches) == {"PPO", "A2C"}
    for algo, ours in (("PPO", trainer.PPO_DEFAULTS), ("A2C", trainer.A2C_DEFAULTS)):
        shared = sorted(set(branches[algo]) & set(ours))
        assert len(shared) >= 5, shared
        for k in shared:
            assert ours[k] == branches[algo][k], (algo, k, ours[k], branches[algo][k])
    assert trainer.PPO_DEFAULTS["grad_clip"] is None and "grad_clip" not in branches["PPO"]       # commented out there
    # the dict every algorithm is merged into: gamma 1, SoftQ exploration, complete episodes
    common = ref["common"]
    assert len(common) == 1 and common[0]["gamma"] == 1 and common[0]["explore"] is True
    assert trainer.PPO_DEFAULTS["gamma"] == trainer.A2C_DEFAULTS["gamma"] == 1.0
    assert ref["softq_exploration"]


def knn_queries(emb):
    """Twenty random nearest-neighbour queries (incl. all-tie and fully masked rows) over the 284 x 32 embeddings."""
    rs = np.random.RandomState(4)
    for trial in range(20):
        q = rs.uniform(-1, 1, (16, 32))
        q[0] = 0.0                                            # every score ties at 0: lowest index wins
        q[1] = emb[1 + trial]                                 # an item's own embedding
        mask = (rs.rand(16, 284) < 0.3).astype(np.int64)
        mask[2] = 0                                           # nothing allowed: all scores -2**31, index 0
        yield q, mask


def item_table_digest(info):
    return digest([[k, info[k]["price"], info[k]["location"]] + list(np.asarray(info[k]["item_vec"], float))
                   for k in sorted(info)])


def test_static_helpers_on_the_real_catalog_and_random_knn_queries(tmp_path):
    """slate.py:28-65,180-191: the item table, action embeddings, location mask and special items read from the
    reference's own dataset/item_info.csv (stored as tests/golden/reference/item_info.csv.gz), and the two
    nearest-neighbour statics on random queries (incl. ties and fully masked rows), mirror class against what the
    reference class returned."""
    from rl4rs_b200.env.slate import SlateState
    ref = expected("static_helpers")
    item_file = str(tmp_path / "item_info.csv")
    with gzip.open(os.path.join(REFERENCE_DIR, "item_info.csv.gz"), "rb") as src, open(item_file, "wb") as dst:
        shutil.copyfileobj(src, dst)
    info_o, emb_o = SlateState.get_iteminfo_from_file(item_file, 284)
    assert digest(emb_o) == ref["action_emb"]
    assert sorted(map(str, info_o)) == sorted(ref["item_ids"]) and item_table_digest(info_o) == ref["item_table"]
    loc_o, sp_o = SlateState.get_mask_from_file(item_file, 284)
    assert digest(loc_o) == ref["location_mask"]
    assert [int(x) for x in sp_o] == ref["special_items"] and len(sp_o) > 0
    for (q, mask), want, want_masked in zip(knn_queries(emb_o), ref["nearest"], ref["nearest_with_mask"]):
        np.testing.assert_array_equal(SlateState.get_nearest_neighbor(q, emb_o), want)
        np.testing.assert_array_equal(SlateState.get_nearest_neighbor_with_mask(q, emb_o, mask), want_masked)


FEATURE_CFG = {"maxlen": 64, "batch_size": 5, "class_num": 2, "dense_feature_num": 432, "category_feature_num": 21,
               "category_hash_size": 100000, "seq_num": 2}


def ragged_state_rows():
    """Twelve batches of five raw state rows with empty / short / over-long sequences, short and over-long dense and
    category lists."""
    rs = np.random.RandomState(8)
    for trial in range(12):
        rows = []
        for i in range(5):
            seqs = [list(rs.randint(1, 284, rs.choice([0, 1, 7, 64, 65, 130]))) for _ in range(2)]
            dense = list(rs.normal(0, 1, rs.choice([32, 72, 432, 440])).astype(np.float64))
            cat = list(rs.randint(0, 100000, rs.choice([10, 12, 21, 25])).astype(np.float64))       # floats in the reference too
            rows.append([0, seqs, dense, cat, [0] * 9, int(rs.randint(2))])
        yield rows


def extracted(out):
    (s, d, c, l), y = out
    return {"seq": digest(s), "dense": digest(d), "cat": digest(c), "len": digest(l), "label": [int(v) for v in y],
            "dense_dtype": str(d.dtype), "cat_dtype": str(c.dtype)}


def test_feature_extraction_mirror_on_random_ragged_rows():
    """datautil.py:34-69: FeatureUtil.feature_extraction, host mirror against what the reference method returned, on raw
    state rows with empty / short / over-long sequences, short and over-long dense and category lists."""
    ours = FeatureUtil(FEATURE_CFG)
    want = expected("feature_extraction")
    for trial, rows in enumerate(ragged_state_rows()):
        out = ours.feature_extraction(rows)
        assert extracted(out) == want[trial], trial
        assert out[0][0].shape == (5, 2, 64)
