"""Generates tests/golden/reference/: what the REFERENCE'S OWN code returns for the inputs of the tests that compare the
project with it, so that those tests run without the reference tree.

    RL4RS_REFERENCE_ROOT=/path/to/RL4RS python tests/golden/make_reference_golden.py

records.npz        compact records (golden_util.fingerprint) of reference rollouts: the 32 random scenarios of
                   tests/test_oracle_vs_reference_random.py, the dnn / widedeep / lstm simulators and the ten fixtures
                   replayed by the reference's full stack (tests/test_reference_graph.py); the reference's RLlib policy
                   model outputs
expected.json      what the reference returned to the smaller checks (gym layer, ingest CLI, trainer hyper-parameters,
                   static helpers, feature extraction, the graph vectors' checkpoints), as digests where it is large
item_info.csv.gz   the reference's dataset/item_info.csv, the input of the static-helper test

Before writing, every comparison the tests make is made here against the live reference too.
"""
import ast
import gzip
import json
import os
import runpy
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS, HERE]

import make_golden                                                      # noqa: E402
import make_nets_golden as mk                                           # noqa: E402
import test_env_base_cpu as envt                                        # noqa: E402
import test_oracle_vs_reference_random as rnd                           # noqa: E402
import test_reference_graph as graph                                    # noqa: E402
from golden_util import REFERENCE_DIR, Golden, digest, fingerprint, golden_names, save_fingerprints   # noqa: E402
from oracle import ref_harness                                          # noqa: E402
from oracle import tf_eager_stub as stub                                # noqa: E402
from oracle.dnn_np import DnnOracle                                     # noqa: E402


def records():
    fps = {}
    for seed in range(32):
        cfg, seq, recs, cat, w, episodes, aseed, np_seed = rnd.scenario(seed)
        rec = make_golden.run_reference(dict(cfg), recs, cat.to_text(), w, seq, rnd.action_source(cfg, aseed),
                                        n_episodes=episodes, seed=np_seed, net=DnnOracle(w, np.float32))
        fps["random/%d" % seed] = fingerprint(rec, seed=seed)
    for algo, seq in (("dnn", False), ("widedeep", True), ("lstm", False)):
        cfg, cat, recs, w = graph.other_simulator_inputs(algo, seq)
        rec = make_golden.run_reference(cfg, recs, cat.to_text(), w, seq, lambda env, ep, t, off: off, full_stack=True)
        fps["simulator/" + algo] = fingerprint(rec)
    for name in golden_names():
        g = Golden(name)
        T = g.config["max_steps"]
        replay = lambda env, ep, t, off, a=g.arr: a["action_in"][ep * T + t]
        rec = make_golden.run_reference(g.config, g.meta["records"], g.meta["catalog_text"], g.weights, g.seq, replay,
                                        n_episodes=g.n_episodes, seed=g.meta.get("np_seed"), full_stack=True)
        fps["fixture_stack/" + name] = fingerprint(rec)
    return fps


def rllib_outputs():
    c = graph.rllib_case()
    out = stub.run_reference_rawstate_model(c["cfg"], c["ck"], c["cat"].astype(np.float32), c["dense"],
                                            c["seq"].astype(np.float32), c["A"])
    masked = stub.run_reference_mask_forward(lambda o: c["logits"].numpy(), c["obs"].numpy(), c["mask"], c["A"])
    masked256 = stub.run_reference_mask_forward(lambda o: c["raw"].numpy(), c["o256"].numpy(), c["mask"], c["A"])
    return {"rllib/scopes": np.array([v[0] for v in out["variables"]]), "rllib/unused": np.array(sorted(out["unused"])),
            "rllib/logits": np.asarray(out["logits"]), "rllib/value": np.asarray(out["value"]),
            "rllib/masked": np.asarray(masked), "rllib/masked256": np.asarray(masked256)}


def env_layer():
    ref_base = ref_harness.install_stubs()[0]
    out = {}
    for name in sorted(envt.CONFIGS):
        for batch in (1, 3):
            config = dict(envt.CONFIGS[name], batch_size=batch, action_size=envt.A)
            ref = envt.drive(ref_base.RecEnvBase, config)
            assert ref == envt.drive(envt.RecEnvBase, config), (name, batch)
            out["%s/%d" % (name, batch)] = envt.seen_digest(ref)
    return out


def ingest():
    from rl4rs_b200.utils import ingest as ours
    ref_harness.install_stubs()
    script = os.path.join(ref_harness.REFERENCE_ROOT, "script", "data_preprocess.py")
    tmp = tempfile.mkdtemp()

    def run_stage(stage, lines):
        src, dst = os.path.join(tmp, "in.csv"), os.path.join(tmp, "out_%s.csv" % stage)
        open(src, "w").write("\n".join(lines))
        argv, sys.argv = sys.argv, [script, src, dst, stage]
        try:
            runpy.run_path(script, run_name="__main__")
        finally:
            sys.argv = argv
        return [x for x in open(dst).read().split("\n") if x]

    out = {}
    for seed in range(8):
        _, ragged = rnd.ragged_sessions(seed)
        np.random.seed(40 + seed)
        aug = run_stage("data_augment", ragged)
        traj = run_stage("slate2trajectory", rnd.augmented_table(aug))
        np.random.seed(40 + seed)
        assert ours.data_augment(ragged) == aug and ours.slate2trajectory(rnd.augmented_table(aug)) == traj, seed
        out[str(seed)] = {"augment": rnd.digest_lines(aug), "augment_lines": len(aug),
                          "trajectory": rnd.digest_lines(traj), "trajectory_lines": len(traj)}
    return out


def trainer_defaults():
    src = open(os.path.join(ref_harness.REFERENCE_ROOT, "script", "modelfree_train.py")).read()
    tree = ast.parse(src)

    def literal(node):
        """A dict literal with non-literal values (config[...] expressions) left out."""
        out = {}
        for k, v in zip(node.keys, node.values):
            if k is None:
                continue
            try:
                out[ast.literal_eval(k)] = ast.literal_eval(v)
            except Exception:
                pass
        return out

    branches = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.If) and isinstance(node.test, ast.Compare) and isinstance(node.test.left, ast.Constant) \
                and node.test.left.value in ("PPO", "A2C"):
            first = node.body[0]
            assert isinstance(first, ast.Assign) and first.targets[0].id == "cfg"
            branches[node.test.left.value] = literal(first.value)
    common = [literal(n) for n in ast.walk(tree) if isinstance(n, ast.Dict)]
    common = [d for d in common if d.get("batch_mode") == "complete_episodes"]
    return {"branches": branches, "common": common, "softq_exploration": '"type": "SoftQ"' in src}


def static_helpers():
    from rl4rs_b200.env.slate import SlateState
    ref_slate = ref_harness.install_stubs()[1]
    item_file = os.path.join(ref_harness.REFERENCE_ROOT, "dataset", "item_info.csv")
    info_r, emb_r = ref_slate.SlateState.get_iteminfo_from_file(item_file, 284)
    loc_r, sp_r = ref_slate.SlateState.get_mask_from_file(item_file, 284)
    info_o, emb_o = SlateState.get_iteminfo_from_file(item_file, 284)
    assert rnd.item_table_digest(info_o) == rnd.item_table_digest(info_r) and digest(emb_o) == digest(emb_r)
    near, near_masked = [], []
    for q, mask in rnd.knn_queries(emb_r):
        near.append([int(x) for x in ref_slate.SlateState.get_nearest_neighbor(q, emb_r)])
        near_masked.append([int(x) for x in ref_slate.SlateState.get_nearest_neighbor_with_mask(q, emb_r, mask)])
    with open(item_file, "rb") as f:
        data = f.read()
    with gzip.GzipFile(os.path.join(REFERENCE_DIR, "item_info.csv.gz"), "wb", compresslevel=9, mtime=0) as f:
        f.write(data)
    return {"action_emb": digest(emb_r), "item_ids": sorted(map(str, info_r)), "item_table": rnd.item_table_digest(info_r),
            "location_mask": digest(loc_r), "special_items": [int(x) for x in sp_r], "nearest": near,
            "nearest_with_mask": near_masked}


def feature_extraction():
    ref = ref_harness.install_stubs()[3].FeatureUtil(rnd.FEATURE_CFG)
    return [rnd.extracted(ref.feature_extraction(rows)) for rows in rnd.ragged_state_rows()]


def nets():
    g = np.load(os.path.join(HERE, "nets", "reference_graph.npz"))
    meta = json.loads(str(g["meta"]))
    out = {"checkpoints": {}}
    for case in sorted(mk.CASES):
        _, ck = mk.checkpoint_of(case)
        r = stub.run_reference_graph(mk.CASES[case][0], mk.NETS_CONFIG, ck, g["seq"].astype(np.float32), g["dense"], g["cat"])
        np.testing.assert_allclose(r["obs"], g[case + "_obs"], rtol=0, atol=1e-13 * max(1.0, np.abs(r["obs"]).max()))
        assert [[s, n, list(sh)] for s, n, sh in r["variables"]] == meta[case]["variables"]
        assert r["layers"] == meta[case]["layers"]
        out["checkpoints"][case] = {name: digest(v) for name, v in ck.items()}
    from rl4rs_b200.utils import tf_checkpoint as tfc
    w, _ = mk.checkpoint_of("dien_stress")
    rd = tfc.TensorBundleReader(tfc.save_dien_checkpoint(os.path.join(tempfile.mkdtemp(), "sim"), w, mk.SMALL))
    ck = {name: rd.get_tensor(name) for name in rd.variables()}
    r = stub.run_reference_graph("dien", mk.NETS_CONFIG, ck, g["seq"].astype(np.float32), g["dense"], g["cat"])
    assert not r["unused"]
    np.testing.assert_array_equal(r["obs"], g["dien_stress_obs"])
    out["checkpoint_file_tensors"] = {name: digest(v) for name, v in ck.items()}
    return out


def main():
    assert ref_harness.reference_available(), "needs the reference tree (RL4RS_REFERENCE_ROOT)"
    os.makedirs(REFERENCE_DIR, exist_ok=True)
    expected = {"env_layer": env_layer(), "ingest": ingest(), "trainer_defaults": trainer_defaults(),
                "static_helpers": static_helpers(), "feature_extraction": feature_extraction(), "nets": nets()}
    with open(os.path.join(REFERENCE_DIR, "expected.json"), "w") as f:
        json.dump(expected, f, indent=0, sort_keys=True)
    fps = records()
    path = os.path.join(REFERENCE_DIR, "records.npz")
    save_fingerprints(path, fps)
    z = dict(np.load(path))
    np.savez_compressed(path, **z, **rllib_outputs())
    for name in sorted(os.listdir(REFERENCE_DIR)):
        print("%-20s %7.1f KB" % (name, os.path.getsize(os.path.join(REFERENCE_DIR, name)) / 1024.0))


if __name__ == "__main__":
    main()
