"""GPU parity in the regimes the benchmark runs in (round-1 verdict, "parity first"):

* the DEFAULT weight set of bench.py (``synth.make_weights(cfg)``: Keras/TF1 initialisers, raw unbounded DIN scores,
  zero biases, category_hash_size 100 000) on DISTINCT synthetic rows -- Slate, SeqSlate-27 and continuous-kNN at B=48;
* full-size batches (4096 and 8192 rows per GPU, the BASELINE configs[1] / north-star per-GPU sizes): a 128-row oracle
  sample of the big env, rows compared by index;
* every AUGRU kernel forced in turn (``r4_set_option('augru_kernel', ...)``): the simulator alone and env fixtures
  through the pair kernel (one recurrence per CTA pair) and the ping-pong kernel (two per pair), plus a launch big
  enough for the natural rule;
* the chunked sequence-cache build (> 8192 sequences) and the multi-wave persistent GEMM (tiles > SMs).

Oracle = oracle/env_np.py + oracle/dien_np.py (f32), reference lines: rl4rs/nets/utils.py:117-125,
rl4rs/env/slate.py:281-308, rl4rs/env/seqslate.py:136-160.  Bar: integers bit-exact, floats 1e-4 (golden_util).
"""
import numpy as np
import pytest

from golden_util import Golden, assert_close_rel
from test_gpu_parity import make_env

pytestmark = pytest.mark.gpu


def _cfg(B, seq, **flags):
    cfg = {"maxlen": 64, "batch_size": B, "action_size": 284, "class_num": 2, "dense_feature_num": 432,
           "category_feature_num": 21, "category_hash_size": 100000, "seq_num": 2, "emb_size": 128,
           "hidden_units": 128, "max_steps": 27 if seq else 9, "page_items": 9, "action_emb_size": 32,
           "is_eval": True, "cache_size": B}
    cfg.update(flags)
    return cfg


def _default_regime(B, seq, n_log=None, **flags):
    """bench.py's regime: default glorot weights (seed 4321), hash 100 000, synthetic log (seed 1234)."""
    from rl4rs_b200 import synth
    cfg = _cfg(B, seq, **flags)
    cat = synth.make_catalog()
    log = synth.make_log(n_log or 4 * B, pages=4 if seq else 1, catalog=cat, hash_size=100000, corrupt_frac=0.1)
    return cfg, cat, log, synth.make_weights(cfg)


@pytest.fixture
def augru_option():
    """Force an AUGRU kernel for one test, back to the rule afterwards."""
    from rl4rs_b200 import _capi

    def force(mode):
        _capi.set_option("augru_kernel", {"auto": 0, "pair": 2, "pp": 3}[mode])
    yield force
    _capi.set_option("augru_kernel", 0)


def _sublog(log, idx):
    from rl4rs_b200.synth import LogSoA
    return LogSoA(**{k: np.ascontiguousarray(getattr(log, k)[idx]) for k in LogSoA.FIELDS})


@pytest.mark.parametrize("kind", ["slate", "seqslate27", "conti"])
def test_default_weights_env_matches_oracle(kind):
    """B=48 distinct rows, the benchmark's weight regime; policy = logged actions with 20 % random replacements
    (discrete) or random / logged embeddings (continuous kNN)."""
    from oracle.dien_np import DienOracle
    from oracle.env_np import OracleEnv
    seq, conti = kind == "seqslate27", kind == "conti"
    B = 48
    cfg, cat, log, w = _default_regime(B, seq, support_rllib_mask=True, simulator_info_fetch=True,
                                       **({"support_conti_env": True} if conti else {}))
    env = make_env(cfg, seq, cat, log, w, output_format="numpy")
    ref = OracleEnv(cfg, log, cat, DienOracle(w, np.float32), seq=seq)
    rs = np.random.RandomState(11)
    o, r = env.reset(), ref.reset()
    assert_close_rel(o["obs"], r["obs"], what="default-weights %s reset obs" % kind)
    np.testing.assert_array_equal(o["action_mask"], r["action_mask"])
    paid = 0
    for t in range(cfg["max_steps"]):
        if conti:
            a = rs.uniform(-1, 1, (B, 32))
            a[:8] = ref.offline_action[:8]
        else:
            a = np.where(rs.rand(B) < 0.8, ref.offline_action, rs.randint(0, 284, B))
        o, rew, done, info = env.step(a)
        r, rrew, rdone, _ = ref.step(a)
        np.testing.assert_array_equal(env.samples.prev_actions, ref.samples.prev_actions, err_msg="prev_actions %d" % t)
        np.testing.assert_array_equal(o["action_mask"], r["action_mask"], err_msg="mask %d" % t)
        np.testing.assert_array_equal(done, rdone)
        np.testing.assert_array_equal(env.samples.get_violation(), ref.samples.get_violation())
        assert_close_rel(o["obs"], r["obs"], what="default-weights %s obs step %d" % (kind, t))
        assert_close_rel(rew, rrew, what="default-weights %s reward step %d" % (kind, t))
        paid += int((np.asarray(rrew) != 0).any())
    assert paid >= (3 if seq else 1)


@pytest.mark.parametrize("B", [4096, 8192])
def test_big_batch_oracle_sample(B):
    """Full-size env (default weights), 128 of its rows replayed through the oracle: obs / mask / reward / violation of
    those rows, every step.  At B=4096 the observation passes run the pair kernel and the 36 864-row reward pass
    whatever the rule picks; at B=8192 every pass is multi-wave."""
    from oracle.dien_np import DienOracle
    from oracle.env_np import OracleEnv
    cfg, cat, log, w = _default_regime(B, False, n_log=B, support_rllib_mask=True)
    env = make_env(cfg, False, cat, log, w, output_format="numpy")
    rs = np.random.RandomState(B)
    idx = np.sort(rs.choice(B, 128, replace=False))
    idx[0], idx[-1] = 0, B - 1
    scfg = dict(cfg, batch_size=128, cache_size=128)
    ref = OracleEnv(scfg, _sublog(log, idx), cat, DienOracle(w, np.float32))
    o, r = env.reset(reset_file=True), ref.reset(reset_file=True)
    assert_close_rel(o["obs"][idx], r["obs"], what="B=%d sample reset obs" % B)
    for t in range(9):
        a = np.asarray(env.offline_action)
        np.testing.assert_array_equal(a[idx], ref.offline_action)
        a = np.where(rs.rand(B) < 0.85, a, rs.randint(0, 284, B))
        o, rew, done, _ = env.step(a)
        r, rrew, rdone, _ = ref.step(a[idx])
        np.testing.assert_array_equal(o["action_mask"][idx], r["action_mask"], err_msg="mask %d" % t)
        assert_close_rel(o["obs"][idx], r["obs"], what="B=%d sample obs step %d" % (B, t))
        assert_close_rel(np.asarray(rew)[idx], rrew, what="B=%d sample reward step %d" % (B, t))
    np.testing.assert_array_equal(env.samples.get_violation()[idx], ref.samples.get_violation())
    assert (np.asarray(rrew) != 0).any()


def _random_feature_rows(R, seed, hash_size):
    rs = np.random.RandomState(seed)
    seq = np.zeros((R, 2, 64), np.int32)
    n = rs.randint(0, 65, (R, 2))
    ids = rs.randint(1, 284, (R, 2, 64))
    keep = np.arange(64)[None, None, :] >= (64 - n)[:, :, None]
    seq[keep] = ids[keep]
    dense = rs.normal(0, 2, (R, 432)).astype(np.float32)
    catf = rs.randint(0, hash_size, (R, 21)).astype(np.int32)
    return seq, dense, catf


@pytest.mark.parametrize("regime", ["default", "stress"])
@pytest.mark.parametrize("kernel", ["pair", "pp"])
def test_dien_forward_each_augru_kernel(kernel, regime, augru_option):
    """The simulator alone on 200 random feature rows through EACH AUGRU kernel, both weight regimes."""
    from oracle.dien_np import DienOracle
    from rl4rs_b200 import synth
    from test_gpu_parity import _synthetic
    if regime == "default":
        cfg, cat, log, w = _default_regime(8, False)
        hs = 100000
    else:
        cfg, cat, log, w = _synthetic(8, False)
        hs = 5000
    env = make_env(cfg, False, cat, log, w, output_format="numpy")
    seq, dense, catf = _random_feature_rows(200, 5, hs)
    augru_option(kernel)
    obs, probs = env.sim.engine.dien_forward(seq, dense, catf)
    o_ref, p_ref = DienOracle(w, np.float32).forward(seq, dense, catf)
    assert_close_rel(obs.cpu().numpy(), o_ref, what="dien obs [%s, %s]" % (kernel, regime))
    assert_close_rel(probs.cpu().numpy(), p_ref, what="dien probs [%s, %s]" % (kernel, regime))


@pytest.mark.parametrize("kernel", ["pair", "pp"])
@pytest.mark.parametrize("name", ["slate_rllib_replay", "seqslate27_plain_mixed"])
def test_env_fixture_each_augru_kernel(name, kernel, augru_option):
    """Two reference-made fixtures end to end with the AUGRU kernel forced (obs + reward passes)."""
    g = Golden(name)
    cfg, a = g.config, g.arr
    if "np_seed" in g.meta:
        np.random.seed(g.meta["np_seed"])
    env = make_env(cfg, g.seq, g.catalog, g.log, g.weights, output_format="numpy")
    augru_option(kernel)
    k = 0
    for ep in range(g.n_episodes):
        obs = env.reset()
        o = obs["obs"] if isinstance(obs, dict) else obs
        assert_close_rel(o, a["reset_obs"][ep], what="%s [%s] reset obs" % (name, kernel))
        for t in range(cfg["max_steps"]):
            obs, reward, done, info = env.step(a["action_in"][k])
            o = obs["obs"] if isinstance(obs, dict) else obs
            assert_close_rel(o, a["step_obs"][k], what="%s [%s] obs step %d" % (name, kernel, k))
            assert_close_rel(np.asarray(reward, dtype=np.float64), a["reward"][k], what="%s [%s] reward step %d" % (name, kernel, k))
            k += 1


def test_dien_forward_large_launch_sampled():
    """8 300 rows in one call: the sequence cache is built in two chunks (> 8192 sequences), the projection GEMMs run
    more tiles than SMs (persistent multi-wave path) and the AUGRU launch (130 tile-sequences) is multi-wave, so the
    natural rule decides the kernel.  Oracle on 160 sampled rows, 32 of them from the second cache chunk."""
    from oracle.dien_np import DienOracle
    cfg, cat, log, w = _default_regime(8, False)
    env = make_env(cfg, False, cat, log, w, output_format="numpy")
    R = 8300
    seq, dense, catf = _random_feature_rows(R, 9, 100000)
    obs, probs = env.sim.engine.dien_forward(seq, dense, catf)
    obs, probs = obs.cpu().numpy(), probs.cpu().numpy()
    assert np.isfinite(obs).all()
    rs = np.random.RandomState(1)
    idx = np.sort(np.concatenate([rs.choice(8192, 128, replace=False), 8192 + rs.choice(R - 8192, 32, replace=False)]))
    o_ref, p_ref = DienOracle(w, np.float32).forward(seq[idx], dense[idx], catf[idx])
    assert_close_rel(obs[idx], o_ref, what="dien obs large launch")
    assert_close_rel(probs[idx], p_ref, what="dien probs large launch")


def test_augru_kernels_agree_bit_patterns_under_load():
    """Stress for the pair kernel's cross-CTA hand-over (round-1 advisor): the same 1 024-row forward 6 times through
    the pair kernel while a second stream keeps the memory system and the remaining SMs busy; every repetition must
    reproduce the first BIT FOR BIT (a stale h / r*h operand read would show up as a changed mantissa), and all of
    them must agree with the ping-pong kernel (a different schedule of the same arithmetic) to the parity tolerance."""
    import torch
    from rl4rs_b200 import _capi
    cfg, cat, log, w = _default_regime(8, False)
    env = make_env(cfg, False, cat, log, w, output_format="numpy")
    seq, dense, catf = _random_feature_rows(1024, 21, 100000)
    eng = env.sim.engine
    try:
        _capi.set_option("augru_kernel", 3)
        base, _ = eng.dien_forward(seq, dense, catf)
        base = base.cpu().numpy()
        _capi.set_option("augru_kernel", 2)
        side = torch.cuda.Stream()
        junk = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
        outs = []
        for rep in range(6):
            with torch.cuda.stream(side):
                for _ in range(20 + 10 * rep):
                    junk.add_(1)                       # HBM + L2 pressure, varying with the repetition
            o, _ = eng.dien_forward(seq, dense, catf)
            outs.append(o.cpu().numpy())
        torch.cuda.synchronize()
    finally:
        _capi.set_option("augru_kernel", 0)
    for o in outs[1:]:
        np.testing.assert_array_equal(o.view(np.uint32), outs[0].view(np.uint32))
    assert_close_rel(outs[0], base, what="pair vs ping-pong kernel")


@pytest.mark.parametrize("kind", ["slate", "seqslate27"])
def test_pay_step_observation_comes_from_the_reward_pass(kind):
    """A paying step's state is the last complete state of its page (slate.py:203-213 vs :117-131, seqslate.py:104-122 vs
    :27-50), so r4_step takes that step's observation from its reward pass instead of launching a second pass over the
    same feature rows (r4_set_option('pay_obs_reuse', 1), the default).  A/B against the separate observation pass:
    same rewards, masks and observations (different AUGRU kernel / tile shapes: fp32 rounding only), and the option
    does change the launch count."""
    from rl4rs_b200 import _capi
    seq = kind == "seqslate27"
    B = 48
    cfg, cat, log, w = _default_regime(B, seq, support_rllib_mask=True)
    runs = {}
    try:
        for reuse in (1, 0):
            _capi.set_option("pay_obs_reuse", reuse)
            env = make_env(cfg, seq, cat, log, w, output_format="numpy")
            rs = np.random.RandomState(3)
            env.reset()
            n0 = env.sim.engine.launch_count()
            steps = []
            for t in range(cfg["max_steps"]):
                a = np.where(rs.rand(B) < 0.8, np.asarray(env.offline_action), rs.randint(0, 284, B))
                o, rew, done, _ = env.step(a)
                steps.append((o["obs"].copy(), o["action_mask"].copy(), np.asarray(rew).copy()))
            runs[reuse] = (steps, env.sim.engine.launch_count() - n0)
    finally:
        _capi.set_option("pay_obs_reuse", 1)
    paid = 0
    for t, ((o1, m1, r1), (o0, m0, r0)) in enumerate(zip(runs[1][0], runs[0][0])):
        np.testing.assert_array_equal(m1, m0)
        assert_close_rel(o1, o0, what="%s pay-step reuse obs step %d" % (kind, t))
        assert_close_rel(r1, r0, what="%s pay-step reuse reward step %d" % (kind, t))
        paid += int((r0 != 0).any())
    assert paid >= 1                            # (a page of 48 random-replaced slates can be all violations: reward 0)
    assert runs[1][1] < runs[0][1], (runs[1][1], runs[0][1])        # one observation pass fewer per paying step
