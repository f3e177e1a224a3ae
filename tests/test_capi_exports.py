"""CPU: the C-ABI library loads and exports every symbol include/rl4rs_b200.h declares."""
import os
import re

import pytest

from rl4rs_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "rl4rs_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(r4_[a-z_0-9]+)\s*\(", text)))


def test_library_builds_and_exports_header_symbols():
    import __graft_entry__ as g
    g.build()
    lib = _capi.load_library()
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
    assert set(syms) == set(_capi.EXPORTS), set(syms) ^ set(_capi.EXPORTS)
    assert lib.r4_abi_version() == 2


def test_create_rejects_bad_config_without_gpu_work():
    import ctypes as C
    lib = _capi.load_library()
    cfg = _capi.R4Config(env_kind=0, flags=0, batch_size=4, max_steps=9, page_items=9, action_size=284,
                         action_emb_size=32, maxlen=32, seq_num=2, dense_feature_num=432,
                         category_feature_num=21, category_hash_size=1000, emb_size=128, hidden_units=128,
                         max_rows_per_pass=0)
    h = C.c_void_p()
    rc = lib.r4_create(C.byref(cfg), 0, C.byref(h))
    assert rc == -1 and not h.value
    assert b"maxlen=64" in lib.r4_last_error(None)


def test_no_cpu_fallback():
    """Constructing an env without a CUDA device must fail loudly, not fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from rl4rs_b200 import synth
    from rl4rs_b200.env.slate import SlateRecEnv, SlateState
    cfg = {"batch_size": 2, "max_steps": 9, "action_size": 284, "category_hash_size": 400,
           "catalog": synth.make_catalog(), "log": synth.make_log(8, hash_size=400),
           "weights": synth.make_weights({"category_hash_size": 400})}
    with pytest.raises(_capi.R4Error):
        SlateRecEnv(cfg, state_cls=SlateState)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under rl4rs_b200/ may import it."""
    pkg = os.path.join(ROOT, "rl4rs_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|import_module\(.oracle|oracle[/.](env_np|dien_np|ref_harness)", re.M)
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(d, f)).read()
                assert not pat.search(src), os.path.join(d, f)


def test_augru_kernel_choice_rule():
    """r4_augru_kernel_for(ctas = 2 x row tiles, sms): 2 = k_augru_pair2 (a CTA pair per tile-sequence), 3 = k_augru_pp (a
    CTA pair per tile, both sequences in flight) -- the cheaper by wave count x measured wave cost (defaults 13 : 24).
    B200 (148 SMs): a 4096-row observation pass = 64 tile-sequences -> pair2 (one wave on 128 SMs beats one ping-pong wave
    on 64); the 36 864-row reward pass = 576 and 8192-row passes = 128 -> ping-pong.  (1 was the round-1 one-CTA kernel,
    deleted: it lost every regime.)"""
    from rl4rs_b200 import _capi
    lib = _capi.load_library()
    f = lib.r4_augru_kernel_for

    def want(ctas, sms, cp=13, cpp=24):
        pairs = sms // 2
        c2, c3 = cp * -(-ctas // pairs), cpp * -(-((ctas + 1) // 2) // pairs)
        return 3 if c3 <= c2 else 2

    assert f(64, 148) == 2 and f(2, 148) == 2 and f(74, 148) == 2
    assert f(576, 148) == 3 and f(128, 148) == 3 and f(148, 148) == 3
    assert f(0, 148) == 0 and f(64, 1) == 0      # bad arguments
    for ctas in range(1, 1200, 7):
        assert f(ctas, 148) == want(ctas, 148), ctas
    # r4_set_option: overrides are validated, and the rule follows the costs it is given
    assert lib.r4_set_option(b"augru_cost_pp", 100) == 0
    assert f(576, 148) == 2 and f(64, 148) == 2          # without the ping-pong kernel: the pair kernel takes every pass
    assert lib.r4_set_option(b"augru_cost_pair", 60) == 0
    assert f(576, 148) == 3
    for k, v in ((b"augru_cost_pair", 13), (b"augru_cost_pp", 24)):
        assert lib.r4_set_option(k, v) == 0
    assert lib.r4_set_option(b"augru_kernel", 1) != 0 and lib.r4_set_option(b"augru_cost_single", 3) != 0   # the deleted kernel
    assert lib.r4_set_option(b"augru_kernel", 7) != 0 and lib.r4_set_option(b"no_such_key", 1) != 0
    assert lib.r4_set_option(b"augru_kernel", 0) == 0


def test_c99_caller_compiles_links_and_runs(tmp_path):
    """INTEGRATION.md section 6: the header is self-contained C99 and the library is callable from plain C (no torch, no
    Python).  tests/c_caller/c_caller.c uses the entry points that need no GPU."""
    import shutil
    import subprocess
    import __graft_entry__ as g
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lib = g.build()
    exe = str(tmp_path / "c_caller")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "c_caller", "c_caller.c"), "-L", os.path.dirname(lib), "-lrl4rs_b200",
                    "-Wl,-rpath," + os.path.dirname(lib), "-o", exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert "abi 2" in out and "obs_dim dien 256 widedeep 3072" in out
    assert "create rc -1 env null" in out and "maxlen=64" in out
    # the ctypes mirrors of the two structs (rl4rs_b200/_capi.py, INTEGRATION.md section 2) have the C layout
    import ctypes as C
    assert "sizeof r4_config %d r4_out %d" % (C.sizeof(_capi.R4Config), C.sizeof(_capi.R4Out)) in out


def test_set_option_accepts_the_documented_keys_and_rejects_removed_ones():
    """r4_set_option: every key the header lists is accepted with a documented value and restored; the keys of the
    removed kernel variants, unknown keys and out-of-range values are R4_ERR_ARG with a message (no GPU involved:
    process-wide host state)."""
    lib = _capi.load_library()
    text = open(os.path.join(ROOT, "include", "rl4rs_b200.h")).read()
    block = text[text.index("Process-wide kernel-choice overrides"):text.index("int r4_set_option")]
    keys = set(re.findall(r'"([a-z_0-9]+)"', block))
    defaults = {"augru_kernel": 0, "augru_cost_pair": 13, "augru_cost_pp": 24, "pay_obs_reuse": 1, "scores_shared_pct": 85}
    assert keys == set(defaults), keys ^ set(defaults)
    try:
        for k, other in (("augru_kernel", 3), ("augru_cost_pair", 7), ("augru_cost_pp", 9), ("pay_obs_reuse", 0),
                         ("scores_shared_pct", 50)):
            assert lib.r4_set_option(k.encode(), other) == 0, k
        # the rule reads the costs just set (7 : 9): one wave of 64 tile-sequences -> pair; 8 waves against 4 -> ping-pong
        assert lib.r4_augru_kernel_for(64, 148) == 2 and lib.r4_augru_kernel_for(592, 148) == 3
    finally:
        for k, v in defaults.items():
            assert lib.r4_set_option(k.encode(), v) == 0, k
    # the kernel variants these keys used to select are gone, and so are the keys
    for k, v in (("augru_pair_impl", 1), ("augru_cluster", 2), ("scores_impl", 2)):
        assert lib.r4_set_option(k.encode(), v) == -1 and k.encode() in lib.r4_last_error(None), k
    assert lib.r4_set_option(b"no_such_option", 1) == -1 and b"no_such_option" in lib.r4_last_error(None)
    assert lib.r4_set_option(b"augru_kernel", 1) == -1 and lib.r4_set_option(b"scores_shared_pct", 5) == -1


def test_host_only_entry_points_agree_with_the_python_side():
    """Pure host arithmetic behind the ABI: parameter count of the policy (flat layout of rl4rs_b200/policy.py), observation
    widths per simulator."""
    import ctypes as C
    from rl4rs_b200.policy import MaskedPolicy
    lib = _capi.load_library()
    lib.r4_policy_num_params.restype = C.c_int
    for A in (284, 50):
        assert lib.r4_policy_num_params(A) == MaskedPolicy(A, "cpu").n_params == 256 * 64 + 64 + 64 * A + A + 64 + 1
    assert [lib.r4_obs_dim(_capi.SIMULATORS[k]) for k in ("dien", "dnn", "widedeep", "lstm")] == [256, 256, 3072, 256]
