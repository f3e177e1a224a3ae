#!/usr/bin/env python
"""bench.py -- env transitions/sec of the B200-native SlateRecEnv hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write what the last timed step computed (.npy)

A "step" is ONE EPISODE of the batched env: reset (row sampling, user-history GRU-1 + input
projections) followed by max_steps x env.step (act, feature assembly, DIEN forward, reward/done),
over `batch_per_gpu` env rows per GPU = batch x max_steps transitions.

Workloads (BASELINE.json configs; defaults give configs[1] at N = 1 and the north-star point at N = 8):
  default            SlateRecEnv-v0, PPO discrete; batch/GPU 4096 at N = 1 (configs[1]), 8192 at N > 1
                     (N = 8: global batch 65 536, the north_star point)            -- override with --batch-per-gpu
  --env seqslate --algo a2c --batch-per-gpu 16384      configs[2]  SeqSlateRecEnv-v0 A2C, 3 pages
  --conti --gpus 4                                     configs[3]  continuous actions + masked kNN, 4 x 8192
  --env seqslate --gpus 8                              configs[4]  SeqSlateRecEnv-v0 PPO, 8 x 8192

JSON keys beyond the base contract:
  value     one training iteration, device-resident: SoftQ rollout of a vector episode (policy + env on the GPU)
            followed by the learner pass (PPO: minibatch SGD epoch; A2C: one step), all hand-written kernels; for
            N > 1 the gradient exchange is the library's own peer-memory kernel (NCCL only as a fallback).
            --conti has no learner in scope (the reference's continuous-action learners are DDPG/TD3): value is the
            rollout with behaviour-policy embeddings + noise through the masked kNN.
  env_only  the same rollout without the learner pass.
  e2e       the reference-facing call with HOST buffers: README.md:14-21 loop, numpy actions in,
            numpy obs/mask/reward out, every copy inside the timed region.
  roofline  the dominant kernel: the tcgen05 AUGRU recurrence (k_augru_pair2 / k_augru_pp, one profile slot), timed
            live with CUDA events on the launching stream during the `value` loop; FLOPs = rows x 2 seq x 64 steps x
            2*(256*512 + 256*256) (DESIGN.md section 4) against the measured sustained bf16 GEMM peak.
  hbm_8d    SURVEY.md section 8(d)'s own HBM figure: transitions/s x algorithmic bytes per transition
            (176 768 B Slate-9, 170 565 B Seq-27) / (N x measured HBM peak), for `value` and `env_only`.
  cpu_baseline  the oracle port (oracle/env_np.py + dien_np.py, run by oracle/cpu_arm.py) on ALL host threads of this box:
            one single-threaded worker process per host thread, the batch's rows spread over them (<= 128 each),
            episodes started together; the same arm is `--impl reference`.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env transitions/sec (SlateRecEnv-v0, batch x steps)"
UNIT = "transitions/s"
BYTES_PER_TRANSITION = {9: 176768, 27: 170565, 36: 169790}     # SURVEY.md section 8(d), dien: 83 732 B per row-forward
G_DNN = 12564                                                   # dnn: algorithmic bytes per row-forward (section 8d)
ROW_FORWARDS_PER_TRANSITION = {9: 19.0 / 9, 27: 55.0 / 27, 36: 73.0 / 36}
CPU_ARM_BUDGET_S = 180.0                                        # --impl reference: warm-up + timed episodes fit in about this
CPU_THREADS_PER_WORKER = 1                                      # CPU arm: one single-threaded worker process per host thread
                                                                # (8 x 1 beats 1 x 8 BLAS threads 9-fold on these matrix sizes)


def base_config(B, seq=False, max_steps=None, conti=False, simulator="dien"):
    cfg = {"epoch": 1, "maxlen": 64, "batch_size": B, "action_size": 284, "class_num": 2,
           "dense_feature_num": 432, "category_feature_num": 21, "category_hash_size": 100000,
           "seq_num": 2, "emb_size": 128, "hidden_units": 128, "page_items": 9,
           "max_steps": max_steps or (27 if seq else 9), "action_emb_size": 32,
           "is_eval": False, "cache_size": 2048, "support_rllib_mask": True}
    if conti:
        cfg["support_conti_env"] = True
    if simulator != "dien":
        cfg["algo"] = simulator                      # slate.py:239-242: rl4rs/nets/<algo>.py
    return cfg


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs"), "bf16_tflops": d.get("bf16_tflops"),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


def cpu_arm_rows(batch, cap):
    """Rows per worker and episode of the CPU arm: the whole batch spread over the workers, at most `cap` each."""
    from oracle import cpu_arm
    W, threads, _ = cpu_arm.plan(CPU_THREADS_PER_WORKER, _cpu_workers_cap())
    return max(1, min(cap, -(-batch // W))), W, threads


def _cpu_workers_cap():
    """One worker per host thread unless the memory limit (RAM or cgroup) says otherwise."""
    from oracle import cpu_arm
    return cpu_arm.workers_cap()


def cpu_reference_episodes(B, seq, episodes, warmup, simulator="dien", parallel=True, log=None, catalog=None, weights=None,
                           budget_s=None, timeout_s=900.0):
    """The reference's CPU path (oracle port, oracle/cpu_arm.py): offline-action replay episodes.  parallel: one
    single-threaded worker process per host thread, B rows each, episodes started together (value = W x B x T / median
    episode); otherwise one process with all its BLAS threads (configs[0], batch 32, the README loop)."""
    from oracle import cpu_arm
    cfg = dict(base_config(B, seq), is_eval=False, cache_size=2048)
    if parallel:
        try:
            return cpu_arm.run_parallel(cfg, seq, simulator, episodes, warmup, threads=CPU_THREADS_PER_WORKER,
                                        workers=_cpu_workers_cap(), budget_s=budget_s, timeout_s=timeout_s)
        except Exception as e:                                # noqa: BLE001 -- e.g. no process spawning in a sandbox
            sys.stderr.write("bench: parallel CPU arm failed (%s); single process\n" % e)
    from rl4rs_b200 import synth
    catalog = catalog or synth.make_catalog()
    log = log or synth.make_log(max(4 * B, 2048), pages=4 if seq else 1, catalog=catalog)
    if weights is None:
        weights = synth.make_dnn_weights(cfg) if simulator == "dnn" else synth.make_weights(cfg)
    return cpu_arm.run_single(cfg, log, catalog, weights, seq, simulator, episodes, warmup, threads=len(cpu_arm.host_cores()))


def cpu_sample_text(r, batch):
    return ("%d of %d env rows per step: %d worker processes x %d rows, one pinned BLAS thread group of %d per worker, "
            "%d of %d host threads busy; one step = one offline-action replay episode = %d transitions; median of %d "
            "episodes, spread (max-min)/median %.2f, NN share of the busy time %.2f"
            % (r["rows_per_episode"], batch, r["workers"], r["rows_per_episode"] // r["workers"], r["threads_per_worker"],
               r["threads"], r["host_cores"], r["transitions_per_episode"], len(r["episode_s"]), r["spread"], r["nn_share"])
            + ("; " + r["note"] if r.get("note") else ""))


def run_reference(args):
    """--impl reference: the oracle port of the reference's CPU env on every host thread; one step = one episode of
    a bounded row sample of the batch (the whole batch when the box has enough threads).  Also reports BASELINE
    configs[0] itself (batch 32, one process, the README loop) over 3 episodes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    seq = args.env == "seqslate"
    rows, W, threads = cpu_arm_rows(args.batch_per_gpu, args.cpu_sample_rows)
    r = cpu_reference_episodes(rows, seq, max(args.steps, 1), max(args.warmup, 1), simulator=args.simulator,
                               budget_s=CPU_ARM_BUDGET_S)
    c1 = cpu_reference_episodes(32, seq, 3, 1, simulator=args.simulator, parallel=False)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["median_s"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, seq),
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                             "sample": cpu_sample_text(r, args.batch_per_gpu),
                             "episode_s": r["episode_s"], "nn_share": r["nn_share"],
                             "configs0_batch32": {"value": c1["value"], "episode_s": c1["episode_s"], "nn_share": c1["nn_share"],
                                                  "threads": c1["threads"]}},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_config(args, seq):
    T = 27 if seq else 9
    env = "SeqSlateRecEnv-v0" if seq else "SlateRecEnv-v0"
    if args.conti:
        learner = "continuous actions (behaviour-policy embeddings + N(0, 0.3) noise) through the masked kNN; no learner pass"
    elif args.algo == "a2c":
        learner = "A2C (MyMaskActionsModel, SoftQ T=1 rollout + one summed-loss step, grad clip 10)"
    else:
        learner = ("PPO discrete (MyMaskActionsModel, SoftQ T=1 rollout + one SGD epoch, sgd_minibatch_size %d TOTAL = %d per GPU)"
                   % (args.sgd_minibatch, args.sgd_minibatch // max(args.gpus, 1)))
    return {"workload": "%s batch=%d/GPU x max_steps=%d, %s, %s simulator, synthetic 283-item catalog + synthetic log "
                        "(seed 1234) + synthetic weights (seed 4321)" % (env, args.batch_per_gpu, T, learner, args.simulator.upper()),
            "batch_per_gpu": args.batch_per_gpu, "global_batch": args.batch_per_gpu * args.gpus,
            "max_steps": T, "simulator": args.simulator, "algo": "none" if args.conti else args.algo,
            "sgd_minibatch_size_total": None if (args.conti or args.algo != "ppo") else args.sgd_minibatch,
            "category_hash_size": 100000,
            "parallelism": "env rows sharded by contiguous blocks, dp%d, no data-path collective" % args.gpus,
            "per_n_defaults": "batch/GPU 4096 at N=1 (BASELINE configs[1]), 8192 at N>1 (N=8: north_star global batch 65 536); "
                              "PPO sgd_minibatch_size 256 x N so that an iteration is 144 x (batch/4096) optimizer steps at every N",
            "simulator_passes": "every observation and every reward is computed; a paying step's observation is row 8 of its "
                                "page's reward rows (the reference evaluates that one feature row twice: slate.py:203-213 = "
                                ":117-131 at j = 8), so %d simulator row-forwards per env row and episode instead of %d "
                                "(R4_NO_PAY_OBS_REUSE=1 launches the duplicate pass)" % ((2 * T + 1 - T // 9), 2 * T + 1),
            "l2": "per-step working set (AUGRU input-projection cache ~0.21 MB/row, 0.87 GB at batch 4096) "
                  "exceeds the 126 MB L2; no explicit flush"}


DUMP_ROWS = 512                                                 # --dump-outputs: env rows kept of the [T, B, ...] arrays
DUMP_LIMIT = 64 << 20


def dump_outputs(dirname, arrays, batch, row_axis):
    """Write what the last timed step handed its caller as DIR/<name>.npy (float32, or float64 where float32 would round),
    keeping a fixed, seeded sample of DUMP_ROWS env rows (axis `row_axis`) of the arrays that hold a feature vector per
    row, so that two builds can be compared."""
    rows = np.sort(np.random.RandomState(0).choice(batch, min(batch, DUMP_ROWS), replace=False))
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        if a.ndim > row_axis + 1 and a.shape[row_axis] == batch:
            a = np.take(a, rows, axis=row_axis)
        out[name] = a.astype(np.float64 if a.dtype.itemsize > 4 or a.dtype.kind in "iu" else np.float32)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT, "outputs to dump: %d bytes" % total
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL's version banner, library
    chatter) was redirected to stderr at start-up so the driver can parse stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1
if __name__ == "__main__":                      # not when imported (tests, the CPU arm's worker processes)
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--env", default="slate", choices=["slate", "seqslate"])
    ap.add_argument("--algo", default="ppo", choices=["ppo", "a2c"])
    ap.add_argument("--conti", action="store_true", help="continuous actions + masked kNN (BASELINE configs[3]); no learner")
    ap.add_argument("--simulator", default="dien", choices=["dien", "dnn"],
                    help="config['algo']: dien (BASELINE configs, tensor-bound) or dnn (nets/dnn.py, the gather-bound simulator)")
    ap.add_argument("--batch-per-gpu", type=int, default=None, help="default: 4096 at N=1, 8192 at N>1")
    ap.add_argument("--sgd-minibatch", type=int, default=None, help="PPO sgd_minibatch_size, TOTAL over GPUs (default 256 x N)")
    ap.add_argument("--cpu-sample-rows", type=int, default=128, help="CPU arm: at most this many env rows per worker process")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernels", action="store_true", help="also print a per-kernel time breakdown (stderr)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if world_env > 1:
        args.gpus = world_env
    if args.batch_per_gpu is None:
        args.batch_per_gpu = 4096 if args.gpus == 1 else 8192
    if args.sgd_minibatch is None:
        args.sgd_minibatch = 256 * args.gpus
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()
    from rl4rs_b200 import synth, gymshim
    from rl4rs_b200.env.slate import SlateRecEnv, SlateState
    from rl4rs_b200.env.seqslate import SeqSlateRecEnv, SeqSlateState
    from rl4rs_b200.trainer import PPOTrainer, A2CTrainer

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = world_env
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    seq = args.env == "seqslate"
    B = args.batch_per_gpu
    cfg = base_config(B, seq, conti=args.conti, simulator=args.simulator)
    T = cfg["max_steps"]
    catalog = synth.make_catalog()
    # the log is generated once from the single seed; rank r samples from its own slice of it
    n_log = max(4 * B, 8192)
    log = synth.make_log(n_log, pages=4 if seq else 1, catalog=catalog, seed=synth.LOG_SEED + rank)
    weights = synth.make_dnn_weights(cfg) if args.simulator == "dnn" else synth.make_weights(cfg)

    def make(fmt):
        c = dict(cfg, catalog=catalog, log=log, weights=weights, output_format=fmt, device=local_rank)
        sim = (SeqSlateRecEnv(c, state_cls=SeqSlateState) if seq else SlateRecEnv(c, state_cls=SlateState))
        return gymshim.make("SeqSlateRecEnv-v0" if seq else "SlateRecEnv-v0", recsim=sim)

    env = make("torch")
    env.seed(rank)
    eng = env.sim.engine
    trainer, learner_launches = None, (lambda: 0)
    if args.conti:
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)

        def rollout_conti():
            env.reset()
            for _ in range(T):
                a = env.offline_action                                  # logged items' embeddings, f64 [B, 32] on the device
                a = a + 0.3 * torch.randn(a.shape, generator=gen, device=dev, dtype=a.dtype)
                obs, reward, done, info = env.step(a)
            return {"obs": obs["obs"], "action_mask": obs["action_mask"], "reward": reward, "done": done}

        episode_device = episode_env_only = rollout_conti
    else:
        trainer = (PPOTrainer({"sgd_minibatch_size": args.sgd_minibatch}, env, seed=0) if args.algo == "ppo"
                   else A2CTrainer({}, env, seed=0))                     # modelfree_train.py:179-217 / :248-304
        learner_launches = lambda: trainer.ops.launches

        def episode_device():                                            # rollout + learner pass
            stats = trainer.train()
            b = trainer.buf
            out = {"obs": b.obs, "action_mask": b.mask, "action": b.action, "logp": b.logp, "value": b.value,
                   "logits": b.logits, "reward": b.reward, "policy_params": trainer.policy.flat}
            out.update({"stats_" + k: np.float64(v) for k, v in stats.items() if isinstance(v, (int, float))})
            return out
        episode_env_only = lambda: trainer.rollout(explore=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for _ in range(args.warmup):
        episode_device()
    launches0 = eng.launch_count() + learner_launches()
    eng.profile(1)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms, last = timed(episode_device, args.steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, B, row_axis=0 if args.conti else 1)
    prof = eng.profile_read()
    eng.profile(0)
    gpu_launches = eng.launch_count() + learner_launches() - launches0   # env kernels + policy/learner kernels
    value = B * world * T * args.steps / (ms / 1e3)
    ms_env, _ = timed(episode_env_only, args.steps)
    env_only = B * world * T * args.steps / (ms_env / 1e3)

    # ---- e2e: reference-facing call, host buffers (README.md:14-21 loop) ------------------------
    env_h = make("numpy")
    env_h.seed(rank)

    def episode_host():
        obs = env_h.reset()
        for _ in range(T):
            a = env_h.offline_action                      # numpy (D2H) -- the logged policy (ids, or embeddings with --conti)
            obs, reward, done, info = env_h.step(a)       # H2D actions, D2H obs + mask + reward
        return reward

    for _ in range(args.warmup):
        episode_host()
    ms_h, _ = timed(episode_host, args.steps)
    e2e = B * world * T * args.steps / (ms_h / 1e3)
    act_bytes = B * 32 * 8 if args.conti else B * 4
    h2d = B * 4 + T * act_bytes
    d2h = (T + 1) * (B * 256 * 4 + B * 284) + T * (B * 8 + act_bytes)

    # ---- per-kernel breakdown (untimed extra episode) -------------------------------------------
    kernels = None
    if rank == 0:
        eng.profile(2)
        episode_env_only()
        torch.cuda.synchronize(dev)
        kernels = eng.profile_read()
        eng.profile(0)
        if args.kernels:
            tot = sum(k["ms"] for k in kernels)
            for k in sorted(kernels, key=lambda k: -k["ms"]):
                sys.stderr.write("%-44s %9.3f ms %5.1f%%  launches %d\n" % (k["name"], k["ms"], 100 * k["ms"] / tot, k["launches"]))

    exchange = None
    if trainer is not None and world > 1:
        exchange = "peer-memory kernel (r4_comm)" if (trainer.comm is not None and trainer.comm.ok) else "nccl all_reduce per step (fallback: %s)" % (trainer.comm.why if trainer.comm else "no kernels")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    au = [p for p in prof if p["name"].startswith("k_augru")]
    roofline = None
    if au:
        au = au[0]
        achieved = au["work"] / (au["ms"] / 1e3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "augru_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        roofline = {"kernel": "AUGRU recurrence, tcgen05.mma.cta_group::2 kind::f16, bf16 hi/lo split x3, fp32 TMEM accumulators: k_augru_pair2 "
                              "(one recurrence per CTA pair) / k_augru_pp (two per pair), chosen per launch by r4_augru_kernel_for",
                    "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "traffic_source": traffic_src or "profiles/augru_traffic.json (ncu --set full capture of an observation-pass launch, committed; not re-measured in this run)",
                    "peak_source": "%s bf16 GEMM, sustained (kernel timed inside a long step)" % peaks["source"],
                    "launches": au["launches"], "avg_launch_ms": au["ms"] / au["launches"],
                    "share_of_step": au["ms"] / ms}
    bpt = BYTES_PER_TRANSITION.get(T, 176768)
    hbm = peaks["hbm_gbs"]
    if args.simulator == "dnn":
        bpt = int(round(G_DNN * ROW_FORWARDS_PER_TRANSITION.get(T, 19.0 / 9)))
        gk = [p for p in prof if p["name"].startswith("k_cat")]
        if gk:
            gk = gk[0]
            gbs = gk["work"] / (gk["ms"] / 1e3) / 1e9
            traffic, traffic_src = None, None
            tp = os.path.join(ROOT, "profiles", "dnn_gather_traffic.json")
            if os.path.exists(tp):
                tj = json.load(open(tp))
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            roofline = {"kernel": "k_cat_pool: Embedding gather + GlobalAveragePooling1D of the dnn simulator, 21 x 512 B rows per "
                                  "feature row staged by cp.async.bulk (1-D TMA) into shared memory, 128-bit reduction reads",
                        "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "traffic": traffic,
                        "traffic_source": traffic_src or "profiles/dnn_gather_traffic.json (ncu capture; the 51 MB table is L2-resident, "
                                                          "so DRAM traffic is far below the algorithmic bytes)",
                        "algorithmic_bytes_per_row": 21 * 4 + 21 * 512, "launches": gk["launches"],
                        "avg_launch_ms": gk["ms"] / gk["launches"], "share_of_step": gk["ms"] / ms,
                        "peak_source": "%s HBM copy bandwidth" % peaks["source"]}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, seq), "clocks": clk,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_h / args.steps,
                    "loop": "README.md:14-21: action = env.offline_action; env.step(action); numpy in/out"},
            "gpu_launches": gpu_launches, "roofline": roofline,
            "hbm_8d": {"bound": "hbm", "bytes_per_transition": bpt, "peak": hbm, "unit": "GB/s", "n_gpus": world,
                       "achieved_value": value * bpt / 1e9, "frac_value": value * bpt / 1e9 / (world * hbm),
                       "achieved_env_only": env_only * bpt / 1e9, "frac_env_only": env_only * bpt / 1e9 / (world * hbm),
                       "note": "SURVEY.md 8(d): transitions/s x algorithmic bytes per transition / (N x measured HBM peak); the DIEN "
                               "simulator is tensor-bound (111.5 MFLOP per row-forward), so its fraction is small by construction; the "
                               "dnn simulator (12 564 B per row-forward) is the gather-bound configuration"},
            "env_only": {"value": env_only, "unit": UNIT, "ms_per_step": ms_env / args.steps,
                         "note": "same rollout without the learner pass (policy sampling still on the GPU)"}}
    if exchange:
        line["gradient_exchange"] = exchange
    if kernels:
        tot = sum(k["ms"] for k in kernels)
        line["kernels"] = [{"name": k["name"], "ms": round(k["ms"], 3), "share": round(k["ms"] / tot, 4),
                            "launches": k["launches"]} for k in sorted(kernels, key=lambda k: -k["ms"])]
    if world == 1 and not args.no_cpu_baseline:
        try:
            rows, _, _ = cpu_arm_rows(B, args.cpu_sample_rows)
            r = cpu_reference_episodes(rows, seq, episodes=3, warmup=1, simulator=args.simulator, budget_s=30.0, timeout_s=240.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                                    "sample": cpu_sample_text(r, B) + "; %.1f s timed" % r["total_s"],
                                    "episode_s": r["episode_s"], "nn_share": r["nn_share"]}
        except Exception as e:                                # noqa: BLE001 -- the GPU line must be printed whatever the CPU leg does
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %s" % e}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
