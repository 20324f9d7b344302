#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: minibatch TD-updates/sec.

Default workload (`--config 2`, BASELINE configs[1]): Discrete DQN (double-Q, huber), synthetic
transitions S=128, A=16, global batch 4096, prioritized replay (fp64 sum tree, capacity 2^20).
`--config 3|4|5` run BASELINE configs[2..4] (QR-DQN 200 atoms B=4096; SAC twin critics S=256
A=32 B=8192; TD3 S=512 A=64 B=16384); the default N=1 line also carries their numbers in a
`configs` array.

One "step" = one full update INCLUDING drawing the minibatch: replay-sample kernel (tree walk +
gather + trainer-batch formatting) -> fused TD-target/loss/backward kernel(s) -> weight
gradients -> fused Adam + soft target update.

  value : K updates, device-timed (CUDA events), all random numbers already in HBM
          (config 2: the K updates are ONE captured CUDA graph).
  e2e   : the same K updates through the public API: per update the host draws the random
          numbers (Python `random` stream, bit-exact with the reference), copies them
          host->device from pinned memory, runs the update and copies the loss device->host.
  roofline     : the fused TD kernel, algorithmic FLOPs / measured duration (events per launch).
  cpu_baseline : the CPU oracle (restatement of the reference's sampler + trainer update, torch
                 fp32 on the host cores) on a bounded number of updates.

N > 1 (torchrun): STRONG scaling of one global minibatch, as SURVEY.md 8e states it -- replay
replicated (identical add stream and identical host random stream, so every rank selects the
same global indices), rank r gathers and trains on rows [r*B/N, (r+1)*B/N), parameters and
optimizer state replicated, the gradient exchange is fused into the Adam kernel over NVLink peer
memory (one launch; plain NCCL all-reduce if peer mapping is unavailable).  `value` = global
minibatch updates/s.  The weak-scaling figure (4096 rows per rank) is kept under detail.weak
(`config` is identical in both arms, so everything run-specific lives in `detail`).

`--impl reference` times the reference algorithm's CPU path (the oracle port: /root/reference
does not exist on the GPU box) with the best host thread count of a sweep.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAMMA, TAU, LR = 0.99, 0.005, 1e-3
CONFIGS = {
    2: dict(algo="dqn", S=128, A=16, B=4096, cap=1 << 20, sizes=[256, 128],
            metric="minibatch_td_updates_per_sec_b4096",
            workload="configs[1]: Discrete DQN double-Q huber, synthetic S=128 A=16 B=4096, "
                     "prioritized replay cap=2^20, MLP 128-256-128-16 relu, Adam 1e-3, tau 0.005"),
    3: dict(algo="qrdqn", S=128, A=32, N=200, B=4096, cap=1 << 20, sizes=[256, 128],
            metric="minibatch_td_updates_per_sec_qrdqn_b4096",
            workload="configs[2]: QR-DQN 200 quantiles double-Q, synthetic S=128 A=32 B=4096, "
                     "prioritized replay cap=2^20, MLP 128-256-128-6400 relu, Adam 1e-3, tau 0.005"),
    4: dict(algo="sac", S=256, A=32, B=8192, cap=1 << 18, sizes=[256, 256],
            metric="minibatch_td_updates_per_sec_sac_b8192",
            workload="configs[3]: SAC twin critics learnable alpha, synthetic S=256 A=32 B=8192 "
                     "(global), prioritized replay cap=2^18, actor/critics [256,256] relu, Adam 1e-3"),
    5: dict(algo="td3", S=512, A=64, B=16384, cap=1 << 18, sizes=[256, 256],
            metric="minibatch_td_updates_per_sec_td3_b16384",
            workload="configs[4]: TD3 twin critics delayed_policy_update=2, synthetic S=512 A=64 "
                     "B=16384 (global), prioritized replay cap=2^18, actor/critics [256,256] relu"),
}
ACTS = ["relu", "relu"]
# kept for the profiling scripts under profiles/
S, A, B, CAP = CONFIGS[2]["S"], CONFIGS[2]["A"], CONFIGS[2]["B"], CONFIGS[2]["cap"]
SIZES = CONFIGS[2]["sizes"]
METRIC, WORKLOAD = CONFIGS[2]["metric"], CONFIGS[2]["workload"]


def _sigma(dims):
    return sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))


def td_kernel_flops(cfg=None, rows=None):
    """Algorithmic FLOPs of one launch of the fused TD kernel (SURVEY.md 8d K2 + K2').
    DQN: 3 forwards (q(s'), q_target(s'), q(s)) + the dX chain of the backward (all layers but
    the first).  SAC / TD3 critic step: actor forward(s) on s' (+ the log-prob re-forward for
    SAC), two target critics, two online critics forward + their dX chains."""
    c = CONFIGS[2] if cfg is None else cfg
    rows = c["B"] if rows is None else rows
    if c["algo"] == "dqn":
        dims = [c["S"]] + c["sizes"] + [c["A"]]
        return 3 * 2 * rows * _sigma(dims) + 2 * rows * _sigma(dims[1:])
    if c["algo"] in ("sac", "td3"):
        actor = [c["S"]] + c["sizes"] + [c["A"] * (2 if c["algo"] == "sac" else 1)]
        crit = [c["S"] + c["A"]] + c["sizes"] + [1]
        n_actor = 2 if c["algo"] == "sac" else 1
        fwd = n_actor * _sigma(actor) + 4 * _sigma(crit)
        return 2 * rows * fwd + 2 * 2 * rows * _sigma(crit[1:])
    return None


def update_flops(cfg, rows):
    """Algorithmic FLOPs of one whole update (forwards + dX + dW), for the update-level rate."""
    if cfg["algo"] == "qrdqn":
        dims = [cfg["S"]] + cfg["sizes"] + [cfg["A"] * cfg["N"]]
        return (3 + 2) * 2 * rows * _sigma(dims) + 10 * rows * cfg["N"] ** 2
    return None


def synth_stream(n, seed, cfg=None):
    import numpy as np

    c = CONFIGS[2] if cfg is None else cfg
    rng = np.random.RandomState(seed)
    st = dict(observation=rng.standard_normal((n, c["S"])).astype(np.float32))
    if c["algo"] in ("sac", "td3"):
        st["action"] = rng.uniform(-0.99, 0.99, (n, c["A"])).astype(np.float32)
    else:
        st["action"] = rng.randint(0, c["A"], n).astype(np.int64)
    st.update(reward=rng.standard_normal(n).astype(np.float32),
              terminal=rng.rand(n) < (1.0 / 200.0),
              priority=rng.uniform(0.1, 10.0, n))
    return st


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.t_mark = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), line.strip()))
        except Exception:
            pass

    def mark(self):
        """Samples from here on belong to the timed regions."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm, reasons = [], set()
        rows = [r for t, r in self.rows if self.t_mark is None or t >= self.t_mark] or \
               [r for _, r in self.rows[-3:]]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                out["sm_max_mhz"] = float(p[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


# ---------------------------------------------------------------------------
# the reference algorithm on the host (oracle port)
# ---------------------------------------------------------------------------
def _cpu_setup(cfg):
    """Build the oracle-side state of one config; returns one() -> loss (a full update
    including the PER sample)."""
    import numpy as np
    import torch

    from oracle import td_oracle as O
    from oracle.replay_oracle import ReplayOracle

    cap, Bc, Sc, Ac = cfg["cap"], cfg["B"], cfg["S"], cfg["A"]
    ro = ReplayOracle(cap, prioritized=True)
    ro.bulk_fill(synth_stream(cap, 1000, cfg))
    gen = torch.Generator().manual_seed(0)
    algo = cfg["algo"]
    extra = synth_stream(256, 555, cfg) if algo == "dqn" else None
    it = [0]
    if algo in ("dqn", "qrdqn"):
        out = Ac * (cfg.get("N", 1))
        q = O.make_net([Sc] + cfg["sizes"] + [out], ACTS + ["linear"], gen)
        for t in O.net_params(q):
            t.requires_grad_(True)
        qt = O.clone_net(q)
        adam = O.AdamState(O.net_params(q), lr=LR)

        def one():
            if extra is not None:  # the online loop: one new transition per update
                i = it[0] % len(extra["terminal"])
                ro.add(**{k: v[i] for k, v in extra.items()})
                it[0] += 1
            ob = ro.sample_transition_batch(Bc)
            term = torch.from_numpy(ob["terminal"])
            batch = dict(
                state=torch.from_numpy(ob["state"]), next_state=torch.from_numpy(ob["next_state"]),
                reward=torch.from_numpy(ob["reward"]).reshape(-1, 1),
                not_terminal=1.0 - term.float().reshape(-1, 1),
                action=torch.nn.functional.one_hot(torch.from_numpy(ob["action"]), Ac).float(),
                possible_next_actions_mask=torch.ones(Bc, Ac), next_action=None)
            if algo == "dqn":
                return O.dqn_update(q, qt, adam, batch, gamma=GAMMA, tau=TAU, loss="huber")[0]
            return O.qrdqn_update(q, qt, adam, batch, gamma=GAMMA, tau=TAU, num_atoms=cfg["N"])[0]
        return one
    actor_out = Ac * (2 if algo == "sac" else 1)
    actor = O.make_net([Sc] + cfg["sizes"] + [actor_out], ACTS + ["linear" if algo == "sac" else "tanh"], gen)
    q1 = O.make_net([Sc + Ac] + cfg["sizes"] + [1], ACTS + ["linear"], gen)
    q2 = O.make_net([Sc + Ac] + cfg["sizes"] + [1], ACTS + ["linear"], gen)
    st = O.SacState(actor, q1, q2, lr=LR) if algo == "sac" else O.Td3State(actor, q1, q2, lr=LR)
    it = [0]

    def one():
        ob = ro.sample_transition_batch(Bc)
        term = torch.from_numpy(ob["terminal"]).float().reshape(-1, 1)
        batch = dict(state=torch.from_numpy(ob["state"]), next_state=torch.from_numpy(ob["next_state"]),
                     reward=torch.from_numpy(ob["reward"]).reshape(-1, 1), not_terminal=1.0 - term,
                     action=torch.from_numpy(ob["action"]),
                     next_action=torch.from_numpy(ob["next_action"]) * (1.0 - term))
        nn = torch.randn(Bc, Ac)
        if algo == "sac":
            r = O.sac_update(st, batch, nn, torch.randn(Bc, Ac), gamma=GAMMA, tau=TAU)
        else:
            r = O.td3_update(st, batch, nn, it[0], gamma=GAMMA, tau=TAU)
        it[0] += 1
        return r["losses"][0]
    return one


def cpu_reference_run(steps, warmup, cfg=None, threads=None):
    """The reference algorithm on the host: PER sample (python loops over an fp64 sum tree, as
    reagent/replay_memory does) + the trainer update (torch fp32).  Returns (updates/s, cores,
    sample description, ms per step)."""
    import torch

    cfg = CONFIGS[2] if cfg is None else cfg
    one = _cpu_setup(cfg)
    cores = threads or os.cpu_count()
    torch.set_num_threads(cores)
    if threads is None:
        # "all the host threads it can use": small GEMMs get SLOWER when oversubscribed, so
        # give the reference its best thread count from a short sweep (1 update each)
        best = None
        for c in sorted({os.cpu_count(), 64, 32, 16, 8}, reverse=True):
            if c > os.cpu_count():
                continue
            torch.set_num_threads(c)
            one()
            t0 = time.perf_counter()
            one()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, c)
        cores = best[1]
        torch.set_num_threads(cores)
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return (steps / dt, cores,
            f"{steps} full updates ({'1 replay add + ' if cfg['algo'] == 'dqn' else ''}PER sample B={cfg['B']} + {cfg['algo']} update) after "
            f"{warmup} warm-up; torch threads={cores} (best of a sweep over <= {os.cpu_count()} cores)",
            dt / steps * 1e3)


def _cpu_steps(cfg, asked):
    """Bounded sample: ~10-30 s of CPU work per config."""
    return {"dqn": min(asked, 60), "qrdqn": 3, "sac": min(asked, 12), "td3": min(asked, 8)}[cfg["algo"]]


def base_config(cfg, world):
    return {"workload": cfg["workload"], "global_batch": cfg["B"],
            "parallelism": f"dp{world}" if world > 1 else "single",
            "l2": "inputs larger than L2: the replay store (%d MiB) is gathered at random rows "
                  "every update" % (cfg["cap"] * cfg["S"] * 4 >> 20)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    steps = _cpu_steps(cfg, min(args.steps, 40))
    # same warm-up count as our arm for config 2 (the driver passes the same flags to both);
    # the slow configs warm up once (one QR-DQN update is ~2 s of host time)
    warm = max(args.warmup, 3) if cfg["algo"] == "dqn" else 1
    v, cores, sample, ms = cpu_reference_run(steps, warm, cfg)
    conf = base_config(cfg, args.gpus)  # identical to our arm's `config`
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": v, "unit": "updates/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": conf,
        "cpu_baseline": {"value": v, "unit": "updates/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {"note": "reference algorithm restated on CPU (oracle/replay_oracle.py + "
                           "oracle/td_oracle.py): /root/reference is not on the GPU box; a CPU arm "
                           "has no ranks: the global minibatch is processed by one process on the "
                           "host cores whatever --gpus says"},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
class Env:
    """rank / world / device / process group + the timing helpers every config shares."""

    def __init__(self):
        import torch

        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.pg = None
        self.collective = None
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.dev)
            self.pg = dist.group.WORLD
            self.collective = "nccl all_reduce of the flat gradient (one per optimizer sub-step)"
            if os.environ.get("RB200_DP_P2P", "1") == "1":
                try:
                    from reagent_b200.training.data_parallel import enable_p2p

                    enable_p2p(self.pg)
                    self.collective = ("gradient exchange fused into the Adam kernel: peer-to-peer "
                                       "stores over NVLink + per-block flags, summed in rank order "
                                       "(no NCCL call on the data path)")
                except Exception as e:  # peer mapping unavailable: plain NCCL
                    self.collective += f" [p2p unavailable: {type(e).__name__}: {e}]"
                    ok = torch.zeros(1, device=self.dev)
                    dist.all_reduce(ok)  # keep ranks in step

    def barrier(self):
        import torch

        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        import torch

        if self.world == 1:
            return ms
        import torch.distributed as dist

        t = torch.tensor([ms], device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def shard(self, Bg):
        from reagent_b200.training.data_parallel import shard_rows

        return shard_rows(Bg, self.rank, self.world)


def build_trainer(cfg, dev, seed=0):
    import torch

    from reagent_b200.core.parameters import EvaluationParameters, RLParameters
    from reagent_b200.optimizer import Optimizer__Union

    torch.manual_seed(seed)  # identical initial weights on every rank (replicated parameters)
    Sc, Ac, sizes = cfg["S"], cfg["A"], cfg["sizes"]
    opt = lambda: Optimizer__Union.default(lr=LR)  # noqa: E731
    rl = RLParameters(gamma=GAMMA, target_update_rate=TAU, q_network_loss="huber")
    if cfg["algo"] == "dqn":
        from reagent_b200.models import FullyConnectedDQN
        from reagent_b200.training import DQNTrainer

        q = FullyConnectedDQN(Sc, Ac, sizes, ACTS)
        qt = q.get_target_network()
        return DQNTrainer(q.to(dev), qt.to(dev), actions=[str(i) for i in range(Ac)], rl=rl,
                          double_q_learning=True, minibatch_size=cfg["B"], optimizer=opt(),
                          evaluation=EvaluationParameters(calc_cpe_in_training=False)).to(dev)
    if cfg["algo"] == "qrdqn":
        from reagent_b200.models import FullyConnectedDQN
        from reagent_b200.training import QRDQNTrainer

        q = FullyConnectedDQN(Sc, Ac, sizes, ACTS, num_atoms=cfg["N"])
        qt = q.get_target_network()
        return QRDQNTrainer(q.to(dev), qt.to(dev), actions=[str(i) for i in range(Ac)], rl=rl,
                            double_q_learning=True, num_atoms=cfg["N"], minibatch_size=cfg["B"],
                            optimizer=opt(),
                            evaluation=EvaluationParameters(calc_cpe_in_training=False)).to(dev)
    from reagent_b200.models import (FullyConnectedActor, FullyConnectedCritic,
                                     GaussianFullyConnectedActor)

    q1 = FullyConnectedCritic(Sc, Ac, sizes, ACTS)
    q2 = FullyConnectedCritic(Sc, Ac, sizes, ACTS)
    if cfg["algo"] == "sac":
        from reagent_b200.training import SACTrainer

        actor = GaussianFullyConnectedActor(Sc, Ac, sizes, ACTS)
        return SACTrainer(actor, q1, q2, rl=rl, q_network_optimizer=opt(),
                          actor_network_optimizer=opt(), alpha_optimizer=opt(),
                          minibatch_size=cfg["B"]).to(dev)
    from reagent_b200.training import TD3Trainer

    actor = FullyConnectedActor(Sc, Ac, sizes, ACTS)
    return TD3Trainer(actor, q1, q2, rl=rl, q_network_optimizer=opt(),
                      actor_network_optimizer=opt(), minibatch_size=cfg["B"],
                      delayed_policy_update=2).to(dev)


def param_tensors(trainer):
    return [p.detach() for p in trainer.parameters()]


DUMP_LIMIT_BYTES = 64 << 20


def last_update_outputs(name, trainer, out, batch):
    """What the last timed update hands its caller, as host arrays named `<name>.<field>`:
    the loss(es) train_batch returned, the replay indices of the batch it trained on (float64,
    exact below 2^53), the batch's Q-values where the trainer exposes them, and every parameter
    after the update."""
    arrays = {f"{name}.indices": batch.indices.reshape(-1).double()}
    for i, loss in enumerate(out if isinstance(out, tuple) else (out,)):
        if loss is not None:
            arrays[f"{name}.loss{i}"] = loss
    if getattr(trainer, "all_action_scores", None) is not None:
        arrays[f"{name}.all_action_scores"] = trainer.all_action_scores
    for pname, p in trainer.named_parameters():
        arrays[f"{name}.{pname}"] = p
    return {k: v.detach().cpu().numpy() for k, v in arrays.items()}


def dump_outputs(path, arrays):
    """Writes every array as `<path>/<name>.npy`."""
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (k, a.dtype)
        np.save(os.path.join(path, k + ".npy"), a)


def dp_check(env, cfg, rb):
    """N > 1: one data-parallel update (row shards, fused gradient exchange) against one
    full-global-batch update on a single rank, from identical parameters and identical draws.
    Returns the worst relative difference of the post-update parameters and the fraction of
    elements off by more than 1e-5 of the tensor's scale (Adam turns gradient elements within
    fp32 noise of zero into +-lr moves; those are counted, not hidden)."""
    import random

    import torch

    Bg = cfg["B"]
    lo, hi = env.shard(Bg)
    t_dp, t_full = build_trainer(cfg, env.dev, seed=7), build_trainer(cfg, env.dev, seed=7)
    state = random.getstate()
    random.seed(99)
    q, pos, _ = rb.host_queries(Bg)
    while pos:
        q, pos, _ = rb.host_queries(Bg)
    random.setstate(state)
    qd = torch.from_numpy(q).to(env.dev)

    def sample(qslice):
        n = qslice.shape[0]
        if cfg["algo"] in ("dqn", "qrdqn"):
            return rb.sample_discrete_dqn_batch(n, cfg["A"], query_dev=qslice)
        import numpy as np

        return rb.sample_policy_network_batch(n, -np.ones(cfg["A"], np.float32),
                                              np.ones(cfg["A"], np.float32), query_dev=qslice)

    if cfg["algo"] in ("sac", "td3"):
        g = torch.Generator(device=env.dev).manual_seed(5)
        noise = {k: torch.randn(Bg, cfg["A"], device=env.dev, generator=g) for k in ("next", "cur")}
        t_full.noise_hook = lambda name, shape, device: noise[name]
        t_dp.noise_hook = lambda name, shape, device: noise[name][lo:hi]
    t_full.train_batch(sample(qd))
    t_dp.train_batch(sample(qd[lo:hi].contiguous()), process_group=env.pg)
    torch.cuda.synchronize()
    worst, frac = 0.0, 0.0
    for a, b in zip(param_tensors(t_dp), param_tensors(t_full)):
        scale = float(b.abs().max()) + 1e-30
        d = (a.double() - b.double()).abs()
        worst = max(worst, float(d.max()) / scale)
        frac = max(frac, float((d > 1e-5 * scale).double().mean()))
    worst = env.max_over_ranks(worst)
    frac = env.max_over_ranks(frac)
    return {"what": "post-update parameters, data-parallel (N ranks) vs single-rank full batch, "
                    "one update from identical state", "max_rel_diff": worst,
            "frac_elements_off_by_1e-5": frac, "ok": bool(frac < 1e-3 and worst < 3 * LR)}


def run_dqn(env, args, clocks):
    """Config 2: value = K updates in one CUDA graph; e2e = FusedDqnStep.step(); roofline of K2."""
    import random

    import numpy as np
    import torch

    from reagent_b200.replay_memory import PrioritizedReplayBuffer
    from reagent_b200.training.fused_step import FusedDqnStep, capture_device_only

    cfg = CONFIGS[2]
    dev, world, pg = env.dev, env.world, env.pg
    K, W = args.steps, max(args.warmup, 3)
    Bg = cfg["B"]
    lo, hi = env.shard(Bg)
    Bl = hi - lo
    rb = PrioritizedReplayBuffer(stack_size=1, replay_capacity=cfg["cap"], batch_size=Bg, device=dev)
    rb.add_batch(**synth_stream(cfg["cap"], 1000, cfg))  # replicated: the same stream on every rank
    trainer = build_trainer(cfg, dev)
    random.seed(1234)  # the same host random stream on every rank -> the same global indices

    check = dp_check(env, cfg, rb) if world > 1 else None

    def timed_loop(step_fn):
        for i in range(W):
            step_fn(i)
        env.barrier()
        clocks.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(K):
            lh = step_fn(W + i)
        e1.record()
        env.barrier()
        t_host = time.perf_counter() - t0
        return env.max_over_ranks(max(e0.elapsed_time(e1), t_host * 1e3)), float(lh[0])

    # ---- e2e, host random numbers: host RNG -> pinned -> H2D (B*8 bytes), loss D2H ----
    fused = FusedDqnStep(trainer, rb, Bg, process_group=pg, prefetch=True, shard=(env.rank, world))
    hostrng_ms, _ = timed_loop(lambda i: fused.step())
    hostrng = {"value": K / (hostrng_ms * 1e-3), "ms_per_step": hostrng_ms / K,
               "h2d_bytes_per_step": fused.h2d_bytes, "d2h_bytes_per_step": fused.d2h_bytes,
               "api": "FusedDqnStep(prefetch=True).step(): the host draws the stratified query "
                      "values (Python `random`), pinned -> H2D, update, loss D2H"}
    del fused

    # ---- e2e (headline): the ONLINE loop through the public API.  Every step the host hands
    # over one new transition (pinned memory -> H2D inside the step), the step inserts it
    # (device-resident replay: validity + sum-tree update), draws the prioritized minibatch
    # with the device copy of Python's MT19937 stream (same indices as the reference), trains,
    # and copies the loss + status back -- one CUDA-graph replay per step ----
    extra = synth_stream(W + K + 4, 555, cfg)  # the same new transitions on every rank
    online = FusedDqnStep(trainer, rb, Bg, process_group=pg, prefetch=True,
                          shard=(env.rank, world), rng="device", online=True)
    e2e_ms, last_loss = timed_loop(
        lambda i: online.step({k: v[i] for k, v in extra.items()}))
    h2d_online, d2h_online = online.h2d_bytes, online.d2h_bytes
    online.dr.sync_to_host()  # the sections below use the host-side API again
    del online

    # ---- the drop-in surface, un-fused: sample_transition_batch -> InputMaker -> generator
    # protocol under the loop (what a user of the reference's workflow calls) ----
    dropin_ms = None
    if world == 1:
        from reagent_b200.gym.preprocessors.trainer_preprocessor import DiscreteDqnInputMaker
        from reagent_b200.training import run_update

        maker = DiscreteDqnInputMaker(num_actions=cfg["A"])
        nd = min(K, 50)
        for i in range(3 + nd):
            if i == 3:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            run_update(trainer, maker(rb.sample_transition_batch(batch_size=Bg)), i)
        torch.cuda.synchronize()
        dropin_ms = (time.perf_counter() - t0) / nd * 1e3

    # ---- roofline of the fused TD kernel: events around each launch, same workload ----
    trainer._kernel_events = []
    for _ in range(W):
        trainer.train_batch(rb.sample_discrete_dqn_batch(Bl, cfg["A"]), process_group=pg)
    trainer._kernel_events = []
    nroof = min(K, 100)
    for _ in range(nroof):
        batch = rb.sample_discrete_dqn_batch(Bl, cfg["A"])
        trainer.tc_prepack()  # keep the weight packing out of the event pair: TD kernel only
        # keep the stream busy while the host enqueues, otherwise the event pair would also
        # time the launch latency of an idle GPU
        torch.cuda._sleep(400_000)
        trainer.train_batch(batch, process_group=pg)
    torch.cuda.synchronize()
    on_tc = trainer._last_td_call[-1] is not None
    durs = [a.elapsed_time(b) for a, b in trainer._kernel_events]
    trainer._kernel_events = None
    kern_ms = sum(durs) / len(durs)

    # ---- value: K updates in one graph, random numbers resident in HBM ----
    def draw(n, nrows, sl):
        out = np.empty((n, sl.stop - sl.start), dtype=np.float64)
        for i in range(n):
            qv, pos, _ = rb.host_queries(nrows)
            # retry-free draws only: strata that would hit the not-yet-valid slot are redrawn
            # (the retry path is host logic, timed in e2e); keeps the graph free of overrides
            while pos:
                qv, pos, _ = rb.host_queries(nrows)
            out[i] = qv[sl]
        return torch.from_numpy(out).to(dev)

    q_warm, q_timed = draw(W, Bg, slice(lo, hi)), draw(K, Bg, slice(lo, hi))
    g_warm = capture_device_only(trainer, rb, Bl, W, q_warm, pg)
    g_timed = capture_device_only(trainer, rb, Bl, K, q_timed, pg)
    g_warm.replay()
    env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g_timed.replay()
    e1.record()
    env.barrier()
    dev_ms = env.max_over_ranks(e0.elapsed_time(e1))
    outputs = None
    if args.dump_outputs:
        # the graph's last update trained on the last batch it keeps; the loss is the
        # workspace scalar train_batch returns
        outputs = last_update_outputs("dqn", trainer, trainer._ws["loss"], g_timed._rb200_keep[-1])

    # ---- weak scaling (secondary): 4096 rows per rank, rank-specific draws ----
    weak = None
    if world > 1:
        tw = build_trainer(cfg, dev)
        random.seed(4321 + env.rank)
        # one eager update first: lazy allocations (workspaces, the optimizer's slice of the
        # peer-memory pool) must not happen inside the graph capture
        tw.train_batch(rb.sample_discrete_dqn_batch(Bg, cfg["A"]), process_group=pg)
        torch.cuda.synchronize()
        qw, qt_ = draw(W, Bg, slice(0, Bg)), draw(K, Bg, slice(0, Bg))
        gw = capture_device_only(tw, rb, Bg, W, qw, pg)
        gt = capture_device_only(tw, rb, Bg, K, qt_, pg)
        gw.replay()
        env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gt.replay()
        e1.record()
        env.barrier()
        wms = env.max_over_ranks(e0.elapsed_time(e1))
        weak = {"rows_per_rank": Bg, "updates_per_s_4096_row_shards": world * K / (wms * 1e-3),
                "ms_per_step": wms / K}

    conf = base_config(cfg, world)
    detail = dict(value_path="K updates in one CUDA graph, query values resident in HBM; "
                             "retry-free draws only (PER retries are host logic, timed in e2e)",
                  final_loss=last_loss, rows_per_rank=Bl, e2e_host_rng=hostrng)
    if weak:
        detail["weak"] = weak
    if env.collective:
        detail["collective"] = env.collective
    if dropin_ms is not None:
        detail["dropin_unfused"] = {
            "ms_per_step": dropin_ms, "updates_per_s": 1e3 / dropin_ms,
            "api": "rb.sample_transition_batch -> DiscreteDqnInputMaker -> train_step_gen under "
                   "training.run_update (the reference workflow's own calls, eager launches)"}
    flops = td_kernel_flops(cfg, Bl)
    res = {
        "value": K / (dev_ms * 1e-3), "ms_per_step": dev_ms / K, "config": conf, "detail": detail,
        "e2e": {"value": K / (e2e_ms * 1e-3), "unit": "updates/s",
                "h2d_bytes_per_step": h2d_online, "d2h_bytes_per_step": d2h_online,
                "ms_per_step": e2e_ms / K,
                "api": "reagent_b200.training.fused_step.FusedDqnStep(rng='device', online=True, "
                       "prefetch=True).step(transition): per step the host stages ONE new "
                       "transition in pinned memory; the captured step copies it to the device, "
                       "inserts it into the replay buffer, draws the minibatch (device MT19937 = "
                       "Python's random stream), trains and returns the loss; the sampler runs one "
                       "update ahead on a second stream"},
        # sample, (weight images unless Adam wrote them), TD step, weight gradients, Adam+Polyak
        "gpu_launches": (4 if (not on_tc or os.environ.get("RB200_ADAM_PACK", "1") == "1") else 5) * K,
        "roofline_kernel": {
            "kernel": ("dqn_td_tc_kernel (fused TD target + loss + dZ chain on tcgen05/TMEM)"
                       if on_tc else "dqn_td_rows_kernel (fused TD target + loss + dZ chain, mma.sync)"),
            "flops": flops, "kernel_ms": kern_ms,
            "pipe_used": ("tcgen05.mma kind::tf32, 3xTF32 as 2 MMAs per k step (N=64 + N=32)"
                          if on_tc else "mma.sync m16n8k8 tf32, 3xTF32"),
            "ncu_file": "profiles/r02_ncu_dqn_td_tc.csv" if on_tc else None},
    }
    if check:
        res["dp_check"] = check
    if outputs is not None:
        res["outputs"] = outputs
    return res


def run_generic(env, args, cfg):
    """Configs 3-5: eager launches; value = K updates device-timed with the random numbers
    resident in HBM; e2e = sample (host RNG -> H2D) + train_batch + loss D2H per update."""
    import random

    import numpy as np
    import torch

    from reagent_b200.replay_memory import PrioritizedReplayBuffer

    dev, world, pg = env.dev, env.world, env.pg
    K = args.steps
    W = 3
    Bg = cfg["B"]
    lo, hi = env.shard(Bg)
    Bl = hi - lo
    rb = PrioritizedReplayBuffer(stack_size=1, replay_capacity=cfg["cap"], batch_size=Bg, device=dev)
    rb.add_batch(**synth_stream(cfg["cap"], 1000, cfg))
    trainer = build_trainer(cfg, dev)
    random.seed(1234)
    cont = cfg["algo"] in ("sac", "td3")
    low, high = -np.ones(cfg["A"], np.float32), np.ones(cfg["A"], np.float32)
    check = dp_check(env, cfg, rb) if world > 1 else None

    def sample(qslice=None):
        if qslice is None:  # public path: host RNG inside, H2D of the query values
            q, pos, idxs = rb.host_queries(Bg)
            kw = dict(query_dev=torch.from_numpy(np.ascontiguousarray(q[lo:hi])).pin_memory().to(dev, non_blocking=True))
            if pos:
                keep = [(p - lo, i) for p, i in zip(pos, idxs) if lo <= p < hi]
                if keep:
                    kw["overrides"] = ([p for p, _ in keep], [i for _, i in keep])
        else:
            kw = dict(query_dev=qslice)
        if cont:
            return rb.sample_policy_network_batch(Bl, low, high, **kw)
        return rb.sample_discrete_dqn_batch(Bl, cfg["A"], **kw)

    def loss_of(out):
        return (out[0][0] if isinstance(out, tuple) else out).reshape(-1)[:1]

    # ---- e2e ----
    loss_pin = torch.zeros(1).pin_memory()
    for i in range(W):
        trainer.train_batch(sample(), i, process_group=pg)
    env.barrier()
    t0 = time.perf_counter()
    for i in range(K):
        out = trainer.train_batch(sample(), W + i, process_group=pg)
        loss_pin.copy_(loss_of(out), non_blocking=True)
    torch.cuda.synchronize()
    env.barrier()
    e2e_ms = env.max_over_ranks((time.perf_counter() - t0) * 1e3)
    last_loss = float(loss_pin[0])

    # ---- value ----
    def draw(n):
        out = np.empty((n, Bl), dtype=np.float64)
        for i in range(n):
            qv, pos, _ = rb.host_queries(Bg)
            while pos:
                qv, pos, _ = rb.host_queries(Bg)
            out[i] = qv[lo:hi]
        return torch.from_numpy(out).to(dev)

    qs = draw(W + K)
    trainer._kernel_events = [] if hasattr(trainer, "_critic_step") else None
    for i in range(W):
        trainer.train_batch(sample(qs[i]), i, process_group=pg)
    if trainer._kernel_events is not None:
        trainer._kernel_events = []
    env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        batch = sample(qs[W + i])
        out = trainer.train_batch(batch, W + i, process_group=pg)
    e1.record()
    env.barrier()
    dev_ms = env.max_over_ranks(e0.elapsed_time(e1))
    outputs = last_update_outputs(cfg["algo"], trainer, out, batch) if args.dump_outputs else None
    kern_ms = None
    if getattr(trainer, "_kernel_events", None):
        durs = [a.elapsed_time(b) for a, b in trainer._kernel_events]
        kern_ms = sum(durs) / len(durs)
    trainer._kernel_events = None
    nlaunch = {"qrdqn": 15, "sac": 12, "td3": 9}[cfg["algo"]]
    conf = base_config(cfg, world)
    detail = dict(value_path="K updates, eager launches, device-timed, query values resident in HBM",
                  final_loss=last_loss, rows_per_rank=Bl)
    if env.collective:
        detail["collective"] = env.collective
    res = {
        "value": K / (dev_ms * 1e-3), "ms_per_step": dev_ms / K, "steps": K, "warmup": W,
        "config": conf, "detail": detail,
        "e2e": {"value": K / (e2e_ms * 1e-3), "unit": "updates/s", "h2d_bytes_per_step": Bl * 8,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / K,
                "api": "rb.sample_%s_batch(...) (host RNG -> pinned -> H2D -> sample kernel) + "
                       "trainer.train_batch(batch) + loss D2H, every update"
                       % ("policy_network" if cont else "discrete_dqn")},
        "gpu_launches": nlaunch * K,
    }
    if kern_ms is not None:
        res["roofline_kernel"] = {
            "kernel": "ac_critic_rows_kernel (fused %s TD target: actor(s') + target critics + "
                      "min + losses + critic dZ chains, mma.sync 3xTF32)" % cfg["algo"].upper(),
            "flops": td_kernel_flops(cfg, Bl), "kernel_ms": kern_ms,
            "pipe_used": "mma.sync m16n8k8 tf32, 3xTF32", "ncu_file": None}
    elif cfg["algo"] == "qrdqn":
        res["roofline_kernel"] = {
            "kernel": "whole QR-DQN update (tc_linear_fwd_kernel on tcgen05: head forward x3 and the "
                      "split-K head backward; qr_head_kernel, wgrad_kernel, adam_soft_kernel)",
            "flops": update_flops(cfg, Bl), "kernel_ms": dev_ms / K,
            "pipe_used": "tcgen05 kind::tf32 (head forward + head dX) + mma.sync tf32 (trunk, wgrad)",
            "ncu_file": None}
    if check:
        res["dp_check"] = check
    if outputs is not None:
        res["outputs"] = outputs
    return res


def roofline_of(rk, peaks):
    if not rk or not rk.get("flops"):
        return None
    peak_tf = float(peaks.get("bf16_tflops", 1700.0))
    src = ("measured (MEASURED_PEAKS.json bf16_tflops, burst: the kernel is timed alone between "
           "events)" if peaks else "fallback 1.7 PF/s")
    ach = rk["flops"] / (rk["kernel_ms"] * 1e-3) / 1e12
    traffic, tsrc = None, None
    if rk.get("ncu_file"):
        try:  # dram bytes of one ncu --set full launch of this kernel, read from the profile
            import csv

            with open(os.path.join(ROOT, rk["ncu_file"])) as f:
                rows = {r[0]: r for r in csv.reader(f) if r}
            rd = float(rows["dram__bytes_read.sum"][2]) * {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1, "Gbyte": 1e9}[rows["dram__bytes_read.sum"][1]]
            wr = float(rows["dram__bytes_write.sum"][2]) * {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1, "Gbyte": 1e9}[rows["dram__bytes_write.sum"][1]]
            traffic = rd + wr
            tsrc = f"dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full launch ({rk['ncu_file']}), bytes"
        except Exception:
            traffic = None
    return {"kernel": rk["kernel"], "bound": "tensor", "achieved": ach, "peak": peak_tf,
            "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": traffic, "traffic_source": tsrc,
            "peak_source": src, "algorithmic_flops_per_launch": rk["flops"],
            "kernel_ms": rk["kernel_ms"], "pipe_used": rk["pipe_used"],
            "executed_over_algorithmic_flops": 3.0,
            "frac_of_3xtf32_ceiling": ach / (peak_tf / 6.0),
            "note": "fp32-parity (1e-5) forces 3xTF32: 3 tensor-core flops per algorithmic flop, "
                    "and TF32 dense peak is half the bf16 peak this fraction is quoted against"}


def run_ours(args):
    env = Env()
    clocks = ClockSampler(env.local)
    clocks.start()  # started before any warm-up: nvidia-smi takes ~1 s to produce its first row
    cfg = CONFIGS[args.config]
    res = run_dqn(env, args, clocks) if cfg["algo"] == "dqn" else run_generic(env, args, cfg)
    extra = []
    if args.config == 2 and env.world == 1 and not args.only:
        for c in (3, 4, 5):
            r = run_generic(env, args, CONFIGS[c])
            r["_cfg"] = c
            extra.append(r)
    clk = clocks.stop()

    # ---- cpu baseline (rank 0, N == 1 only).  Runs LAST: its worker threads would otherwise
    # keep spinning on the host cores while the e2e loops (host-paced) are being timed ----
    cpu = {}
    if env.world == 1 and not args.no_cpu_baseline:
        for c in [args.config] + [r["_cfg"] for r in extra]:
            cc = CONFIGS[c]
            v, cores, sample, _ = cpu_reference_run(_cpu_steps(cc, args.cpu_steps), 1 if c != 2 else 2, cc)
            cpu[c] = {"value": v, "unit": "updates/s", "cores": cores, "kind": "port", "sample": sample}
    if env.rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for r in [res] + extra for k, v in r["outputs"].items()})
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass

    def finish(r, c):
        out = {"metric": CONFIGS[c]["metric"], "value": r["value"], "unit": "updates/s",
               "ms_per_step": r["ms_per_step"], "config": r["config"], "e2e": r["e2e"],
               "gpu_launches": r["gpu_launches"], "detail": r["detail"]}
        rl = roofline_of(r.get("roofline_kernel"), peaks)
        if rl:
            out["roofline"] = rl
        if c in cpu:
            out["cpu_baseline"] = cpu[c]
        if "dp_check" in r:
            out["dp_check"] = r["dp_check"]
        return out

    main = finish(res, args.config)
    line = {
        "metric": main["metric"], "value": main["value"], "unit": "updates/s", "n_gpus": env.world,
        "steps": res.get("steps", args.steps), "warmup": res.get("warmup", max(args.warmup, 3)),
        "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": main["config"],
        "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "clocks": clk,
    }
    for k in ("roofline", "cpu_baseline", "dp_check", "detail"):
        if k in main:
            line[k] = main[k]
    if extra:
        line["configs"] = [dict(finish(r, r["_cfg"]), steps=r["steps"], warmup=r["warmup"],
                                n_gpus=1, note="global batch of this config on ONE GPU")
                           for r in extra]
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--only", action="store_true", help="config 2: skip the configs 3-5 array")
    ap.add_argument("--cpu-steps", type=int, default=60)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed update of each config "
                         "computed (loss, sampled indices, Q-values, parameters) as DIR/<name>.npy; "
                         "inputs are seeded, so runs with the same arguments are comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        try:
            run_ours(args)
        finally:
            import torch.distributed as dist

            if dist.is_available() and dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
