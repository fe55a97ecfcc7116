#!/usr/bin/env python
"""bench.py -- learner env-steps/sec on the Atari 84x84x4 hot path (BASELINE.json metric).

  --workload ppo     (default) C2 breakout_ppo.yaml at E=32: per iteration T=128 batched inference calls over the E stacked
                     observations, GAE over [E,T], PPO.train = 4 epochs x 13 shuffled minibatches of 320 (52 SGD steps).
                     N>1: E=32 envs PER rank (weak scaling), gradients all-reduced in-graph every SGD step.
  --workload ppo-c5  C5: E=512, BATCH_SIZE=4096 (N=65536, 64 SGD steps); N>1 shards the 512 envs and every minibatch
                     over the ranks (strong scaling, 4096/N samples per rank per step).
  --workload impala  C3 breakout_impala.yaml at E=64: T=128 inference calls (B=64) + 16 V-trace SGD steps of
                     4 trajectories x 128 steps (B*T = 512).
  --workload dqn     C4 breakout_dqn.yaml, batch 512: 32 SGD steps on a 2^16-transition device replay + the 4 batched
                     greedy-action calls (B=32) that produce the 128 transitions those steps consume (1 step / 4 transitions).

  value : samples consumed / device time, rollout already resident in HBM (synthetic, seeded)
  e2e   : the same iteration through the reference-facing plugin API (Algorithm.predict / prepare_data / train) with
          HOST numpy buffers; H2D/D2H inside the timed region
  --impl reference : the CPU restatement of the reference learner (oracle/) on the host cores, same workload
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A = 4
STATE = (84, 84, 4)
METRIC = "learner env-steps/sec (Atari 84x84x4 PPO)"


def metric_name(workload):
    """BASELINE.json's metric for the PPO workloads; the IMPALA / DQN lines name their algorithm."""
    return METRIC.replace("PPO", {"impala": "IMPALA", "dqn": "DQN"}.get(workload, "PPO"))

WORKLOADS = {
    "ppo": dict(kind="ppo", E=32, T=128, B=320, epochs=4, scaling="weak", flop_per_env_step=164e6,
                cpu_sample=dict(infer=128, sgd=52),
                desc="breakout_ppo C2: PpoCnn E=32 T=128 N=4096 B=320 x4 epochs (52 SGD steps) + 128 batched inference calls + GAE"),
    "ppo-c5": dict(kind="ppo", E=512, T=128, B=4096, epochs=4, scaling="strong", flop_per_env_step=164e6,
                   cpu_sample=dict(infer=8, sgd=4),
                   desc="breakout_ppo C5: PpoCnn E=512 T=128 N=65536 B=4096 x4 epochs (64 SGD steps) + 128 batched inference calls (B=512) + GAE"),
    "impala": dict(kind="impala", E=64, T=128, B=512, scaling="weak", flop_per_env_step=7.57e6 * 4,
                   cpu_sample=dict(infer=128, sgd=16),
                   desc="breakout_impala C3: ImpalaCnnOpt E=64 T=128 N=8192, 16 V-trace SGD steps of 4x128 samples + 128 batched inference calls (B=64)"),
    "dqn": dict(kind="dqn", E=32, B=512, replay=1 << 16, train_steps=32, scaling="weak", flop_per_env_step=85.5e6 * 128,
                cpu_sample=dict(infer=4, sgd=4),
                desc="breakout_dqn C4: DqnCnn batch 512, 32 SGD steps on a 65536-transition device replay + 4 greedy-action calls (B=32) = 128 env steps"),
}
PPO_CFG = {"CRITIC_LOSS_COEF": 1.0, "ENTROPY_LOSS": 0.003, "LOSS_CLIPPING": 0.1, "LR": 0.00025, "MAX_GRAD_NORM": 5.0,
           "SUMMARY": False, "VF_SHARE_LAYERS": True, "activation": "relu", "hidden_sizes": [256],
           "action_type": "Categorical", "init_seed": 0}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf=p["bf16_tflops"], tf_sus=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def samples_per_iteration(wl):
    if wl["kind"] == "dqn":
        return 4 * wl["train_steps"]
    return wl["E"] * wl["T"]


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's restatement of the reference learner on host cores
# ------------------------------------------------------------------------------------------------
def cpu_threads():
    """Fixed thread count (stable run to run): all host cores up to 32 -- the small convolutions of these networks stop
    scaling beyond that in torch-CPU and oversubscription only adds variance."""
    return max(1, min(32, os.cpu_count() or 1))


def make_cpu_state(name):
    import torch
    from oracle import xt_oracle as orc
    from xingtian_b200 import synth
    wl = WORKLOADS[name]
    torch.set_num_threads(cpu_threads())
    st = dict(wl=wl, name=name, threads=cpu_threads())
    if wl["kind"] == "ppo":
        arch = orc.ppo_cnn_arch()     # C5: the bounded sample draws its calls from a 32-env rollout
        st.update(arch=arch, ro=synth.ppo_rollout(0, wl["E"] if name != "ppo-c5" else 32, wl["T"]),
                  learner=orc.PpoLearner(arch, orc.init_weights(arch, seed=0), lr=0.00025, batch_size=wl["B"], ent_coef=0.003,
                                         clip_ratio=0.1, num_sgd_iter=wl["epochs"]))
    elif wl["kind"] == "impala":
        arch = orc.impala_cnn_arch()
        st.update(arch=arch, ro=synth.ppo_rollout(0, wl["E"], wl["T"]),
                  learner=orc.ImpalaLearner(arch, orc.init_weights(arch, seed=0, baseline_norm_std=0.01), lr=0.0005, sample_batch_step=wl["T"]))
    else:
        arch = orc.dqn_cnn_arch()
        st.update(arch=arch, tr=synth.replay_transitions(0, 4096), learner=orc.DqnLearner(arch, orc.init_weights(arch, seed=0)))
    return st


def cpu_iteration(st, full=True):
    """One iteration of the workload on the CPU; workloads whose full iteration would take minutes run the bounded
    sample of WORKLOADS[..]['cpu_sample'] and are extrapolated from the measured per-call times.  Returns seconds."""
    import torch
    from oracle import xt_oracle as orc
    wl, learner, arch = st["wl"], st["learner"], st["arch"]
    smp = wl["cpu_sample"]
    rng = np.random.default_rng(0)
    if wl["kind"] == "ppo":
        ro = st["ro"]
        E_ro = ro["value"].shape[0]
        T, B = wl["T"], wl["B"]
        w = dict(zip(learner.names, learner.params))
        n_inf_total, n_sgd_total = T, wl["epochs"] * ((wl["E"] * T + B - 1) // B)
        u = rng.random((wl["E"], A)).astype(np.float32) * 0.998 + 0.001
        t0 = time.perf_counter()
        with torch.no_grad():
            for t in range(smp["infer"]):
                rows = (np.arange(wl["E"]) % E_ro) * T + (t % T)
                logits, v = orc.forward(arch, w, ro["obs"][rows])
                orc.gumbel_argmax(logits.numpy(), u)
        t_inf = (time.perf_counter() - t0) / smp["infer"]
        t0 = time.perf_counter()
        advs = [orc.gae(ro["value"][e], ro["reward"][e * T:(e + 1) * T], ro["done"][e * T:(e + 1) * T]) for e in range(E_ro)]
        t_gae = (time.perf_counter() - t0) * wl["E"] / E_ro
        adv = np.concatenate([a[0] for a in advs]).astype(np.float32)
        ov = np.concatenate([a[1] for a in advs]); tv = np.concatenate([a[2] for a in advs]).astype(np.float32)
        n_ro = E_ro * T
        t0 = time.perf_counter()
        for s in range(smp["sgd"]):
            mb = rng.integers(0, n_ro, min(B, wl["E"] * T))
            learner.sgd_step(ro["obs"][mb], ro["action"][mb], ro["logp"][mb], adv[mb], ov[mb], tv[mb])
        t_sgd = (time.perf_counter() - t0) / smp["sgd"]
        return t_inf * n_inf_total + t_gae + t_sgd * n_sgd_total
    if wl["kind"] == "impala":
        ro = st["ro"]
        E, T = wl["E"], wl["T"]
        w = dict(zip(learner.names, learner.params))
        t0 = time.perf_counter()
        with torch.no_grad():
            for t in range(smp["infer"]):
                rows = np.arange(E) * T + (t % T)
                logits, base = orc.forward(arch, w, ro["obs"][rows])
                orc.gumbel_argmax(logits.numpy(), rng.random((E, A)).astype(np.float32) * 0.998 + 0.001)
        t_inf = (time.perf_counter() - t0) / smp["infer"]
        k = wl["B"] // T
        t0 = time.perf_counter()
        for s in range(smp["sgd"]):
            sl = slice(s * k * T, (s + 1) * k * T)
            learner.train(ro["obs"][sl], [ro["logits"][sl], ro["action"][sl], ro["done"][sl], ro["reward"][sl].astype(np.float32)])
        t_sgd = (time.perf_counter() - t0) / smp["sgd"]
        return t_inf * T + t_sgd * (E // k)
    tr = st["tr"]
    B = wl["B"]
    t0 = time.perf_counter()
    for t in range(smp["infer"]):
        np.argmax(learner.predict(tr["obs"][t * wl["E"]:(t + 1) * wl["E"]]), 1)
    t_inf = (time.perf_counter() - t0) / smp["infer"]
    t0 = time.perf_counter()
    for s in range(smp["sgd"]):
        mb = rng.integers(0, len(tr["action"]), B)
        learner.train(tr["obs"][mb], tr["action"][mb], tr["reward"][mb], tr["next_obs"][mb], tr["done"][mb])
    t_sgd = (time.perf_counter() - t0) / smp["sgd"]
    return t_inf * 4 + t_sgd * wl["train_steps"]


def sample_desc(name):
    wl = WORKLOADS[name]
    smp = wl["cpu_sample"]
    full = {"ppo": (128, 52), "ppo-c5": (128, 64), "impala": (128, 16), "dqn": (4, 32)}[name]
    if (smp["infer"], smp["sgd"]) == full:
        return "the full iteration (%d inference calls + %d SGD steps); torch-CPU fp32 restatement of the reference learner (oracle/), %d threads" % (
            full[0], full[1], cpu_threads())
    return ("%d of %d inference calls + %d of %d SGD steps, extrapolated to the full iteration from the measured per-call times; "
            "torch-CPU fp32 restatement of the reference learner (oracle/), %d threads" % (smp["infer"], full[0], smp["sgd"], full[1], cpu_threads()))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    st = make_cpu_state(args.workload)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_iteration(st)
    times = [cpu_iteration(st) for _ in range(args.steps)]
    t = float(np.mean(times))
    val = samples_per_iteration(wl) / t
    out = {"impl": "reference", "metric": metric_name(args.workload), "value": val, "unit": "env-steps/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
           "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": wl["desc"]},
           "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": st["threads"], "host_cpus": os.cpu_count(), "kind": "port",
                            "sample": sample_desc(args.workload)},
           "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "note": "one CPU process on rank 0 regardless of --gpus"}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------
# B200 arm: per-workload device-resident iteration and plugin-API (host buffer) iteration
# ------------------------------------------------------------------------------------------------
class PpoBench(object):
    def __init__(self, wl, rank, world, dev, local):
        import torch
        import xingtian_b200 as xb
        from xingtian_b200 import synth
        self.wl, self.world = wl, world
        strong = wl["scaling"] == "strong"
        self.E = wl["E"] // world if strong else wl["E"]
        self.T, self.B = wl["T"], (wl["B"] // world if strong else wl["B"])
        if strong and (wl["E"] % world or wl["B"] % world):
            raise SystemExit("ppo-c5 needs a rank count that divides 512 envs and the 4096-sample minibatch")
        cfg = dict(PPO_CFG, BATCH_SIZE=self.B, NUM_SGD_ITER=wl["epochs"])
        info = {"actor": {"model_name": "PpoCnn", "state_dim": list(STATE), "action_dim": A, "input_dtype": "uint8",
                          "model_config": cfg, "device": "cuda:%d" % local, "max_predict_batch": max(self.B, self.E)}}
        self.alg = xb.alg_builder("PPO", info, {"instance_num": self.E, "agent_num": 1})
        self.model = self.alg.actor
        E, T = self.E, self.T
        self.n = E * T
        # rollouts: distinct seeds per rank; large E is tiled from a 64-env rollout to bound host memory
        base = synth.ppo_rollout(rank, min(E, 64), T)
        rep = (E + min(E, 64) - 1) // min(E, 64)
        self.ro = {k: (np.concatenate([v] * rep)[:(E * T if k != "value" else E)] if rep > 1 else v) for k, v in base.items()}
        store = self.model.rollout
        store.reserve(self.n)
        store.obs[:self.n].copy_(torch.from_numpy(self.ro["obs"]))
        self.store = store
        self.reward_d = torch.from_numpy(self.ro["reward"].astype(np.float32)).to(dev)
        self.done_d = torch.from_numpy(self.ro["done"].view(np.uint8)).to(dev)
        self.value_d = torch.zeros(E, T + 1, device=dev)
        self.step_idx = (torch.arange(E, dtype=torch.int32, device=dev)[None, :] * T + torch.arange(T, dtype=torch.int32, device=dev)[:, None]).contiguous()
        self.act_t = torch.empty(T, E, dtype=torch.int32, device=dev); self.logp_t = torch.empty(T, E, device=dev)
        self.val_t = torch.empty(T + 1, E, device=dev)
        self.alg.sign_clip_reward = True
        self.train_batch = self.B
        self.h2d = 2 * self.n * int(np.prod(STATE)) + self.n * (4 + 4 + 4 + 1) + E * 4 + wl["epochs"] * self.n * 4
        self.d2h = T * E * 12 + wl["epochs"] * ((self.n + self.B - 1) // self.B) * 4

    def device_iteration(self, ev=None):
        import torch
        from xingtian_b200 import capi
        from xingtian_b200.engine import _ptr, stream_ptr
        m, st, E, T, n = self.model, self.store, self.E, self.T, self.n
        if ev: ev[0].record()
        m.rollout_infer_device(st.obs, self.step_idx, E, T, self.act_t, self.logp_t, self.val_t)
        self.val_t[T].copy_(self.val_t[T - 1])            # bootstrap value (synthetic rollout: no next observation)
        st.action[:n].copy_(self.act_t.t().reshape(-1)); st.old_logp[:n].copy_(self.logp_t.t().reshape(-1))
        self.value_d.copy_(self.val_t.t())
        if ev: ev[1].record()
        capi.check(capi.lib().xtb_gae(_ptr(self.value_d), _ptr(self.reward_d), _ptr(self.done_d), E, T, 0.99, 0.95, 1,
                                      _ptr(st.adv), _ptr(st.old_v), _ptr(st.target_v), stream_ptr()))
        if ev: ev[2].record()
        loss = m.train_device(n)
        if ev: ev[3].record()
        return loss

    def outputs(self):
        """What the last device_iteration handed its caller: sampled actions, log-probs and values [T, E], GAE advantages
        and value targets [E*T], the loss of every SGD step and the trained weights."""
        st, n = self.store, self.n
        return dict(action=self.act_t, logp=self.logp_t, value=self.val_t[:self.T], adv=st.adv[:n], target_v=st.target_v[:n],
                    loss=self.model.last_losses, weights=self.model.get_weights())

    def e2e_setup(self):
        E, T, ro = self.E, self.T, self.ro
        self.host_obs = [np.ascontiguousarray(ro["obs"][np.arange(E) * T + t]) for t in range(T)]
        self.traj = []
        # the frames reach the device once, inside predict(): trajectories refer to them by (env, first step, steps)
        self.model.keep_predict_obs(E, T)
        for e in range(E):
            sl = slice(e * T, (e + 1) * T)
            self.traj.append(dict(ring_rows=(e, 0, T), action=ro["action"][sl], logp=ro["logp"][sl],
                                  value=ro["value"][e], reward=ro["reward"][sl], done=ro["done"][sl]))
        self.h2d -= self.n * int(np.prod(STATE))

    def e2e_iteration(self):
        self.model._obs_ring["t"] = 0
        for t in range(self.T):
            self.model.predict(self.host_obs[t])           # H2D obs (kept in the device ring), D2H (action, logp, value)
        for e in range(self.E):
            self.alg.prepare_data(self.traj[e])            # H2D trajectory (pinned ring), device GAE
        return self.alg.train()                            # D2H loss trace


class ImpalaBench(object):
    def __init__(self, wl, rank, world, dev, local):
        import torch
        import xingtian_b200 as xb
        from xingtian_b200 import synth
        self.wl, self.world = wl, world
        self.E, self.T, self.B = wl["E"], wl["T"], wl["B"]
        info = {"actor": {"model_name": "ImpalaCnnOpt", "state_dim": list(STATE), "action_dim": A, "input_dtype": "uint8",
                          "state_mean": 0.0, "state_std": 255.0, "max_batch": self.B, "device": "cuda:%d" % local,
                          "model_config": {"LR": 0.0005, "sample_batch_step": self.T, "grad_norm_clip": 40.0, "init_seed": 0}}}
        self.alg = xb.alg_builder("IMPALAOpt", info, {"instance_num": self.E, "agent_num": 1, "BATCH_SIZE": self.B})
        self.model = self.alg.actor
        E, T = self.E, self.T
        self.n = E * T
        self.ro = synth.ppo_rollout(rank, E, T)
        self.obs = torch.from_numpy(self.ro["obs"]).to(dev)
        self.bp = torch.from_numpy(self.ro["logits"]).to(dev)
        self.action = torch.from_numpy(self.ro["action"]).to(dev)
        self.done = torch.from_numpy(self.ro["done"].view(np.uint8)).to(dev)
        self.reward = torch.from_numpy(self.ro["reward"].astype(np.float32)).to(dev)
        self.step_idx = (torch.arange(E, dtype=torch.int32, device=dev)[None, :] * T + torch.arange(T, dtype=torch.int32, device=dev)[:, None]).contiguous()
        self.act_t = torch.empty(T, E, dtype=torch.int32, device=dev); self.logp_t = torch.empty(T, E, device=dev)
        self.val_t = torch.empty(T, E, device=dev)
        self.loss = torch.zeros(1, device=dev)
        self.train_batch = self.B
        self.h2d = 2 * self.n * int(np.prod(STATE)) + self.n * (A * 4 + 4 + 1 + 4)
        self.d2h = T * E * (A * 4 + 4 + 4) + (self.n // self.B) * 4

    def device_iteration(self, ev=None):
        import torch
        from xingtian_b200 import capi
        from xingtian_b200.engine import _ptr, stream_ptr
        m, E, T = self.model, self.E, self.T
        net = m.net
        if ev: ev[0].record()
        # batched policy inference of the actors' T steps: one CUDA graph (forward + fused heads + Philox sampling per step)
        m.rollout_infer_device(self.obs, self.step_idx, E, T, self.act_t, self.logp_t, self.val_t)
        if ev: ev[1].record()
        if ev: ev[2].record()
        for s in range(self.n // self.B):
            sl = slice(s * self.B, (s + 1) * self.B)
            m.train_device(self.obs[sl], self.bp[sl], self.action[sl], self.done[sl], self.reward[sl], self.B, self.loss)
        if ev: ev[3].record()
        return self.loss

    def outputs(self):
        """Sampled actions, log-probs and values [T, E] of the last iteration, the loss of its last SGD step and the
        trained weights."""
        return dict(action=self.act_t, logp=self.logp_t, value=self.val_t, loss=self.loss, weights=self.model.get_weights())

    def e2e_setup(self):
        E, T, ro = self.E, self.T, self.ro
        self.host_obs = [np.ascontiguousarray(ro["obs"][np.arange(E) * T + t]) for t in range(T)]
        self.traj = []
        for e in range(E):
            sl = slice(e * T, (e + 1) * T)
            self.traj.append(dict(cur_state=ro["obs"][sl], logit=ro["logits"][sl], action=ro["action"][sl],
                                  reward=ro["reward"][sl].astype(np.float32), done=ro["done"][sl]))

    def e2e_iteration(self):
        for t in range(self.T):
            self.alg.predict(self.host_obs[t])
        for e in range(self.E):
            self.alg.prepare_data(self.traj[e])
        return self.alg.train()


class DqnBench(object):
    def __init__(self, wl, rank, world, dev, local):
        import torch
        import xingtian_b200 as xb
        from xingtian_b200 import synth
        self.wl, self.world = wl, world
        self.E, self.B, self.steps = wl["E"], wl["B"], wl["train_steps"]
        info = {"actor": {"model_name": "DqnCnn", "state_dim": list(STATE), "action_dim": A, "input_dtype": "uint8",
                          "max_batch": self.B, "device": "cuda:%d" % local, "model_config": {"LR": 0.00015, "init_seed": 0}}}
        self.alg = xb.alg_builder("DQN", info, {"instance_num": self.E, "agent_num": 1, "BATCH_SIZE": self.B,
                                                "BUFFER_SIZE": wl["replay"]})
        self.model = self.alg.actor
        tr = synth.replay_transitions(rank, 4096)
        reps = wl["replay"] // 4096
        for _ in range(reps):                               # fill the ring with 2^16 transitions
            self.alg.prepare_data(dict(cur_state=tr["obs"], action=tr["action"], reward=tr["reward"], next_state=tr["next_obs"], done=tr["done"]))
        self.tr = tr
        rng = np.random.default_rng(rank)
        self.idx = torch.from_numpy(rng.integers(0, wl["replay"], (self.steps, self.B)).astype(np.int32)).to(dev)
        self.idx_cur = torch.empty(self.B, dtype=torch.int32, device=dev)     # fixed address: one captured graph serves every step
        self.n = 4 * self.steps
        self.loss = torch.zeros(1, device=dev)
        self.act = torch.empty(self.E, dtype=torch.int32, device=dev)
        self.train_batch = self.B
        self.h2d = self.n * 2 * int(np.prod(STATE)) + self.n * (4 + 4 + 1) + 4 * self.E * int(np.prod(STATE)) + self.steps * self.B * 4
        self.d2h = 4 * self.E * A * 4 + self.steps * 4

    def device_iteration(self, ev=None):
        from xingtian_b200 import capi
        from xingtian_b200.engine import _ptr, stream_ptr
        m, b = self.model, self.alg.buff
        if ev: ev[0].record()
        for t in range(4):                                  # greedy actions for the next 4 x E env steps
            q = m.forward_device(b.obs[t * self.E:(t + 1) * self.E], self.E)
            capi.check(m.net.lib.xtb_argmax(_ptr(q), self.E, A, _ptr(self.act), stream_ptr()))
        if ev: ev[1].record()
        if ev: ev[2].record()
        for s in range(self.steps):
            self.idx_cur.copy_(self.idx[s])
            m.train_td_device(self.alg.target_actor, b.obs, b.action, b.reward, b.next_obs, b.done, self.B, 0.99, self.loss,
                              idx=self.idx_cur)
        if ev: ev[3].record()
        return self.loss

    def outputs(self):
        """Greedy actions [E] of the last inference call, the loss of the last SGD step and the trained weights."""
        return dict(action=self.act, loss=self.loss, weights=self.model.get_weights())

    def e2e_setup(self):
        tr = self.tr
        self.host_obs = [np.ascontiguousarray(tr["obs"][t * self.E:(t + 1) * self.E]) for t in range(4)]
        sl = slice(0, self.n)
        self.chunk = dict(cur_state=tr["obs"][sl], action=tr["action"][sl], reward=tr["reward"][sl], next_state=tr["next_obs"][sl], done=tr["done"][sl])

    def e2e_iteration(self):
        for t in range(4):
            np.argmax(self.model.predict(self.host_obs[t]), 1)
        self.alg.prepare_data(self.chunk)
        loss = 0.0
        for s in range(self.steps):
            loss = self.alg.train()
        return loss


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Write each output as <out_dir>/<name>.npy: float64 stays float64, everything else becomes float32 (the integer
    outputs are small indices, exact in float32).  A weight dict is written as one array, its tensors flattened and
    concatenated in parameter order."""
    arrays = {}
    for name, x in outputs.items():
        if isinstance(x, dict):
            x = np.concatenate([np.asarray(v).ravel() for v in x.values()])
        elif hasattr(x, "cpu"):
            x = x.cpu().numpy()
        x = np.asarray(x)
        arrays[name] = x.astype(np.float64 if x.dtype == np.float64 else np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from xingtian_b200 import capi, engine
    from xingtian_b200.engine import _ptr, stream_ptr
    lib = capi.lib()
    dev = torch.device("cuda", local)
    wl = WORKLOADS[args.workload]
    comm = engine.GradComm(device=dev) if world > 1 else None          # before the model: graphs are keyed on it
    np.random.seed(1234 + rank)            # the models draw their action-sampling seed from numpy's global stream
    bench = {"ppo": PpoBench, "impala": ImpalaBench, "dqn": DqnBench}[wl["kind"]](wl, rank, world, dev, local)
    model = bench.model
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)    # > 126 MB L2
    n_global = wl["E"] * wl["T"] if wl["scaling"] == "strong" else bench.n * world     # samples all ranks consume per iteration

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    np.random.seed(1234 + rank)
    for _ in range(args.warmup):
        flush.fill_(1)
        bench.device_iteration()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0, replays0 = lib.xtb_launch_count(), lib.xtb_graph_replay_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        flush.fill_(i)                           # L2 flush between timed iterations (outside the events)
        ev[i][0].record()
        bench.device_iteration()
        ev[i][1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bench.outputs())
    ms_local = sum(a.elapsed_time(b) for a, b in ev)
    launches = lib.xtb_launch_count() - launches0
    replays = lib.xtb_graph_replay_count() - replays0
    seg = {"infer": [], "post": [], "train": []}
    for _ in range(2):
        e4 = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        bench.device_iteration(ev=e4)
        torch.cuda.synchronize()
        seg["infer"].append(e4[0].elapsed_time(e4[1])); seg["post"].append(e4[1].elapsed_time(e4[2])); seg["train"].append(e4[2].elapsed_time(e4[3]))
    breakdown = {k: float(np.mean(v)) for k, v in seg.items()}
    # ---- e2e through the plugin API with host buffers ----------------------------------------------
    bench.e2e_setup()
    bench.e2e_iteration()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        bench.e2e_iteration()
    barrier()
    e2e_s_local = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    # ---- max over ranks --------------------------------------------------------------------------
    tt = torch.tensor([ms_local, e2e_s_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, e2e_s = float(tt[0]), float(tt[1])
    if rank != 0:
        hard_exit()           # multi-rank: leave without communicator / process-group teardown (see hard_exit)
    # ---- roofline of the dominant kernel: every tensor-core layer op of one SGD minibatch is launched alone (`reps`
    #      launches back to back inside one CUDA-event pair on the launching stream, operands L2-resident as they are in
    #      the step); the one with the largest time is reported with its ALGORITHMIC flops (2*M*N*K) against the measured
    #      bf16 tensor peak.
    pk = peaks()
    net = model.net
    Bt = bench.train_batch
    obs_src = bench.store.obs if wl["kind"] == "ppo" else (bench.obs if wl["kind"] == "impala" else bench.alg.buff.obs)
    net.ensure_batch(Bt)
    net.forward(obs_src, Bt)
    for name, _, _, _ in model.arch["layers"]:
        net.tensor_grad(name)[:Bt].normal_()
    shapes = {"obs": STATE}
    ops = []
    for li, (name, kind, src, sp) in enumerate(model.arch["layers"]):
        ish = shapes[src]
        if kind == "conv" and not (sp["pad"] == "valid" and sp["k"] == ish[0]):
            if sp["pad"] == "same":
                oh, ow = -(-ish[0] // sp["s"]), -(-ish[1] // sp["s"])
            else:
                oh, ow = (ish[0] - sp["k"]) // sp["s"] + 1, (ish[1] - sp["k"]) // sp["s"] + 1
            shapes[name] = (oh, ow, sp["cout"])
            gm, gn, gk = Bt * oh * ow, sp["cout"], sp["k"] * sp["k"] * ish[2]
        else:
            nn = sp["cout"] if kind == "conv" else sp["n"]
            shapes[name] = (1, 1, nn) if kind == "conv" else (nn,)
            gm, gn, gk = Bt, nn, int(np.prod(ish))
        if gn < 16:
            continue                                        # the small heads run on CUDA cores / inside the fused heads kernel
        for which, tag in ((0, "forward"), (1, "weight-gradient"), (2, "data-gradient")):
            if which == 2 and src == "obs":
                continue
            ops.append((li, which, "%s %s (M=%d N=%d K=%d)" % (name, tag, gm, gn, gk), 2.0 * gm * gn * gk))
    reps = 20
    best = None
    per_op = {}
    for li, which, label, flop in ops:
        run = lambda: capi.check(lib.xtb_net_bench_layer(net.handle, li, which, _ptr(obs_src), None, Bt, stream_ptr()))
        for _ in range(3):
            run()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            run()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        per_op[label] = round(ms * 1e3, 2)
        if best is None or ms > best[0]:
            best = (ms, label, flop, li, which)
    k_ms, k_label, k_flop, k_li, k_which = best
    run = lambda: capi.check(lib.xtb_net_bench_layer(net.handle, k_li, k_which, _ptr(obs_src), None, Bt, stream_ptr()))
    cold = []
    for _ in range(5):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); run(); b.record()
        torch.cuda.synchronize()
        cold.append(a.elapsed_time(b))
    achieved = k_flop / (k_ms * 1e-3) / 1e12
    traffic = None
    try:   # dram bytes of this kernel from the committed ncu --set full capture (profiles/), if present
        with open(os.path.join(ROOT, "profiles", "r2_dominant_kernel.json")) as f:
            traffic = json.load(f).get("dram_bytes_per_launch", {}).get("%s:L%d/%d" % (args.workload, k_li, k_which))
    except Exception:
        pass
    kname = "bp_wgrad_kernel" if k_which == 1 else "bp_rows_kernel"
    roofline = {"kernel": kname + ": " + k_label, "bound": "tensor", "achieved": achieved, "peak": pk["tf"],
                "unit": "TFLOP/s", "frac": achieved / pk["tf"], "peak_source": pk["src"] + " bf16 burst (cuBLAS)",
                "traffic": traffic, "ms_per_launch": k_ms, "ms_single_launch_cold_l2": float(np.median(cold)),
                "us_per_op": per_op,
                "note": "ms_per_launch = mean of 20 back-to-back launches (CUDA events on the launching stream, launch gap included); "
                        "flops are algorithmic 2MNK, bf16x3 issues 2-3 tensor-core MACs per algorithmic MAC; traffic = dram bytes "
                        "of the cold-cache ncu capture in profiles/"}
    ms_per_step = ms_total / args.steps
    value = n_global / (ms_per_step * 1e-3)
    whole = {"achieved_tflops": value * wl["flop_per_env_step"] / 1e12 / world,
             "frac_of_sustained_bf16": value * wl["flop_per_env_step"] / 1e12 / world / pk["tf_sus"]}
    # ---- cpu baseline (rank 0, N=1) --------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        st = make_cpu_state(args.workload)
        cpu_iteration(st)
        tc = float(np.mean([cpu_iteration(st) for _ in range(2)]))
        cpu = {"value": samples_per_iteration(wl) / tc, "unit": "env-steps/s", "cores": st["threads"], "host_cpus": os.cpu_count(),
               "kind": "port", "sample": sample_desc(args.workload)}
    out = {"metric": metric_name(args.workload), "value": value, "unit": "env-steps/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
           "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32 (bf16x3 split on tcgen05, fp32 accumulate in TMEM)", "data": "synthetic",
           "config": {"workload": wl["desc"]},
           "timing": "CUDA events per iteration, max over ranks; 256 MiB L2 flush between timed iterations; parallelism dp%d, %s scaling" % (world, wl["scaling"]),
           "clocks": clocks, "gpu_launches": int(launches), "graph_replays": int(replays),
           "e2e": {"value": n_global / e2e_s, "unit": "env-steps/s", "h2d_bytes_per_step": bench.h2d, "d2h_bytes_per_step": bench.d2h,
                   "ms_per_step": e2e_s * 1e3, "steps": args.steps},
           "roofline": roofline, "whole_step": whole, "breakdown_ms": breakdown, "cpu_baseline": cpu}
    print(json.dumps(out))
    if world > 1:
        hard_exit()


def hard_exit():
    """Multi-rank runs end here: rank 0 may still be timing single-kernel launches or the CPU baseline for a long time
    after the other ranks are done, and NCCL / process-group destructors of ranks that finish at different times can
    block on each other.  Everything measured has been reduced already, so the process just leaves."""
    sys.stdout.flush(); sys.stderr.flush()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ppo", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0, b200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
