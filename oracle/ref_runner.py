"""TEST / MEASUREMENT INFRASTRUCTURE ONLY.  Time the UNMODIFIED reference's PPO minibatch step on the host cores.

Used by `bench.py --impl reference` and by bench.py's `cpu_baseline` leg when the reference is staged
(`oracle/stage_ref.py` -> `oracle/_ref/`).  The timed region is exactly the reference's
minibatch body, urban_planning/agents/urban_planning_agent.py:327-337:
    tensorfy(states_b) -> value_loss -> ppo_entropy_loss -> loss.backward() -> clip_policy_grad -> optimizer.step
with the reference's own modules (`create_sgnn_model`) and methods (`AgentPG.value_loss`,
`UrbanPlanningAgent.ppo_entropy_loss`, `AgentPPO.clip_policy_grad`).
"""
from __future__ import annotations

import os
import time
import types

import numpy as np


def available() -> bool:
    from oracle import stage_ref
    return stage_ref.staged_root() is not None


class ReferenceStepper:
    def __init__(self, max_num_nodes: int, max_num_edges: int, flat=None, seed: int = 111):
        from oracle import stage_ref
        root = stage_ref.staged_root()
        if root is None:
            raise RuntimeError("the reference is not staged under oracle/_ref (oracle/stage_ref.py)")
        os.environ["UPB_REFERENCE_ROOT"] = root
        from oracle import ref_shim
        ref_shim.REFERENCE_ROOT = root
        ref_shim.install()
        import torch
        from urban_planning.agents.urban_planning_agent import UrbanPlanningAgent, tensorfy
        from khrylib.rl.agents import AgentPG, AgentPPO
        self.torch, self.tensorfy, self.root = torch, tensorfy, root
        policy_net, value_net, ac = ref_shim.build_reference_model(max_num_nodes, max_num_edges, seed)
        if flat is not None:
            from drl_urban_planning_b200 import params as PL
            sd = PL.to_state_dict(np.asarray(flat, np.float32))
            ac.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
        duck = types.SimpleNamespace()
        duck.policy_net, duck.value_net = policy_net, value_net
        duck.trans_policy = duck.trans_value = lambda s: s
        duck.clip_epsilon = 0.2
        duck.policy_grad_clip = [(policy_net.parameters(), 1), (value_net.parameters(), 1)]   # urban_planning_agent.py:46
        for fn, owner in (("ppo_entropy_loss", UrbanPlanningAgent), ("value_loss", AgentPG),
                          ("clip_policy_grad", AgentPPO)):
            setattr(duck, fn, types.MethodType(getattr(owner, fn), duck))
        self.duck, self.ac = duck, ac
        self.opt = torch.optim.Adam(ac.parameters(), lr=4e-4, eps=1e-5, weight_decay=0.0)

    def step(self, states, actions, adv, ret, fixed, ind):
        """One minibatch step; `states` are numpy 9-array states (tensorfy is inside the timed region, :327)."""
        torch, d = self.torch, self.duck
        states_b = self.tensorfy(states, torch.device("cpu"))
        value_loss = d.value_loss(states_b, ret)
        surr, ent = d.ppo_entropy_loss(states_b, actions, adv, fixed, ind)
        loss = surr + 0.5 * value_loss + 0.01 * ent
        self.opt.zero_grad()
        loss.backward()
        d.clip_policy_grad()
        self.opt.step()
        return float(loss.item())


def step_time(states, actions, flat, steps: int, warmup: int, threads: int, n_cap: int, e_cap: int) -> float:
    """Seconds per minibatch step of the reference on `threads` torch threads."""
    import warnings
    import torch
    torch.set_num_threads(threads)
    n = len(states)
    rng = np.random.default_rng(5)
    adv = torch.tensor(rng.standard_normal((n, 1)).astype(np.float32))
    ret = torch.tensor(rng.standard_normal((n, 1)).astype(np.float32))
    fixed = torch.full((n, 1), -4.0)
    ind = torch.arange(n)
    act = torch.tensor(np.asarray(actions, np.float32))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = ReferenceStepper(n_cap, e_cap, flat)
        times = []
        for k in range(warmup + steps):
            t0 = time.perf_counter()
            ref.step(states, act, adv, ret, fixed, ind)
            if k >= warmup:
                times.append(time.perf_counter() - t0)
    return float(np.mean(times))
