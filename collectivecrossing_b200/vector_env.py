"""Vectorised multi-agent view for learners (SURVEY.md §8 f-3).

The reference trains with RLlib: one ``CollectiveCrossingEnv`` per env-runner actor, a
``policy_mapping_fn`` that sends ``boarding_*`` agents to the policy "boarding" and ``exiting_*``
agents to "exiting" (``examples/training_script.py:26-47``), observation dicts rebuilt per step.
``VectorCollectiveCrossing`` exposes N device envs in the shape a learner consumes directly:

* observations as ONE float32 tensor ``[N, A, 6+4A]`` on the device, with per-policy views
  ``[N, B, L]`` / ``[N, E, L]`` (agents of a policy are contiguous in agent order, so these are
  zero-copy slices) and flat ``[N*B, L]`` batches;
* actions as one int8 tensor ``[N, A]`` or a ``{policy: [N, n_agents_of_policy]}`` dict;
* masks instead of missing dict keys: ``valid`` (the agent had reward / truncated entries this
  step, i.e. was alive at step start), ``obs_valid`` (it had an observation entry), plus
  ``terminateds`` / ``truncateds`` per agent and the ``__all__`` flags per env;
* the reference's naming: ``possible_agents``, ``policy_mapping_fn``, per-agent spaces.

``to_multi_agent_dicts(n)`` rebuilds the reference's five dicts for one env — what an RLlib
``MultiAgentEnv`` runner would be handed — from the tensors of the last step (used by the tests to
pin this view against the single-env facade).  Everything runs through ``BatchedCollectiveCrossing``
(one fused kernel launch per step); nothing here touches the oracle.
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Any

import numpy as np
import torch

from . import _abi, _spaces
from .batched import BatchedCollectiveCrossing, StepOutput

POLICIES = ("boarding", "exiting")


def policy_mapping_fn(agent_id: str, *args: Any, **kwargs: Any) -> str:
    """examples/training_script.py:32-47"""
    return "boarding" if agent_id.startswith("boarding_") else "exiting"


@dataclass
class VectorStep:
    """One step of all envs; every tensor lives on the device and aliases the env's buffers."""

    obs: torch.Tensor          # [N, A, L] float32 (rows of agents without ``obs_valid`` are stale / post-reset)
    rewards: torch.Tensor      # [N, A] float32, 0 where not ``valid``
    terminateds: torch.Tensor  # [N, A] bool (defined for every agent every step, terminateds.py:37-82)
    truncateds: torch.Tensor   # [N, A] bool (meaningful where ``valid``)
    valid: torch.Tensor        # [N, A] bool: rewards / truncateds entries exist (alive at step start)
    obs_valid: torch.Tensor    # [N, A] bool: observation / info entries exist (collectivecrossing.py:243)
    terminated_all: torch.Tensor  # [N] bool
    truncated_all: torch.Tensor   # [N] bool
    was_reset: torch.Tensor       # [N] bool: the env was auto-reset in this launch; ``obs`` shows the new episode
    raw: StepOutput


class VectorCollectiveCrossing:
    """N CollectiveCrossing envs for a learner; see the module docstring."""

    def __init__(self, config: Any, num_envs: int, device: Any = "cuda:0", *, seed: int = 0, auto_reset: bool = True,
                 global_env_offset: int = 0, reset_rng: str = "philox"):
        if isinstance(config, dict):  # RLlib env_config dicts
            from .configs import CollectiveCrossingConfig

            config = CollectiveCrossingConfig(**config)
        self.config = config
        self.env = BatchedCollectiveCrossing(config, num_envs, device, seed=seed, obs_dtype="float32", reward_dtype="float32",
                                             auto_reset=auto_reset, with_info=True, global_env_offset=global_env_offset,
                                             reset_rng=reset_rng)
        self.num_envs = self.env.num_envs
        self.num_agents = self.env.num_agents
        self.num_boarding = config.num_boarding_agents
        self.possible_agents = [f"boarding_{i}" for i in range(config.num_boarding_agents)] + [
            f"exiting_{i}" for i in range(config.num_exiting_agents)]
        self.policy_slices = {"boarding": slice(0, self.num_boarding), "exiting": slice(self.num_boarding, self.num_agents)}
        n_obs = self.env.obs_len
        self.single_action_space = _spaces.Discrete(5)
        self.single_observation_space = _spaces.Box(low=-1, high=max(config.width, config.height) - 1, shape=(n_obs,), dtype=np.float32)
        self.action_spaces = {a: self.single_action_space for a in self.possible_agents}
        self.observation_spaces = {a: self.single_observation_space for a in self.possible_agents}
        self._actions = torch.zeros((self.num_envs, self.num_agents), dtype=torch.int8, device=self.env.device)
        self._last: VectorStep | None = None

    # ---- reference-style accessors ---------------------------------------------------------------------
    policy_mapping_fn = staticmethod(policy_mapping_fn)

    def policy_of(self, agent_id: str) -> str:
        return policy_mapping_fn(agent_id)

    def close(self) -> None:
        self.env.close()

    # ---- reset / step ----------------------------------------------------------------------------------
    def reset(self, *, seed: int | torch.Tensor | None = None) -> torch.Tensor:
        """All envs.  ``seed=None``: counter-based placement (``reset_rng="numpy"``: every env continues its numpy
        generator, the reference's ``reset()``); an int ``s``: env n is reset like the reference's ``reset(seed=s+n)``
        (numpy-exact PCG64 placement); a tensor: one seed per env.  With ``reset_rng="numpy"``, ``reset(seed=s)``
        followed by ``step`` with auto-reset reproduces N reference envs seeded ``s + n``, episode after episode."""
        if seed is None:
            return self.env.reset()
        if not torch.is_tensor(seed):
            seed = torch.arange(self.num_envs, dtype=torch.int64, device=self.env.device) + int(seed)
        return self.env.reset_seeded(seed.to(self.env.device, torch.int64))

    def _wrap(self, out: StepOutput) -> VectorStep:
        af = out.agent_flags
        self._last = VectorStep(out.obs, out.reward, (af & _abi.O_TERM_VALUE) != 0, (af & _abi.O_TRUNC_VALUE) != 0,
                                (af & _abi.O_ALIVE_PREV) != 0, (af & _abi.O_OBS_PRESENT) != 0, out.terminated_all, out.truncated_all,
                                out.was_reset, out)
        return self._last

    def step(self, actions: torch.Tensor | dict[str, torch.Tensor] | None = None, *, policy: str = "external") -> VectorStep:
        """``actions``: int8 ``[N, A]``, or ``{"boarding": [N, B], "exiting": [N, E]}`` as two policies
        would emit them; agents that are done or inactive may hold any valid action (the reference ignores
        them, collectivecrossing.py:398).  ``policy`` selects an on-device baseline policy instead."""
        if policy != "external":
            return self._wrap(self.env.step(policy=policy))
        if isinstance(actions, dict):
            for name, sl in self.policy_slices.items():
                if sl.stop > sl.start:
                    self._actions[:, sl] = actions[name].to(self._actions.device, torch.int8).reshape(self.num_envs, sl.stop - sl.start)
            actions = self._actions
        return self._wrap(self.env.step(actions))

    # ---- per-policy batches ----------------------------------------------------------------------------
    def policy_view(self, t: torch.Tensor, policy: str) -> torch.Tensor:
        """The rows of ``t`` ([N, A, ...]) that belong to ``policy``: a zero-copy slice ``[N, n, ...]``."""
        return t[:, self.policy_slices[policy]]

    def policy_batch(self, step: VectorStep, policy: str) -> dict[str, torch.Tensor]:
        """Flat per-policy batch ``[N*n, ...]`` (copies only where the slice is not contiguous)."""
        def flat(t):
            v = self.policy_view(t, policy)
            return v.reshape(v.shape[0] * v.shape[1], *v.shape[2:])
        return {"obs": flat(step.obs), "rewards": flat(step.rewards), "terminateds": flat(step.terminateds),
                "truncateds": flat(step.truncateds), "valid": flat(step.valid), "obs_valid": flat(step.obs_valid)}

    # ---- the reference's dict view of one env --------------------------------------------------------------
    def to_multi_agent_dicts(self, n: int, step: VectorStep | None = None):
        """``(observations, rewards, terminateds, truncateds, infos)`` of env ``n`` for the last step, as
        ``CollectiveCrossingEnv.step`` returns them (collectivecrossing.py:204-261)."""
        step = step or self._last
        if step is None:
            raise RuntimeError("no step taken yet")
        raw = step.raw
        rows, rew = raw.obs[n].cpu().numpy(), raw.reward[n].cpu().numpy()
        af, ai, ef = raw.agent_flags[n].cpu().numpy(), raw.agent_info[n].cpu().numpy(), int(raw.env_flags[n])
        obs, rewards, terms, truncs, infos = {}, {}, {}, {}, {}
        for k, a in enumerate(self.possible_agents):
            bits = int(af[k])
            terms[a] = bool(bits & _abi.O_TERM_VALUE)
            if bits & _abi.O_ALIVE_PREV:
                rewards[a] = float(rew[k])
                truncs[a] = bool(bits & _abi.O_TRUNC_VALUE)
            if bits & _abi.O_OBS_PRESENT:
                obs[a] = rows[k].copy()
                infos[a] = {"agent_type": "boarding" if k < self.num_boarding else "exiting",
                            "in_tram_area": bool(ai[k] & _abi.I_IN_TRAM_AREA), "at_door": bool(ai[k] & _abi.I_AT_DOOR),
                            "active": bool(ai[k] & _abi.I_ACTIVE), "at_destination": bool(ai[k] & _abi.I_AT_DESTINATION)}
        terms["__all__"] = bool(ef & _abi.E_TERMINATED_ALL)
        truncs["__all__"] = bool(ef & _abi.E_TRUNCATED_ALL)
        return obs, rewards, terms, truncs, infos
