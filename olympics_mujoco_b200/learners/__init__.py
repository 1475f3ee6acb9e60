"""Learner-side hooks of the hot path, named as the reference names them.

* ``compute_gae``            mushroom_rl.utils.value_functions.compute_gae, call site
  ``imitation_lib/imitation/gail_TRPO.py:126-128`` (+ the advantage normalisation of :128)
* ``finish_path`` / ``normalize_advantage_ppo``   ``PPOBuffer.finish_path`` ``rl/algos/ppo.py:68-84``, bootstrap :195-196,
  ``advantages = returns - values`` and normalisation :334-336
* ``DiscriminatorReward.make_discrim_reward``     ``GAIL.make_discrim_reward`` ``gail_TRPO.py:320-327`` with the
  ``Standardizer`` side effect of ``networks.py:68-81``

* ``ExpertDataset`` / ``GailDiscriminatorLoss`` / ``VDBLoss`` / ``DiscriminatorReward.fit_batch``   the data side of
  ``GAIL._fit_discriminator`` (``gail_TRPO.py:167-220``): expert minibatch (``minibatch_generator`` over
  ``create_dataset``'s ``states`` / ``next_states``, ``utils/trajectory.py:129-193``), forward pass on
  [policy batch; expert batch], the losses of ``imitation_lib/utils/math.py:11-86`` with the VDB beta update, and the
  logging statistics of ``gail_TRPO.py:222-258``.  The weight update itself (autograd + Adam) stays the learner's.

Everything operates on time-major ``[T, n]`` (or ``[n]``) CUDA tensors of this rank's env shard; the value network and
the policy stay the learner's (PyTorch)."""
from __future__ import annotations

import torch

from .. import distributed as D
from .. import kernels as Kn


def compute_gae(v, v_next, r, absorbing, last, gamma, lam, normalize=False):
    """-> (v_target, adv) like the reference; ``v`` / ``v_next`` are V(s), V(s') evaluated by the caller.  With
    ``normalize`` the advantage is standardised over ALL ranks' transitions: (adv - mean) / (np.std + 1e-8)."""
    v_target, adv = Kn.gae(r, v, v_next, absorbing, last, gamma, lam)
    if normalize:
        mom = D.all_reduce_moments(Kn.moments_scalar(adv))
        Kn.normalize(adv, Kn.adv_stats(mom, unbiased=False, eps=1e-8), out=adv)
    return v_target, adv


def finish_path(rewards, values, gamma, path_end=None, v_next=None, last_val=None):
    """-> (returns, advantages = returns - values) for a rollout buffer; ``last_val`` = (not done) * V(s_T).

    Over a [T, n] buffer filled by ``StickFigureA3.step(a, autoreset=True, max_traj_len=L)``, with ``info["path_end"]``
    and ``info["final_obs"]`` of every step stacked and ``obs_T`` the observation returned by the last step::

        finish_path(rewards, values, gamma, path_end=path_end, v_next=V(final_obs), last_val=V(obs_T))

    A path that ended by ``done`` bootstraps 0, one cut at ``max_traj_len`` bootstraps V of its own last observation, and
    one still running at the end of the buffer bootstraps V(obs_T) -- the reference sampler's ``(not done) * V(state)``."""
    return Kn.ppo_returns(rewards, values, gamma, path_end=path_end, v_next=v_next, v_last=last_val)


def normalize_advantage_ppo(adv, eps=1e-5):
    """ppo.py:336 over every rank's buffer: (adv - mean) / (torch.std (unbiased) + eps), in place."""
    mom = D.all_reduce_moments(Kn.moments_scalar(adv))
    return Kn.normalize(adv, Kn.adv_stats(mom, unbiased=True, eps=eps), out=adv)


class DiscriminatorReward:
    """The reward side of GAIL / VAIL for the UnitreeH1 configuration (state-only discriminator,
    ``use_next_states=False, use_actions=False``; ``examples/imitation_learning/utils.py:151-179``).  The input width
    n_in is that of ``params["w1"]``: the kinematic observation of the env's variant, ``env.get_kinematic_obs_mask()``
    (1..64 inputs)."""

    def __init__(self, kind, params, device="cuda", seed=0):
        self.kind = kind.lower()
        self.disc = Kn.Discriminator(self.kind, params)
        self.standardizer = D.Standardizer(self.disc.n_in, device=device)
        self._gen = torch.Generator(device=device).manual_seed(seed)

    def make_discrim_reward(self, state, action=None, next_state=None, eps=None, update_standardizer=True):
        """state [n_in, n] (SoA) -> reward [n] float32.  Like the reference, every call first folds the batch into the
        standardiser's running sums (all ranks), then standardises with the updated statistics."""
        if update_standardizer:
            self.standardizer.update(state)
        mean, std = self.standardizer.snapshot_f32()
        if self.kind == "vail" and eps is None:
            eps = torch.randn((self.disc.z, state.shape[-1]), device=state.device, generator=self._gen)
        return self.disc.reward(state, mean, std, eps=eps if self.kind == "vail" else None)


class ExpertDataset:
    """Device-resident expert transitions built from ``env.create_dataset()`` (``loco_env_base.py:926-968``): the
    ``states`` rows plus the final ``next_states`` row, stored SoA ``[D, N + 1]`` so that ``next_states[i]`` is row
    ``i + 1`` (``trajectory.py:170-171``).  ``sample(batch)`` is the expert half of a discriminator-fit batch."""

    def __init__(self, dataset, state_mask=None, device="cuda", seed=0):
        import numpy as np
        states, nxt = np.asarray(dataset["states"]), np.asarray(dataset["next_states"])
        full = np.concatenate([states, nxt[-1:]], axis=0)
        if state_mask is not None:
            full = full[:, np.asarray(state_mask)]
        self.n = states.shape[0]
        self.table = Kn.to_soa(full)                       # [D, N + 1]
        self.seed, self.draws = int(seed), 0

    def sample(self, batch, want_next=False, want_idx=False):
        """-> (states [D, batch], next_states | None, idx | None); every call is a new draw.  A batch larger than the
        dataset wraps into further permutation epochs (each epoch is a sample without replacement)."""
        out = Kn.expert_minibatch(self.table, self.n, self.seed, self.draws, batch, want_next, want_idx)
        self.draws += 1
        return out


class GailDiscriminatorLoss:
    """``imitation_lib/utils/math.py:11-38`` over a [policy; expert] logit vector of ALL ranks: bce - entcoeff *
    mean(logit_bernoulli_entropy).  ``__call__`` -> (loss, d loss / d logit of the local samples, stats dict)."""

    def __init__(self, entcoeff=1e-3):
        self.entcoeff = float(entcoeff)

    def _sums(self, logit, n_plcy, target, kl):
        sums, grad = Kn.disc_loss_stats(logit, n_plcy, target=target, kl=kl, entcoeff=self.entcoeff, want_grad=True)
        sums = D.all_reduce_moments(sums).tolist()          # one 72-byte all-reduce; the host read is the fit's metric
        n_p, n_d = sums[7], sums[8]
        n = n_p + n_d
        stats = dict(bce=sums[0] / n, bernoulli_ent=sums[1] / n, kl=sums[2] / n,
                     accuracy_gen=sums[3] / max(n_p, 1), accuracy_exp=sums[4] / max(n_d, 1),
                     d_out_gen=sums[5] / max(n_p, 1), d_out_exp=sums[6] / max(n_d, 1), n=n)
        return stats, grad

    def __call__(self, logit, n_plcy, target=None, kl=None):
        stats, grad = self._sums(logit, n_plcy, target, None)
        loss = stats["bce"] - self.entcoeff * stats["bernoulli_ent"]
        return loss, grad / stats["n"], stats


class VDBLoss(GailDiscriminatorLoss):
    """``math.py:41-86`` (``use_bernoulli_ent=False``): bce + beta * (mean KL - info_constraint), then
    ``beta <- max(0, beta + lr_beta * bottleneck)``.  The returned gradient is that of the bce term with respect to the
    logits; the bottleneck term's gradient flows through mu / logvar in the learner's autograd."""

    def __init__(self, info_constraint, lr_beta, entcoeff=1e-3):
        super().__init__(entcoeff)
        self.info_constraint, self.lr_beta, self.beta = float(info_constraint), float(lr_beta), 0.1

    def __call__(self, logit, n_plcy, target=None, kl=None):
        saved, self.entcoeff = self.entcoeff, 0.0          # no entropy term in the VDB gradient
        try:
            stats, grad = self._sums(logit, n_plcy, target, kl)
        finally:
            self.entcoeff = saved
        bottleneck = stats["kl"] - self.info_constraint
        loss = stats["bce"] + self.beta * bottleneck
        stats.update(bottleneck=bottleneck, beta_used=self.beta)
        self.beta = max(0.0, self.beta + self.lr_beta * bottleneck)
        return loss, grad / stats["n"], stats


def _fit_batch(self, plcy_state, expert, loss, eps=None, noisy_targets=False, logging_forwards=False):
    """One epoch of ``GAIL._fit_discriminator`` up to (not including) the weight update: sample the expert half, fold
    [policy; expert] into the standardiser, forward, loss + statistics.
    ``plcy_state`` [n_in, n]; ``expert`` an ExpertDataset masked to the same n_in columns.
    -> (loss value, stats, batch dict with ``inputs`` [n_in, 2n], ``logit``, ``kl``, ``dlogit``, ``target``).

    Standardiser bookkeeping, as the reference does it: the discriminator's input standardiser and ``_D_standardizer``
    are ONE object (``examples/imitation_learning/utils.py``), and it updates on EVERY forward (``networks.py:66-71``).
    One fit epoch therefore folds the [policy; expert] batch in TWICE before the batch is standardised -- the explicit
    ``update_mean_std`` (``gail_TRPO.py:200-201``) and the forward inside ``D.fit`` -- and, when a summary writer is
    attached, ``_discriminator_logging`` (:222-258) runs six more forwards afterwards (two on the full batch, two on
    each half: four batch-equivalents).  The same counts are replayed here (``logging_forwards`` = a writer is attached);
    the moment sums of a batch are computed once and added with the multiplicity."""
    n = plcy_state.shape[-1]
    assert plcy_state.shape[0] == self.disc.n_in and expert.table.shape[0] == self.disc.n_in
    demo, _, _ = expert.sample(n)
    inputs = torch.cat([plcy_state, demo], dim=1)
    batch_moments = Kn.moments(inputs)
    self.standardizer.update_from_moments(2.0 * batch_moments)
    mean, std = self.standardizer.snapshot_f32()
    if self.kind == "vail" and eps is None:
        eps = torch.randn((self.disc.z, 2 * n), device=inputs.device, generator=self._gen)
    fw = self.disc.forward(inputs, mean, std, eps=eps if self.kind == "vail" else None)
    target = None
    if noisy_targets:                                       # gail_TRPO.py:204-206
        u = torch.rand(2 * n, device=inputs.device, generator=self._gen)
        target = torch.cat([0.01 + 0.09 * u[:n], 0.80 + 0.19 * u[n:]])
    value, dlogit, stats = loss(fw["logit"], n, target=target, kl=fw.get("kl"))
    if logging_forwards:
        self.standardizer.update_from_moments(4.0 * batch_moments)
    return value, stats, dict(inputs=inputs, target=target, dlogit=dlogit, eps=eps, **fw)


DiscriminatorReward.fit_batch = _fit_batch


def ppo_update_losses(logp, old_logp, adv, mask, values, returns, clip=0.2, vf_coeff=0.5, entropy=None, act=None,
                      act_mirror=None, action_mirror=None):
    """``PPO.update_policy`` (``rl/algos/ppo.py:231-282``) over ALL ranks' minibatch shards -> (dict of the six values it
    returns, d actor_loss / d log_probs, d critic_loss / d values), the gradients scaled for the global mean."""
    sums, dlogp, dvalues = Kn.ppo_loss_stats(logp, old_logp, adv, clip, mask=mask, values=values, returns=returns,
                                             vf_coeff=vf_coeff, entropy=entropy, act=act, act_mirror=act_mirror,
                                             action_mirror=action_mirror)
    n_local = logp.numel()
    s = D.all_reduce_moments(sums).tolist()
    n = s[6]
    nu = act.shape[0] if act is not None else (entropy.shape[0] if entropy is not None else 1)
    out = dict(actor_loss=-s[0] / n, entropy_penalty=-s[1] / (n * nu), critic_loss=vf_coeff * s[2] / n, approx_kl=s[3] / n,
               mirror_loss=s[4] / (n * nu), clip_fraction=s[5] / n)
    scale = n_local / n
    return out, dlogp * scale, (dvalues * scale if dvalues is not None else None)
