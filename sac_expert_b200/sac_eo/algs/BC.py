"""``BC`` - behaviour cloning from expert OBSERVATIONS through the learned models, reference interface
(``/root/reference/sac_eo/algs/BC.py``).  ``_update(num_timesteps, expert_reg)`` only calls ``_update_actor``
(:303-307): the expert-observation MSE of the SAC-EO actor step with weight 1 and nothing else, one Adam step of
``self.actor_optimizer`` (:113).  Model fitting, the adaptive-weight bookkeeping and the buffers are inherited from
``SAC_exp`` (the reference duplicates that code in BC.py)."""
import numpy as np

from .SAC_expert import SAC_exp
from ..common.lockstep import Request, inline, np_random


class BC(SAC_exp):
    def _update_steps(self, num_timesteps, expert_reg):
        """``BC._update`` (:303-307)."""
        yield from self._update_actor_steps(expert_reg)

    def _update_actor_steps(self, expert_reg):
        """``BC._update_actor`` (:309-363).  Host RNG consumption as in the reference: one ``self.rng.shuffle`` of the
        expert rows when two models are used (:330-332), then one ``np.random.normal`` draw per ``actor.sample`` call
        (continuous_actors.py:297)."""
        s_expert, _, sp_expert, _, _ = expert_reg
        s_expert, sp_expert = np.asarray(s_expert, np.float32), np.asarray(sp_expert, np.float32)
        E, B, A = len(s_expert), self.sac_batch_size, self.a_dim
        if E != self.pop.spec.E:
            raise ValueError(f"expert_reg carries {E} rows, the device population was built for {self.pop.spec.E}")
        key = (id(expert_reg[0]), id(expert_reg[2]))
        expert = None if key == self._last_expert else (s_expert, sp_expert)
        self._last_expert = key
        rand = np_random()
        if self._n_models() == 1:
            perm = np.arange(E)
            u_exp = [rand.normal(size=(E, A))]
        else:
            order = np.arange(E)
            self.rng.shuffle(order)
            halves = np.array_split(order, len(self.models))
            if len(halves[0]) != len(halves[1]):
                raise ValueError("two-model expert term needs an even number of expert rows (BC.py:334-347)")
            perm = np.concatenate(halves[:2])
            u_exp = [rand.normal(size=(len(halves[0]), A)), rand.normal(size=(len(halves[1]), A))]
        zeros = np.zeros((B, A))
        noise = np.concatenate([zeros, zeros] + u_exp + [zeros], 0).astype(np.float32)     # only the expert block is read
        perm = perm.astype(np.int32)
        losses = yield Request("update", self.pop, self.agent, ("bc", noise.shape, perm.shape), bc=True, idx=None, noise=noise,
                               perm=perm, expert=expert, eps=None)
        self.last_losses = dict(BC_MSE_loss=float(losses[3]))
        self.logger.log_train({"BC_MSE_loss": losses[3]})                                 # :360-363

    _update_actor = inline(_update_actor_steps)
