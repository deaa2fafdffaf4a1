"""``init_actor`` with the reference's signature (``/root/reference/sac_eo/actors/init_actor.py:8-31``): a
``SquashedGaussianActor`` with ``actor_squash`` (the SAC / SAC-EO learner), a ``GaussianActor`` otherwise (the reference's
on-policy actor and the format of its MPO experts)."""
from .continuous_actors import GaussianActor, SquashedGaussianActor


def init_actor(env, actor_layers, actor_activations, actor_gain, actor_std_mult, actor_init_type, actor_layer_norm,
               actor_weights, actor_per_state_std=False, actor_squash=False, actor_output_norm=False):
    if actor_squash:
        actor = SquashedGaussianActor(env, actor_layers, actor_activations, actor_gain, actor_init_type, actor_layer_norm,
                                      actor_std_mult, actor_per_state_std, actor_output_norm)
    else:
        if actor_output_norm:
            raise ValueError("actor_output_norm is not supported by the CUDA path")
        actor = GaussianActor(env, actor_layers, actor_activations, actor_gain, actor_init_type, actor_layer_norm,
                              actor_std_mult, actor_per_state_std, actor_output_norm)
    if actor_weights is not None:
        actor.set_weights(actor_weights)
    return actor
