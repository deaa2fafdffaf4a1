"""Weight-list conventions of the reference networks (``/root/reference/sac_eo/common/nn_utils.py``):
Keras ``Sequential`` of ``Dense`` layers, ``y = x @ W + b``, ``W: [in, out]``, ``get_weights()`` order
``[W0, b0, W1, b1, W2, b2]``; orthogonal(sqrt 2) hidden / orthogonal(gain) final initialisation, zero biases.
Actors, critics and reward networks the project trains have two hidden layers (every BASELINE config is 2x256 / 2x512);
dynamics models have 1 to 8, and weight lists of any depth are built for actors that are only acted (expert policies)."""
import math

import numpy as np

ACTIVATIONS = ("tanh", "relu", "elu")


def broadcast_activations(layers, activations):
    """One activation string is broadcast to all hidden layers (nn_utils.py:7-8)."""
    acts = list(activations)
    if len(layers) > 1 and len(acts) == 1:
        acts = acts * len(layers)
    for a in acts:
        if a not in ACTIVATIONS:
            raise ValueError("activations must be tanh, relu or elu")
    if len(acts) != len(layers):
        raise AssertionError("activations must be list of length len(layers)")
    return tuple(acts)


def check_two_hidden(layers):
    if len(layers) != 2:
        raise ValueError("sac_expert_b200 supports exactly two hidden layers per network (got %r)" % (layers,))
    return tuple(int(h) for h in layers)


MODEL_MAX_HIDDEN = 8     # include/saceo.h SACEO_POLICY_MAX_HIDDEN


def check_model_hidden(layers):
    """Hidden widths of a dynamics model: 1 to MODEL_MAX_HIDDEN layers, each at least 1 wide."""
    hidden = tuple(int(h) for h in layers)
    if not 1 <= len(hidden) <= MODEL_MAX_HIDDEN or min(hidden) < 1:
        raise ValueError("sac_expert_b200 dynamics models have 1 to %d hidden layers of width >= 1 (got %r)"
                         % (MODEL_MAX_HIDDEN, layers))
    return hidden


def trainable_names(n_hidden):
    """Keras variable order of a Sequential of n_hidden + 1 Dense layers: W0, b0, ..., Wn, bn."""
    return ["%s%d" % (k, l) for l in range(n_hidden + 1) for k in ("W", "b")]


def _orthogonal(rng, rows, cols, gain):
    a = rng.standard_normal((max(rows, cols), min(rows, cols)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if rows < cols:
        q = q.T
    return (gain * q[:rows, :cols]).astype(np.float32)


def create_nn_weights(in_dim, out_dim, layers, gain, init_type="orthogonal", rng=None):
    """Initial weight list of ``create_nn`` (nn_utils.py:86-138)."""
    rng = rng if rng is not None else np.random.default_rng(np.random.randint(2 ** 31))
    dims = [in_dim] + list(layers) + [out_dim]
    ws = []
    for l in range(len(layers) + 1):
        rows, cols = dims[l], dims[l + 1]
        last = l == len(layers)
        if init_type == "orthogonal":
            w = _orthogonal(rng, rows, cols, gain if (last and gain) else math.sqrt(2.0))
        elif init_type == "var":          # VarianceScaling(uniform, fan_out)
            scale = gain if (last and gain) else 0.333
            lim = math.sqrt(3.0 * scale / cols)
            w = rng.uniform(-lim, lim, (rows, cols)).astype(np.float32)
        elif init_type == "uniform":      # glorot_uniform
            lim = math.sqrt(6.0 / (rows + cols))
            w = rng.uniform(-lim, lim, (rows, cols)).astype(np.float32)
        else:
            raise ValueError("init_type must be orthogonal, var or uniform")
        ws += [w, np.zeros(cols, np.float32)]
    return ws


def flat_to_list(shapes, weights):
    out, o = [], 0
    for sh in shapes:
        n = int(np.prod(sh))
        out.append(np.reshape(weights[o:o + n], sh))
        o += n
    return out


def list_to_flat(weights):
    return np.concatenate([np.reshape(w, [-1]) for w in weights], -1)
