"""Host side of the RNG contract (csrc/om_math.cuh ``om_draw``): Philox4x32-10, key = seed, counter =
(env_id, reset_count, stream, 0); integers by multiply-shift.  Plain Python integers -- used for the few draws the HOST
takes (which model a MultiMuJoCo reset switches to, loco_env_base.py:586-589)."""

_M0, _M1, _W0, _W1, _MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF

STREAM_MODEL_RESET = 32            # the model switch of a whole reset() (MultiMuJoCo; om_h1_draw_models)
STREAM_PARTIAL_MODEL_RESET = 33    # the model one env draws at its own partial reset (om_h1_reset_envs)


def philox4x32_10(counter, key):
    c0, c1, c2, c3 = (int(x) & _MASK for x in counter)
    k0, k1 = (int(x) & _MASK for x in key)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _MASK, p1 & _MASK, ((p0 >> 32) ^ c3 ^ k1) & _MASK, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def philox_randint(seed, env_id, count, stream, n):
    """First output word of the contract's draw -> integer in [0, n)."""
    seed = int(seed)
    w = philox4x32_10((env_id, count, stream, 0), (seed & _MASK, (seed >> 32) & _MASK))
    return (w[0] * int(n)) >> 32


def env_model_draw(seed, env_id, count, n_models, random=True):
    """The model that env ``env_id`` (global id) holds after its env object's reset number ``count`` (0-based) when every
    env draws its own (``per_env_weight``; ``om_h1_draw_models`` on the device): random -- the shared draw keyed on the env
    instead of the object; round robin -- model ``(env_id + count + 1) mod n_models``.  Env id 0 follows the sequence a
    shared MultiMuJoCo env object picks."""
    if random:
        return philox_randint(seed, env_id, count, STREAM_MODEL_RESET, n_models)
    return (int(env_id) + int(count) + 1) % int(n_models)


def env_partial_model_draw(seed, env_id, j, n_models, prev_index, random=True):
    """The model env ``env_id`` (global id) holds after its own ``j``-th partial reset (0-based; ``reset(mask=...)`` or
    ``step(autoreset=True)`` with ``per_env_weight``; ``om_h1_reset_envs`` on the device): random -- the draw of stream 33
    keyed on the env and its partial-reset count; round robin -- the model after ``prev_index``.  A stream of its own, so the
    draws of whole resets (stream 32, ``env_model_draw``) never meet these."""
    if random:
        return philox_randint(seed, env_id, j, STREAM_PARTIAL_MODEL_RESET, n_models)
    return (int(prev_index) + 1) % int(n_models)
