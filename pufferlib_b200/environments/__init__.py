"""Device-native env kinds and how a creator callable maps to one.

The reference passes ``env_creator`` callables to ``vector.make`` and the backend calls each one N times
(vector.py:79).  The B200 backend instead asks the creator which native kind it stands for and builds ONE
device-resident multi-env (the PufferEnv seam, pufferlib/environment.py:1-21).  A creator is recognised by a
``b200_kind`` attribute (ours) or by name for the reference's own ``make_squared``
(pufferlib/environments/ocean/environment.py:28-31), so the reference's creator can be passed unchanged.
"""
import numpy as np

from pufferlib_b200.exceptions import APIUsageError

# kinds whose observation is a structured record: the np.dtype(align=True) of the native Dict space with gymnasium's
# sorted keys (emulation.py:68-80), i.e. the `emulated_observation_dtype` of the reference's GymnasiumPufferEnv
OBS_RECORD_DTYPE = {
    'spaces': np.dtype([('flat', np.int8, (5,)), ('image', np.float32, (5, 5))], align=True),
}

KNOWN_BY_NAME = {'make_squared': 'squared', 'make_breakout': 'breakout', 'make_snake': 'snake', 'make_pong': 'pong',
                 'make_spaces': 'spaces'}


def resolve(creator, args, kwargs):
    """-> (kind name, iparam list of 8 ints) for pb_env_config."""
    kind = getattr(creator, 'b200_kind', None)
    if kind is None:
        kind = KNOWN_BY_NAME.get(getattr(creator, '__name__', ''), None)
    if kind is None:
        raise APIUsageError(
            f'env creator {creator!r} has no device-native kind: the B200 backend only runs '
            f'{sorted(set(KNOWN_BY_NAME.values()))} (no CPU fallback)')
    kwargs = dict(kwargs or {})
    iparam = [0] * 8
    if kind == 'squared':
        names = ('distance_to_target', 'num_targets')
        vals = dict(zip(names, args or ()))
        vals.update({k: kwargs.pop(k) for k in list(kwargs) if k in names})
        if vals.get('num_targets', 1) != 1:
            raise APIUsageError('squared: only num_targets=1 (the reference default) is implemented on the device')
        iparam[0] = int(vals.get('distance_to_target', 3))
    elif kind == 'breakout':
        iparam[0] = int(kwargs.pop('max_ticks', 0))
    elif kind == 'snake':
        iparam[0] = int(kwargs.pop('max_ticks', 0))
    elif kind == 'pong':
        iparam[0] = int(kwargs.pop('max_score', 0))
        iparam[1] = int(kwargs.pop('max_ticks', 0))
    elif kind == 'spaces' and args:
        raise APIUsageError('spaces: the env takes no arguments')
    if kwargs:
        raise APIUsageError(f'{kind}: unexpected env kwargs {sorted(kwargs)}')
    return kind, iparam


def _creator(kind):
    def make(*args, **kwargs):
        raise APIUsageError(
            f"'{kind}' is a device-native env: pass this creator to pufferlib_b200.vector.make(..., "
            f'backend=pufferlib_b200.vector.B200); it cannot be instantiated on the CPU')
    make.__name__ = 'make_' + kind
    make.b200_kind = kind
    return make
