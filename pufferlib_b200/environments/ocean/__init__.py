"""Mirror of pufferlib.environments.ocean (reference: ocean/environment.py:6-26): ``env_creator(name)``."""
from pufferlib_b200.environments import _creator

make_squared = _creator('squared')
make_breakout = _creator('breakout')
make_snake = _creator('snake')
make_pong = _creator('pong')
make_spaces = _creator('spaces')

_CREATORS = {'squared': make_squared, 'breakout': make_breakout, 'snake': make_snake, 'pong': make_pong,
             'spaces': make_spaces}


def env_creator(name='squared'):
    try:
        return _CREATORS[name]
    except KeyError:
        raise ValueError('Invalid environment name')
