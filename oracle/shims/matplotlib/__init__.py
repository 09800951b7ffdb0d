"""Do-nothing stand-in for matplotlib (plots only; see oracle/shims/plotnine).  TEST INFRASTRUCTURE ONLY."""

from plotnine import INERT as _INERT


def __getattr__(name):
  if name.startswith('__'):
    raise AttributeError(name)
  return _INERT
