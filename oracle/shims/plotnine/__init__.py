"""Do-nothing stand-in for plotnine, which the reference's analysis modules import at module level (for plots
only).  Every attribute is one inert object that can be called, indexed into and added to; nothing is computed.
TEST INFRASTRUCTURE ONLY (oracle/gen_score_checks.py)."""


class _Inert:

  def __call__(self, *args, **kwargs):
    return self

  def __getattr__(self, name):
    if name.startswith('__'):
      raise AttributeError(name)
    return self

  def __add__(self, other):
    return self

  __radd__ = __add__


INERT = _Inert()


def __getattr__(name):
  if name.startswith('__'):
    raise AttributeError(name)
  return INERT
