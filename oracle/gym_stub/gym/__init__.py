"""Minimal structural stand-in for `gym` (TEST INFRASTRUCTURE ONLY).

`gym` is not installed in this image and there is no network.  The reference
environment (marlenv/ of the original project) needs gym only structurally (base classes,
spaces with .n/.shape/.sample(), the registry).  This stub lets the *unmodified*
reference be imported so it can be used to generate golden vectors
(tests/golden/make_golden.py) and to pin the oracle.  It implements none of the
Snake arithmetic and is never on the product path.
"""
from . import spaces, error          # noqa: F401
from .core import Env, Wrapper       # noqa: F401
from .envs.registration import register, make   # noqa: F401
from . import utils, vector          # noqa: F401

__version__ = "0.0-stub"
