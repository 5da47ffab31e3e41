"""ofdm-course_b200 -- B200-native batched OFDM link chain behind the reference's function names.

Import it as ``import ofdm_b200`` (the root-level alias module) or
``importlib.import_module("ofdm-course_b200")``.  The package needs its CUDA library
(``lib/libofdm_b200.so``, built by ``make -C ofdm-course_b200`` or ``__graft_entry__.build()``);
there is no CPU fallback.
"""
from . import _cabi  # noqa: F401
from .link import *  # noqa: F401,F403
from .link import Context, OfdmError, default_context, pack_bits, unpack_bits, CONSTELLATIONS, DEFAULT_REGISTER  # noqa: F401
from . import sweep  # noqa: F401,E402
from .sweep import Group  # noqa: F401,E402
from . import layouts  # noqa: F401,E402
