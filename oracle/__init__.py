"""oracle -- CPU checkers for rawspeed_b200.  TEST INFRASTRUCTURE ONLY.

Two checkers live here:

* ``oracle.port``  -- ctypes binding of ``librs_oracle.so`` (our C99 restatement of
  the reference algorithm, ``rs_oracle.c``; each function cites the reference
  file:line it follows).
* ``oracle.ref``   -- ctypes binding of ``_ref/libref.so`` (the UNMODIFIED reference
  compiled by ``oracle/Makefile``), when it has been built; without it, the reference's
  answers recorded under ``tests/golden/ref_calls/`` (``ref.available()``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  ``rawspeed_b200`` never does.
"""
from . import port, synth  # noqa: F401

try:  # the reference arm is optional (absent until `make -C oracle ref`)
    from . import ref  # noqa: F401
    HAVE_REF = ref.live()   # the timed legs need the library itself, not its recorded answers
except OSError:  # pragma: no cover
    ref = None
    HAVE_REF = False
