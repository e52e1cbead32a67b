"""oracle/ -- TEST INFRASTRUCTURE ONLY.

CPU checkers for the block-codec path of pg_cryogen:

* ``oracle.ref``  -- ctypes binding of ``oracle/_ref/libcryoref.so``: the reference's
  UNMODIFIED compression.c + storage.c (compiled from the pg_cryogen sources by
  oracle/Makefile, PG_CRYOGEN_SRC) on top of the image's liblz4 1.9.4 / libzstd 1.5.5;
  without it, the codec calls go to those two libraries directly.
* ``oracle.port`` -- ctypes binding of ``oracle/libcryooracle.so``: our plain-C
  restatement of the LZ4 block format and the zstd frame format (RFC 8878).

Only tests/, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl
reference`` legs of bench.py may import this package.  The product
(``pg_cryogen_b200`` and ``libcryogpu.so``) never does.
"""
