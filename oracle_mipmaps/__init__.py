"""CPU oracle of rule R12 (r3_generate_mipmaps) — TEST INFRASTRUCTURE.  Only tests/, tools/ and __graft_entry__.build() import this
package; rend3_b200/ never does.  libr3_oracle_mipmaps.so works on the CPU oracle's context (oracle/r3_oracle.h) and exports
r3o_generate_mipmaps / r3o_readback_texels; `load_oracle_backend()` binds them next to the oracle's own entry points."""
import ctypes
import os
import subprocess

_DIR = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_DIR)
LIB_PATH = os.path.join(_DIR, "libr3_oracle_mipmaps.so")
_SRC = os.path.join(_DIR, "r3_oracle_mipmaps.c")
_CC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"   # the system compiler: it has libgomp
# strict IEEE f32 in source order, no contraction, no fast-math: the flags of the CPU oracle (oracle/Makefile)
CFLAGS = ["-O3", "-mavx2", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-Wall", "-Wextra"]


def build(force: bool = False) -> str:
    deps = [_SRC] + [os.path.join(_ROOT, p) for p in ("oracle/r3_oracle.h", "include/r3_layouts.h", "include/rend3_b200.h", "include/r3_srgb_tables.h")]
    stale = force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps if os.path.exists(d))
    if stale:
        try:
            subprocess.run([_CC] + CFLAGS + ["-shared", "-o", LIB_PATH, _SRC, "-lm"], check=True, capture_output=True, text=True)
        except (subprocess.CalledProcessError, FileNotFoundError) as e:   # keep a prebuilt .so usable on boxes without gcc
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"mipmap oracle build failed: {getattr(e, 'stderr', e)}")
    return LIB_PATH


class _OracleLib:
    """The CPU oracle's library with the two R12 entry points added (attribute lookup falls through to the oracle)."""

    def __init__(self, base: ctypes.CDLL, mips: ctypes.CDLL):
        self._base, self._mips = base, mips

    def __getattr__(self, name):
        if name in ("r3o_generate_mipmaps", "r3o_readback_texels"):
            return getattr(self._mips, name)
        return getattr(self._base, name)


def load_oracle_backend():
    """A rend3_b200.backend.Backend on the CPU oracle that also implements generate_mipmaps / readback_texels."""
    import oracle
    from rend3_b200.backend import Backend

    return Backend(_OracleLib(ctypes.CDLL(oracle.build()), ctypes.CDLL(build())), "r3o_", 0)
