"""The CPU oracle with the death fog (tests/death_fog_oracle.h): the reference the device's fog is checked against.

The library is oracle/nmmo_oracle.c, unchanged but for two inserted lines: the include of death_fog_oracle.h just
before player_update, and `if (death_fog_update(e, row)) return;` where player_update's Resources.update part begins.
It is built into a temporary directory keyed by the sources' hash, and bound by a second instance of oracle/oracle.py,
so FogOracleEnv has exactly OracleEnv's interface.  With NC_DEATH_FOG = -1 it steps what OracleEnv steps
(test_death_fog.py::test_fog_oracle_without_fog_is_the_oracle).
"""
from __future__ import annotations

import hashlib
import importlib.util
import os
import subprocess
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
ORACLE_SRC = ROOT / "oracle" / "nmmo_oracle.c"
FOG_SRC = Path(__file__).resolve().parent / "death_fog_oracle.h"
SPEC_H = ROOT / "include" / "nmmo_spec.h"

_DEF = "static void player_update(OEnv *e, int row) {\n"
_HOOK = "  a[EA_TIME_ALIVE]++;\n  /* Resources.update */\n"


def _patched_source() -> str:
    src = ORACLE_SRC.read_text()
    for anchor in (_DEF, _HOOK):
        assert src.count(anchor) == 1, f"oracle/nmmo_oracle.c: expected one {anchor!r}"
    src = src.replace(_DEF, f'#include "{FOG_SRC}"\n' + _DEF)
    return src.replace(_HOOK, "  a[EA_TIME_ALIVE]++;\n  if (death_fog_update(e, row)) return;\n  /* Resources.update */\n")


def build() -> Path:
    src = _patched_source()
    key = hashlib.sha256((src + FOG_SRC.read_text() + SPEC_H.read_text()).encode()).hexdigest()[:16]
    out_dir = Path(tempfile.gettempdir()) / f"nmmo_b200_fog_oracle_{os.getuid()}_{key}"
    lib = out_dir / "libfogoracle.so"
    if lib.exists():
        return lib
    out_dir.mkdir(parents=True, exist_ok=True)
    c_file = out_dir / "nmmo_fog_oracle.c"
    c_file.write_text(src)
    tmp = out_dir / f"libfogoracle.{os.getpid()}.so"
    # the oracle's own flags (oracle/Makefile); -I oracle/ resolves its "../include/nmmo_spec.h"
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fPIC", "-Wall", "-Wno-stringop-overflow", "-I", str(ORACLE_SRC.parent),
                           "-shared", "-o", str(tmp), str(c_file), "-lm"])
    os.replace(tmp, lib)
    return lib


def _binding():
    spec = importlib.util.spec_from_file_location("fog_oracle_binding", ROOT / "oracle" / "oracle.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod._LIB = build()
    mod.build = lambda force=False: mod._LIB
    return mod


_mod = _binding()
FogOracleEnv = _mod.OracleEnv
