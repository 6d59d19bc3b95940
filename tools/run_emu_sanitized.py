"""Runs the emulator parity suites against a sanitizer build of the host-emulation library, so that every parity case
doubles as a check of the kernels' index math.

AddressSanitizer (red zones between the arena sub-buffers, exactly sized shared memory per launch):
    LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0 python tools/run_emu_sanitized.py
UndefinedBehaviorSanitizer, trapping (misaligned float2 / float4 accesses, signed overflow, shifts):
    python tools/run_emu_sanitized.py --ubsan

Race check of the shared-memory exchanges (plain emulator build; the emulated threads of a block run one after the
other up to their next barrier, in this order -- a missing barrier gives a stale or poisoned read under one of them):
    python tools/run_emu_sanitized.py --order reverse
    python tools/run_emu_sanitized.py --order shuffle

A few minutes each; the CPU suite itself runs the shorter tests/test_abi_walk.py.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.chdir(ROOT)

from libmultiviewnative_b200 import _build  # noqa: E402

args = sys.argv[1:]
ubsan = "--ubsan" in args
args = [a for a in args if a != "--ubsan"]
order = None
if "--order" in args:
    i = args.index("--order")
    order = args[i + 1]
    del args[i:i + 2]
    os.environ["LMVN_EMU_ORDER"] = order
if order is None and not ubsan and "libasan" not in os.environ.get("LD_PRELOAD", ""):
    sys.exit("preload libasan (see the docstring): the interpreter itself is not an AddressSanitizer build")
_path = _build.build_emu() if order else (_build.build_emu(ubsan=True) if ubsan else _build.build_emu(asan=True))
_build.build_emu = lambda force=False, asan=False, ubsan=False: _path  # the fixtures load whatever build_emu() returns

import pytest  # noqa: E402

sys.exit(pytest.main(["-x", "-q", "-m", "not gpu", "tests/test_emu_parity.py", "tests/test_slabs_emu.py",
                      "tests/test_call_history.py", "tests/test_generic_extents.py"] + args))
