"""CPU: the per-thread stack frame of every kernel of libsb_b200.so stays within what the rule recursion leaves room for.

The thread engine's rules recurse on the per-thread stack, whose size sb_create sets to 48 KB (cudaLimitStackSize, DESIGN.md
section 2): about 700 bytes per nesting level and MAXDEPTH 60 levels leave room for a kernel frame of at most 6,144 bytes,
the frame of k_env_step_heur, the largest that runs the recursion today.  A kernel with a larger frame would overflow the
stack on a deep trigger chain, so every kernel, present and future, is held to that bound.  cuobjdump ships with the CUDA
toolkit and reads the frames from the library without a GPU."""
import os
import re
import shutil
import subprocess

import pytest

MAX_STACK = 6144
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def cuobjdump():
    for c in (os.path.join(CUDA, "bin", "cuobjdump"), shutil.which("cuobjdump")):
        if c and os.path.exists(c):
            return c
    pytest.fail("cuobjdump not found (CUDA toolkit at %s)" % CUDA)


def kernel_frames():
    """{mangled kernel name: STACK bytes} of the built library"""
    import __graft_entry__ as g
    g.build()
    from monsoon_b200 import _lib
    out = subprocess.run([cuobjdump(), "-res-usage", _lib.SO_PATH], check=True, capture_output=True, text=True).stdout
    frames = dict(re.findall(r"Function (\S+):\s*\n\s*REG:\d+ STACK:(\d+)", out))
    return {k: int(v) for k, v in frames.items()}


def test_every_kernel_frame_fits_the_recursion_limit():
    frames = kernel_frames()
    assert len(frames) > 50, "cuobjdump listed %d kernels" % len(frames)
    for name in ("k_env_step_heur", "k_search_simulate", "k_ismcts_begin", "k_ismcts_simulate", "k_ismcts_end"):
        assert any(name in k for k in frames), name
    over = {k: v for k, v in frames.items() if v > MAX_STACK}
    assert not over, over
