"""Profiling / experiment builds of the library: only the W = 4 unit (config C3) and the C-ABI unit.
usage: python profiles/build_variant.py <out.so> [extra nvcc flags, e.g. -DCYG_CTA_TIMING -DCYG_MAX_BLOCK_THREADS=768]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cygym_b200 import _capi  # noqa: E402

out = os.path.abspath(sys.argv[1])
log = _capi.compile_units(out, widths=(4,), extra=["-DCYG_FAST_BUILD"] + sys.argv[2:], obj_dir=os.path.join(os.path.dirname(out), "obj"))
print(out, "cyg_step_kernel<4, false, false> spill bytes:", _capi._step_kernel_spill(log))
