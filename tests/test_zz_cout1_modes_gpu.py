"""The Cout = 1 convolution with ASB_COUT1_NO_MMA (conv_cout1_kernel takes the shapes of conv_cout1_mma_kernel) and
ASB_NO_COUT1 (the tensor-core convolution takes every Cout = 1 shape), against tests/ref64_mem.py.

Both variables are read once per process, so each mode runs in a child process that traces its own launch.  Once a
child has traced, short profiler captures in the parent process have come back without any kernel on a B200 (see the
comment above ``_MODE_SCRIPT`` in tests/test_seq_kernels_gpu.py): a persistent-kernel case of tests/test_schedule_gpu.py
that ran after such a child saw an empty trace.  pytest collects the files of a directory in name order, so this file
is named to run after every other file that profiles in its own process.  Keep child-process traces here.
"""
import os
import subprocess
import sys

import pytest
import torch

from artspeech_b200 import ops
from tests import test_mem_kernels_gpu as mem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_MODE_SCRIPT = r"""
import pathlib, sys, torch
sys.path.insert(0, sys.argv[1])
from artspeech_b200 import ops
from tests.test_schedule_gpu import launches
tmp = pathlib.Path(sys.argv[2])
d = torch.load(tmp / "in.pt")
pw = ops.pack_conv(d["w"].float(), d["bias"], d["taps"], d["x"].dtype, "cuda")
xg, lg = d["x"].cuda(), d["lens"].cuda()
(raw, act), ks = launches(lambda: ops.conv(xg, pw, raw=torch.float32, act_out=torch.float32, act=ops.ACT_TANH,
                                           scale=0.5, lens=lg), tmp, "mode")
torch.cuda.synchronize()
torch.save({"raw": raw.cpu(), "act": act.cpu(), "kernels": [k for k, _ in ks]}, tmp / "out.pt")
"""


@pytest.mark.parametrize("env,kernel,path", [("ASB_COUT1_NO_MMA", "conv_cout1_kernel<true>", "fp32"),
                                             ("ASB_NO_COUT1", "conv_halo_sw_kernel<16, 32, true>", None)])
def test_cout1_env_modes(env, kernel, path, tmp_path):
    """The vocoder's conv_post shape (Cin 32, 7 taps, bf16) with the mma kernel, or every Cout = 1 kernel, switched
    off; lens T, 255, 0."""
    x, w, bias, taps, lens = mem._c1_inputs(32, 7, 1, 1000, mem.BF16, 1.0, 17)
    torch.save({"x": x, "w": w, "bias": bias, "taps": taps, "lens": lens}, tmp_path / "in.pt")
    r = subprocess.run([sys.executable, "-c", _MODE_SCRIPT, ROOT, str(tmp_path)], env=dict(os.environ, **{env: "1"}),
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = torch.load(tmp_path / "out.pt")
    got = [k for k in res["kernels"] if k.split("<")[0] in mem.MEM_KERNELS + mem.CONV_KERNELS]
    assert got == [kernel], res["kernels"]
    mem._check(kernel, res["raw"], *mem._c1_ref(x, w, bias, taps, lens, 0.5, ops.ACT_NONE, mem.F32, path),
               f"{env} raw")
    mem._check(kernel, res["act"], *mem._c1_ref(x, w, bias, taps, lens, 0.5, ops.ACT_TANH, mem.F32, path),
               f"{env} tanh")
    print(f"[mem] {env}: {kernel}, worst err/bound {mem.WORST[kernel]:.3g}")
