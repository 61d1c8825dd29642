"""GPU: the persistent GEMM / conv kernel (IMAGD_GEMM_PERSISTENT=1) on multi-wave problems with every LINEAR epilogue
ingredient.

The library reads the switch once per process, so a process started without it cannot reach the persistent kernel. There
the `persistent` fixture runs this module once in a child process with the switch on, and each test asserts the outcome its
own id had in that run."""
import os
import subprocess
import sys
import xml.etree.ElementTree as ET

import pytest
import torch

from conftest import rel_l2
from oracle import ops_ref

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
SWITCH_ON = os.environ.get("IMAGD_GEMM_PERSISTENT") == "1"


@pytest.fixture(scope="module")
def persistent(cuda_device, tmp_path_factory):
    """None when this process has the switch on; otherwise {test name: (outcome, message)} of the module run with it on."""
    if SWITCH_ON:
        return None
    report = tmp_path_factory.mktemp("persist") / "report.xml"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        f"--junitxml={report}"], cwd=root, env=dict(os.environ, IMAGD_GEMM_PERSISTENT="1"),
                       capture_output=True, text=True, timeout=1200)
    assert report.exists(), r.stdout[-3000:] + r.stderr[-3000:]
    out = {}
    for case in ET.parse(report).iter("testcase"):
        bad = [c for c in case if c.tag in ("failure", "error", "skipped")]
        out[case.get("name")] = (bad[0].tag, (bad[0].get("message") or "")[:2000]) if bad else ("passed", "")
    return out


def _ran_with_switch_on(persistent, request):
    """True when this process must run the test body itself; otherwise checks the child run's outcome for this id."""
    if persistent is None:
        return True
    outcome, msg = persistent.get(request.node.name, ("missing", "not reported by the IMAGD_GEMM_PERSISTENT=1 run"))
    assert outcome == "passed", f"{request.node.name} with IMAGD_GEMM_PERSISTENT=1: {outcome}: {msg}"
    return False


def _rand(shape, dev, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


@pytest.mark.parametrize("M,N,K", [(65536, 320, 320), (65536, 960, 320), (16384, 640, 2560), (40000, 328, 72),
                                   (70000, 64, 640), (33000, 136, 128)])
def test_persistent_gemm(cuda_device, persistent, request, M, N, K):
    if not _ran_with_switch_on(persistent, request):
        return
    from imagdressing_b200 import ops

    a, w = _rand((M, K), cuda_device, 1).to(BF), _rand((N, K), cuda_device, 2, K ** -0.5).to(BF)
    b, res = _rand((N,), cuda_device, 3), _rand((M, N), cuda_device, 4).to(BF)
    out = ops.gemm(a, w, bias=b, residual=res)
    assert rel_l2(out, ops_ref.gemm_ref(a, w, b, residual=res)) < 1e-2
    assert torch.equal(out, ops.gemm(a, w, bias=b, residual=res))
    plain = ops.gemm(a, w)
    assert rel_l2(plain, ops_ref.gemm_ref(a, w)) < 1e-2


@pytest.mark.parametrize("NB,H,W,Cin,Cout", [(16, 64, 64, 320, 320), (16, 32, 32, 640, 640), (16, 16, 16, 1280, 1280),
                                             (5, 80, 64, 320, 320), (9, 24, 18, 128, 64)])
def test_persistent_conv3x3(cuda_device, persistent, request, NB, H, W, Cin, Cout):
    if not _ran_with_switch_on(persistent, request):
        return
    from imagdressing_b200 import ops

    x = _rand((NB, H, W, Cin), cuda_device, 13).to(BF)
    w = _rand((Cout, Cin, 3, 3), cuda_device, 14, (9 * Cin) ** -0.5).to(BF)
    bias, temb = _rand((Cout,), cuda_device, 15), _rand((NB, Cout), cuda_device, 16)
    res = _rand((NB, H, W, Cout), cuda_device, 17).to(BF)
    out = ops.conv3x3(x, ops_ref.conv3x3_pack(w), bias=bias, rowvec=temb, residual=res)
    assert rel_l2(out, ops_ref.conv3x3_ref(x, w, bias, temb, res)) < 1e-2
