"""CPU checks of distance networks other than the shipped 256 x 4: which shapes the drop-in MPPI accepts, the C ABI's
n_hidden / hidden_width fields, and the library's own rejection of a shape outside the supported family."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from optimalmodulationds_b200.MPPI import _network_arrays
from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAMILY = "1 to 4 hidden layers of one width W <= 256"


def _net(d, O, layers, P=3):
    torch.manual_seed(0)
    return RobotSdfCollisionNet(in_channels=d + P, out_channels=O, skips=[], layers=layers)


@pytest.mark.parametrize("layers", [[128] * 2, [128] * 3, [64] * 4, [200] * 3, [256] * 1, [256] * 4])
@pytest.mark.parametrize("d,O", [(2, 1), (2, 2), (7, 7), (7, 9)])
def test_network_arrays_accepts_the_supported_family(layers, d, O):
    W, b = _network_arrays(_net(d, O, layers))
    L, width = len(layers), layers[0]
    assert len(W) == len(b) == L + 1
    assert tuple(W[0].shape) == (width, 3 * (d + 3))
    assert all(tuple(w.shape) == (width, width) for w in W[1:L])
    assert tuple(W[L].shape) == (O, width) and tuple(b[L].shape) == (O,)
    assert all(w.dtype == torch.float32 and w.is_contiguous() for w in W + b)


@pytest.mark.parametrize("layers", [[256, 128], [512] * 2, [256] * 5, []])
def test_network_arrays_rejects_other_shapes_and_names_the_family(layers):
    with pytest.raises(NotImplementedError, match=FAMILY):
        _network_arrays(_net(7, 9, layers))


def test_network_arrays_rejects_skip_connections():
    net = _net(7, 9, [128] * 3)
    net.model.skips = [1]          # what the reference's MLPRegression records for a network with skips
    with pytest.raises(NotImplementedError, match="skip"):
        _network_arrays(net)


@pytest.fixture(scope="module")
def capi():
    from optimalmodulationds_b200 import build, _capi
    build.build()
    _capi.load()
    return _capi


def test_net_shape_fields_match_the_c_compiler(capi, tmp_path):
    fields = ["n_point_dim", "n_hidden", "hidden_width", "W_host", "b_host"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dsmppi_b200.h"', 'int main(void){',
             'printf("size %zu\\n", sizeof(dsmppi_net));']
    lines += [f'printf("{f} %zu %zu\\n", offsetof(dsmppi_net, {f}), sizeof(((dsmppi_net*)0)->{f}));' for f in fields]
    lines.append('return 0;}')
    src = tmp_path / "net_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "net_layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = {l.split()[0]: [int(x) for x in l.split()[1:]] for l in subprocess.check_output([str(exe)], text=True).splitlines()}
    assert out["size"][0] == C.sizeof(capi.Net) == 4 * 4 + 10 * 8      # unchanged by the two int16 fields
    for f in fields:
        assert out[f] == [getattr(capi.Net, f).offset, getattr(capi.Net, f).size], f
    assert out["n_hidden"][0] == 12 and out["hidden_width"][0] == 14     # where `int32_t reserved` was


@pytest.mark.parametrize("n_hidden,width", [(5, 256), (-1, 128), (2, 257), (3, -4)])
def test_context_creation_rejects_an_unsupported_shape(capi, n_hidden, width):
    """Status 2 with a message naming the family, before any device is touched."""
    lib = capi.load()
    net = capi.Net()
    net.n_dof, net.n_out, net.n_point_dim = 2, 2, 3
    net.n_hidden, net.hidden_width = n_hidden, width
    W = [torch.zeros(256, 15)] + [torch.zeros(256, 256)] * 3 + [torch.zeros(2, 256)]
    b = [torch.zeros(256)] * 4 + [torch.zeros(2)]
    for i in range(5):
        net.W_host[i], net.b_host[i] = W[i].data_ptr(), b[i].data_ptr()
    dh = torch.zeros(3, 4)
    handle = C.c_void_p()
    assert lib.dsmppi_ctx_create(C.byref(handle), C.byref(net), dh.data_ptr(), 16, 0) == 2
    assert not handle.value
    assert b"1..4 hidden layers of one width 1..256" in lib.dsmppi_last_error()
