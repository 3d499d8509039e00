"""CPU-side checks of the value-network action choice (snp_value_lookahead, CrowdEngine.set_value_network / predict): every bad
argument is refused before anything touches the device (the pointers are dummies), the network is packed in the documented layout,
networks the kernel does not evaluate are refused, and the kernel compiles for sm_100a without spills."""
import ctypes
import os
import re
import subprocess
import tempfile

import pytest
import torch

DUMMY = ctypes.c_void_p(4096)
E, N, A = 3, 700, 81
CADRL = [13, 150, 100, 100, 1]


def _crowd(L, **kw):
    args = dict(E=E, N=N, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY, robot=DUMMY)
    args.update(kw)
    return L.SnpCrowd(**args)


def _args(L, widths=CADRL, **kw):
    g = L.SnpValueArgs(type=3, A=A, theta_and_omega_visible=0, next=DUMMY, actions=DUMMY, dt=0.25, gamma=0.9, layers=len(widths) - 1,
                       weights=DUMMY, values=DUMMY, best=DUMMY, reached=DUMMY)
    g.widths = (ctypes.c_int32 * 7)(*(list(widths) + [0] * (7 - len(widths))))
    for k, v in kw.items():
        setattr(g, k, v)
    return g


CASES = ["null_crowd", "null_args", "E0", "N0", "E_big", "A0", "A_big", "no_dyn", "no_stat", "no_robot", "no_next", "no_actions", "no_weights",
         "no_values", "no_best", "no_reached", "type9", "dtype", "layers0", "layers7", "input12", "input15_hidden", "input13_visible",
         "last2", "hidden0", "hidden257"]


@pytest.mark.parametrize("case", CASES)
def test_value_lookahead_refuses_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    c, g = _crowd(L), _args(L)
    if case == "null_crowd":
        rc = lib.snp_value_lookahead(None, ctypes.byref(g), None)
    elif case == "null_args":
        rc = lib.snp_value_lookahead(ctypes.byref(c), None, None)
    else:
        if case in ("E0", "N0"):
            c = _crowd(L, **{case[0]: 0})
        elif case == "E_big":
            c = _crowd(L, E=65536)
        elif case == "A0":
            g.A = 0
        elif case == "A_big":
            g.A = 65536
        elif case in ("no_dyn", "no_stat", "no_robot"):
            c = _crowd(L, **{case[3:]: None})
        elif case.startswith("no_"):
            setattr(g, case[3:], None)
        elif case == "type9":
            g.type = 9
        elif case == "dtype":
            c = _crowd(L, dtype=7)
        elif case == "layers0":
            g.layers = 0
        elif case == "layers7":
            g = _args(L, widths=[13, 8, 8, 8, 8, 8, 1])
            g.layers = 7
        elif case == "input12":
            g = _args(L, widths=[12, 150, 1])
        elif case == "input15_hidden":
            g = _args(L, widths=[15, 150, 1])
        elif case == "input13_visible":
            g.theta_and_omega_visible = 1
        elif case == "last2":
            g = _args(L, widths=[13, 150, 2])
        elif case == "hidden0":
            g = _args(L, widths=[13, 150, 0, 1])
        elif case == "hidden257":
            g = _args(L, widths=[13, 257, 1])
        rc = lib.snp_value_lookahead(ctypes.byref(c), ctypes.byref(g), None)
    assert rc == -1, case
    assert "snp_value_lookahead" in lib.snp_last_error().decode(), case


def _cadrl_sequential(seed, widths=CADRL):
    torch.manual_seed(seed)
    layers = []
    for i in range(len(widths) - 1):
        layers.append(torch.nn.Linear(widths[i], widths[i + 1]))
        if i + 2 < len(widths):
            layers.append(torch.nn.ReLU())
    return torch.nn.Sequential(*layers)


def test_set_value_network_packs_the_documented_layout():
    """Layer by layer: W transposed ([in][out] row-major) then b; unpacked, it is the state_dict."""
    from social_navigation_pyenvs_b200.engine import value_network_layout
    for widths in (CADRL, [15, 7, 1], [13, 1]):
        net = _cadrl_sequential(3, widths)
        got_widths, packed = value_network_layout(net)
        assert got_widths == widths
        assert packed.dtype == torch.float32 and packed.device.type == "cpu"
        sd, off = net.state_dict(), 0
        for i in range(len(widths) - 1):
            k, o = widths[i], widths[i + 1]
            W = packed[off:off + k * o].reshape(k, o).t()
            off += k * o
            b = packed[off:off + o]
            off += o
            assert torch.equal(W, sd[f"{2 * i}.weight"]) and torch.equal(b, sd[f"{2 * i}.bias"])
        assert off == packed.numel()


def test_a_cadrl_value_network_qualifies_directly_and_through_its_attribute():
    """CADRL's ValueNetwork holds its mlp in `value_network`; the module itself and that attribute pack alike."""
    from social_navigation_pyenvs_b200.engine import value_network_layout

    class ValueNetwork(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.value_network = _cadrl_sequential(5)

        def forward(self, state):
            return self.value_network(state)

    vn = ValueNetwork()
    a, b = value_network_layout(vn), value_network_layout(vn.value_network)
    assert a[0] == b[0] == CADRL and torch.equal(a[1], b[1])


@pytest.mark.parametrize("case", ["tanh", "relu_last", "out2", "two_linears", "input14", "wide", "seven_layers", "empty"])
def test_set_value_network_refuses_what_the_kernel_does_not_evaluate(case):
    from social_navigation_pyenvs_b200.engine import value_network_layout
    nn = torch.nn
    if case == "tanh":
        net = nn.Sequential(nn.Linear(13, 150), nn.Tanh(), nn.Linear(150, 1))
    elif case == "relu_last":
        net = nn.Sequential(nn.Linear(13, 150), nn.ReLU(), nn.Linear(150, 1), nn.ReLU())
    elif case == "out2":
        net = nn.Sequential(nn.Linear(13, 150), nn.ReLU(), nn.Linear(150, 2))
    elif case == "two_linears":
        net = nn.Sequential(nn.Linear(13, 150), nn.Linear(150, 1))
    elif case == "input14":
        net = nn.Sequential(nn.Linear(14, 150), nn.ReLU(), nn.Linear(150, 1))
    elif case == "wide":
        net = nn.Sequential(nn.Linear(13, 257), nn.ReLU(), nn.Linear(257, 1))
    elif case == "seven_layers":
        net = _cadrl_sequential(0, [13] + [8] * 6 + [1])
    else:
        net = nn.Sequential()
    with pytest.raises(ValueError):
        value_network_layout(net)


def test_value_kernel_compiles_for_sm100a_without_spills():
    """csrc/snp_value.cu under the build's flags with -Xptxas -v: no kernel spills or keeps a stack frame (DESIGN 4.7 states the
    register counts)."""
    from social_navigation_pyenvs_b200 import build
    with tempfile.TemporaryDirectory() as tmp:
        cmd = ["nvcc", "-Xptxas=-v", *build.NVCC_FLAGS, "-c", os.path.join(build.CSRC, "snp_value.cu"), "-o", os.path.join(tmp, "v.o")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'", r.stderr)
    assert sum("k_value" in k for k in kernels) == 6, kernels  # k_value (weights staged or not) and k_value_fold, fp32 and fp64
    frames = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(frames) >= 6 and all(f == ("0", "0", "0") for f in frames), frames
