"""Pins oracle/net_ref.py (the CPU fp32 restatement of the network) against
the golden head tensors the unmodified reference produced (tests/golden/net_*.npz),
at the benchmarked 512 x 512 shape too."""
import numpy as np
import pytest
import torch

import centerpose_b200 as cpb
from centerpose_b200 import synth
from oracle import net_ref
from tests.util import golden, golden_threads, net_case_inputs

CASES = ["net_dla34_b2_96x128", "net_dlav1_b1_64x64", "net_dla34track_b1_64x96"]


def _run_oracle(g):
    arch, trk = str(g["arch"]), bool(int(g["tracking"]))
    opt = cpb.default_opt(arch, tracking_task=trk)
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    sd = synth.seeded_state_dict(m, seed=int(g["wseed"]), offset_std=float(g["offset_std"]))
    x, extra = net_case_inputs(g)
    kw = {k: torch.from_numpy(v) for k, v in extra.items()}
    with golden_threads():
        return net_ref.forward(torch.from_numpy(x), sd, opt.heads, arch, **kw), opt


def _check_golden(name):
    g = golden(name)
    out, opt = _run_oracle(g)
    assert list(out) == list(opt.heads)
    for h in opt.heads:
        want = g["head_" + h]
        got = out[h].numpy()
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), h


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    _check_golden(name)


def test_oracle_matches_live_reference():
    """At the benchmarked 512 x 512 shape: the heads the reference computed on the same seeded weights and input."""
    _check_golden("net_dla34_b1_512")


def test_dcn_restatement_matches_reference_cpp():
    """oracle DCN vs the reference's own C++ CPU op (oracle/_ref, outputs committed as dcn_*.npz)."""
    from tests.util import dcn_case_inputs
    for name in ("dcn_small", "dcn_edge_big_offsets"):
        g = golden(name)
        x, off, mask, w, bias = [torch.from_numpy(a) for a in dcn_case_inputs(g)]
        got = net_ref.dcn_v2_forward_ref(x, off, mask, w, bias).numpy()
        assert np.abs(got - g["out"]).max() <= 1e-5


def test_dcn_zero_offset_identity():
    """DCNv2/testcuda.py:32-67 check_zero_offset: identity weights, zero offsets, mask 0.5 => 2*out == in."""
    x = torch.randn(2, 16, 7, 9, generator=torch.Generator().manual_seed(0))
    w = torch.zeros(16, 16, 3, 3)
    for c in range(16):
        w[c, c, 1, 1] = 1.0
    out = net_ref.dcn_v2_forward_ref(x, torch.zeros(2, 18, 7, 9), torch.full((2, 9, 7, 9), 0.5), w, torch.zeros(16))
    assert (2 * out - x).abs().max().item() <= 1e-6
