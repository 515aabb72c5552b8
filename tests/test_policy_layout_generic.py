"""The policy image of `roboy_policy_rollout` for every robot (`roboy_policy_layout`, include/roboy_b200.h), on the CPU."""
import numpy as np
import pytest
import torch

from gym_roboy_b200 import _native as N
from gym_roboy_b200.rollout import MlpPolicy, pack_policy_image

H = 64


def header_formula(D, A):
    """The layout as the header comment states it."""
    a8 = -(-A // 8) * 8
    net = lambda W: dict(W1=0, B1=64 * D, W2=64 * D + 64, B2=64 * D + 4160, W3=64 * D + 4224, B3=64 * D + 4224 + 64 * W,  # noqa: E731
                         size=64 * D + 4224 + 65 * W)
    vf, pi = net(8), net(a8)
    std = vf["size"] + pi["size"]
    lognorm = std + a8
    return vf, pi, 0, vf["size"], std, lognorm, -(-(lognorm + 1) // 4) * 4, a8


def test_layout_for_every_robot():
    for J in range(1, 16):
        for A in range(1, 65):
            D = 3 * J
            off = N.policy_layout(D, A)
            vf, pi, o_vf, o_pi, o_std, o_ln, total, a8 = header_formula(D, A)
            assert [off[k] for k in (N.POLICY_LAYOUT_W1, N.POLICY_LAYOUT_B1, N.POLICY_LAYOUT_W2, N.POLICY_LAYOUT_B2,
                                     N.POLICY_LAYOUT_W3)] == [vf[k] for k in ("W1", "B1", "W2", "B2", "W3")]
            assert off[N.POLICY_LAYOUT_VF_B3] == vf["B3"] and off[N.POLICY_LAYOUT_PI_B3] == pi["B3"]
            assert (off[N.POLICY_LAYOUT_VF], off[N.POLICY_LAYOUT_PI], off[N.POLICY_LAYOUT_STD], off[N.POLICY_LAYOUT_LOGNORM],
                    off[N.POLICY_LAYOUT_FLOATS]) == (o_vf, o_pi, o_std, o_ln, total)
            # every section 16-byte aligned; the sections tile the image in order, without gaps or overlaps
            sections = []
            for base, b3, W in ((o_vf, vf["B3"], 8), (o_pi, pi["B3"], a8)):
                sections += [(base, base + 64 * D), (base + 64 * D, base + 64 * D + 64), (base + 64 * D + 64, base + 64 * D + 64 + 4096),
                             (base + 64 * D + 4160, base + 64 * D + 4224), (base + 64 * D + 4224, base + b3), (base + b3, base + b3 + W)]
            sections += [(o_std, o_std + a8), (o_ln, o_ln + 1)]
            for (s0, e0), (s1, _) in zip(sections, sections[1:]):
                assert s0 % 4 == 0 and e0 == s1, (J, A, sections)
            assert sections[-1][1] <= total < sections[-1][1] + 4 and total % 4 == 0
    msj = N.policy_layout(9, 8)
    assert (msj[N.POLICY_LAYOUT_B1], msj[N.POLICY_LAYOUT_W2], msj[N.POLICY_LAYOUT_B2], msj[N.POLICY_LAYOUT_W3],
            msj[N.POLICY_LAYOUT_VF_B3], msj[N.POLICY_LAYOUT_PI_B3]) == (N.POLICY_OFF_B1, N.POLICY_OFF_W2, N.POLICY_OFF_B2,
                                                                        N.POLICY_OFF_W3, N.POLICY_OFF_B3, N.POLICY_OFF_B3)
    assert msj[N.POLICY_LAYOUT_PI_B3] + 8 == N.POLICY_NET_FLOATS
    assert (msj[N.POLICY_LAYOUT_VF], msj[N.POLICY_LAYOUT_PI], msj[N.POLICY_LAYOUT_STD], msj[N.POLICY_LAYOUT_LOGNORM],
            msj[N.POLICY_LAYOUT_FLOATS]) == (N.POLICY_OFF_VF, N.POLICY_OFF_PI, N.POLICY_OFF_STD, N.POLICY_OFF_LOGNORM,
                                             N.POLICY_IMAGE_FLOATS)


@pytest.mark.parametrize("dims", [(0, 8), (10, 8), (48, 8), (9, 0), (9, 65), (-3, 4)])
def test_layout_refuses_other_dims(dims):
    with pytest.raises(N.RoboyNativeError):
        N.policy_layout(*dims)


@pytest.mark.parametrize("J,A", [(1, 1), (2, 5), (6, 14), (5, 11), (3, 8), (15, 64), (10, 33)])
def test_packed_image_reproduces_the_torch_forward_pass(J, A):
    """The image decoded with nothing but the header formula gives the torch policy's mean, value, std and log-density
    constant (float32 rounding); the MSJ image is the one the MSJ layout constants describe."""
    D = 3 * J
    torch.manual_seed(J * 100 + A)
    pol = MlpPolicy(D, A)
    with torch.no_grad():
        pol.log_std.copy_(torch.linspace(-1.2, 0.4, A))
    img = pack_policy_image(pol).numpy().astype(np.float64)
    vf, pi, o_vf, o_pi, o_std, o_ln, total, a8 = header_formula(D, A)
    assert img.size == total
    obs = torch.randn(257, D)

    def fwd(base, L, W):
        w1 = img[base + L["W1"]: base + L["B1"]].reshape(D, H)
        b1 = img[base + L["B1"]: base + L["W2"]]
        w2 = img[base + L["W2"]: base + L["B2"]].reshape(H, H)
        b2 = img[base + L["B2"]: base + L["W3"]]
        w3 = img[base + L["W3"]: base + L["B3"]].reshape(H, W)
        b3 = img[base + L["B3"]: base + L["B3"] + W]
        return np.tanh(np.tanh(obs.double().numpy() @ w1 + b1) @ w2 + b2) @ w3 + b3

    with torch.no_grad():
        mean, value = pol(obs)
    m = fwd(o_pi, pi, a8)
    v = fwd(o_vf, vf, 8)
    assert np.allclose(m[:, :A], mean.double().numpy(), rtol=1e-5, atol=1e-6)
    assert np.all(m[:, A:] == 0) and np.all(v[:, 1:] == 0)
    assert np.allclose(v[:, 0], value.double().numpy(), rtol=1e-5, atol=1e-6)
    assert np.array_equal(img[o_std: o_std + A], pol.log_std.detach().exp().double().numpy())
    assert np.all(img[o_std + A: o_ln] == 0)
    assert np.isclose(img[o_ln], -0.5 * np.log(2 * np.pi) * A - float(pol.log_std.sum()), rtol=1e-6)
    if (J, A) == (3, 8):
        assert (o_pi, o_std, o_ln, total) == (N.POLICY_OFF_PI, N.POLICY_OFF_STD, N.POLICY_OFF_LOGNORM, N.POLICY_IMAGE_FLOATS)


def test_pack_asserts_the_shapes():
    pol = MlpPolicy(18, 14)
    pol.pi[4] = torch.nn.Linear(64, 13)   # an output layer that does not match act_dim
    with pytest.raises(AssertionError):
        pack_policy_image(pol)
