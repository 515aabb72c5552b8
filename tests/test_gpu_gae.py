"""The GAE kernel (roboy_gae) against a numpy float32 restatement of its operation order, bit for bit, and against a float64
reference within a bound derived from that order.  The library is built with -fmad=false, so the float32 order alone
fixes the result:
    nonterminal = done ? 0 : 1
    delta = (r + (gamma * V_next) * nonterminal) - V
    A     = delta + ((gamma * lam) * nonterminal) * A_next
    R     = A + V
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GAMMA, LAM = 0.99, 0.95
U32 = 2.0 ** -24


def gae_f32(rew, val, done, last, gamma, lam):
    f = np.float32
    g, gl = f(gamma), f(f(gamma) * f(lam))
    T = rew.shape[0]
    adv, ret = np.empty_like(rew), np.empty_like(rew)
    next_v, a = last.copy(), np.zeros_like(last)
    with np.errstate(all="ignore"):
        for t in range(T - 1, -1, -1):
            nt = np.where(done[t] != 0, f(0), f(1)).astype(np.float32)
            delta = (rew[t] + (g * next_v) * nt) - val[t]
            a = delta + (gl * nt) * a
            adv[t], ret[t] = a, a + val[t]
            next_v = val[t]
    return adv, ret


def gae_f64_with_bound(rew, val, done, last, gamma, lam):
    """Exact recurrence in float64 on the same float32 inputs (gamma, lam as their float32 values), and per element a bound
    on the float32 kernel's distance from it: each rounded operation adds at most u |its result|, and an error in A_next
    reaches A scaled by gamma lam nonterminal."""
    g = float(np.float32(gamma))
    gl = g * float(np.float32(lam))
    u = 1.01 * U32
    T = rew.shape[0]
    adv, ret, err_a, err_r = (np.empty(rew.shape) for _ in range(4))
    next_v, a, e = last.astype(np.float64), np.zeros(last.shape), np.zeros(last.shape)
    for t in range(T - 1, -1, -1):
        nt = np.where(done[t] != 0, 0.0, 1.0)
        r, v = rew[t].astype(np.float64), val[t].astype(np.float64)
        gv = g * next_v * nt
        delta = r + gv - v
        local = u * (2 * np.abs(gv) + np.abs(r + gv) + np.abs(delta))   # gamma*V, the add, the subtract
        ga = gl * nt * a
        local += u * (2 * gl * nt * np.abs(a) + np.abs(ga) + np.abs(delta + ga))   # gamma*lam, its products, the add
        e = local + gl * nt * e * (1 + 3 * u)
        a = delta + ga
        adv[t], err_a[t] = a, e
        ret[t] = a + v
        err_r[t] = e + u * np.abs(a + v) + u * e
        next_v = v
    return adv, ret, err_a, err_r


def run_gae(rew, val, done, last, gamma=GAMMA, lam=LAM, as_bool=False):
    from gym_roboy_b200.rollout import gae
    to = lambda a: torch.as_tensor(a, device=DEV)  # noqa: E731
    d = to(done != 0) if as_bool else to(done)
    adv, ret = gae(to(rew), to(val), d, to(last), gamma, lam)
    return adv.cpu().numpy(), ret.cpu().numpy()


def same_bits(x, y):
    """bit patterns equal, NaN at the same places (the payload of a NaN is not specified)"""
    nx, ny = np.isnan(x), np.isnan(y)
    return np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint32), y[~ny].view(np.uint32))


def inputs(T, n, seed, p_done=0.02):
    rng = np.random.default_rng(seed)
    rew = rng.normal(-3, 2, (T, n)).astype(np.float32)
    rew[rng.random((T, n)) < 0.01] = np.float32(999.0)
    val = rng.normal(-50, 10, (T, n)).astype(np.float32)
    done = (rng.random((T, n)) < p_done).astype(np.uint8)
    done[0, ::7] = 1                                  # ends at t = 0 and t = T - 1
    done[T - 1, 3::7] = 1
    done[:, 5::97] = 1                                # all-done rows
    done[done != 0] = rng.choice(np.array([1, 2, 128, 255], np.uint8), int((done != 0).sum()))   # any non-zero byte is done
    last = rng.normal(-50, 10, n).astype(np.float32)
    return rew, val, done, last


# stride of the kernel's grid-stride loop on a B200: 148 SMs x 8 CTAs x 256 threads = 303,104
@pytest.mark.parametrize("T,n", [(1, 1), (1, 4097), (7, 303_104 * 2 + 37), (64, 5000), (3, 303_103)])
@pytest.mark.parametrize("as_bool", [False, True])
def test_gae_is_the_float32_recurrence_bit_for_bit(T, n, as_bool):
    rew, val, done, last = inputs(T, n, T * 1000 + n % 1000)
    adv, ret = run_gae(rew, val, done, last, as_bool=as_bool)
    want_adv, want_ret = gae_f32(rew, val, done, last, GAMMA, LAM)
    assert same_bits(adv, want_adv) and same_bits(ret, want_ret)
    a64, r64, ea, er = gae_f64_with_bound(rew, val, done, last, GAMMA, LAM)
    assert (np.abs(adv - a64) <= ea).all() and (np.abs(ret - r64) <= er).all()
    assert ea.max() <= 1e-5 * np.abs(a64).max()       # (the bound is a few float32 ulps, not vacuous)


def test_gae_nan_and_infinities_propagate_as_in_float32():
    T, n = 6, 4096
    rew, val, done, last = inputs(T, n, 3)
    rew[2, 0:64] = np.nan
    val[3, 64:128] = np.inf                            # with done: 0 * inf = NaN, as in float32
    done[3, 64:96] = 1
    val[1, 128:160] = -np.inf
    last[160:192] = np.inf
    done[T - 1, 160:176] = 1                           # inf * nonterminal 0 -> NaN
    rew[4, 192:224] = np.inf
    rew[4, 224:256] = -np.inf
    val[4, 224:256] = -np.inf                          # -inf - -inf = NaN
    for gamma, lam in ((GAMMA, LAM), (1.0, 1.0), (0.0, 0.5)):
        adv, ret = run_gae(rew, val, done, last, gamma, lam)
        want_adv, want_ret = gae_f32(rew, val, done, last, gamma, lam)
        assert same_bits(adv, want_adv) and same_bits(ret, want_ret), (gamma, lam)
        assert np.isnan(adv).any() and np.isinf(adv).any()


@pytest.mark.parametrize("T,n", [(0, 100), (5, 0), (0, 0)])
def test_gae_of_an_empty_rollout_writes_nothing(T, n):
    import ctypes
    from gym_roboy_b200 import _native
    sentinel = -12345.0
    arena = torch.full((4096,), sentinel, dtype=torch.float32, device=DEV)
    dones = torch.full((64,), 7, dtype=torch.uint8, device=DEV)
    p = lambda t, off: ctypes.c_void_p(t.data_ptr() + 4 * off)  # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _native.check(_native.load().roboy_gae(T, n, p(arena, 0), p(arena, 512), ctypes.c_void_p(dones.data_ptr()), p(arena, 1024),
                                           GAMMA, LAM, p(arena, 2048), p(arena, 3072), stream))
    torch.cuda.synchronize()
    assert bool((arena == sentinel).all()) and bool((dones == 7).all())
