"""The chain-move entries of the C ABI as a whole: their cached CUDA graphs follow option changes,
and every entry refuses bad arguments with the same message."""
import ctypes as C
import math
import struct

import numpy as np
import pytest

import raytracerfortran_b200 as rt
from raytracerfortran_b200 import _lib, chains

from test_gpu_chains import _dev, _setup

pytestmark = pytest.mark.gpu


def test_the_two_likelihood_constants_differ_for_13_sources():
    n = 13.0
    reference = math.log(1.0 / math.pow(2.0 * math.pi, n / 2.0))
    stable = -(n / 2.0) * math.log(2.0 * math.pi)
    assert struct.pack("<d", reference) != struct.pack("<d", stable)


def _moves_then_option_change(option, fresh_capture, graph):
    """One call with `option` at 0, one with it at 1 on the same buffers.  With `fresh_capture`, a
    call on other buffers in between makes the second call capture its graph anew."""
    import torch
    B, ldk, nsrc, n_moves = 400, 6, 13, 5
    k, voro, so, sd, tobs, sigma, ll = _setup(B, ldk, nsrc, 71)
    prior, sd_prior, pk = chains.prior_array(), chains.sd_prior_array(), chains.poisson_pk(3.01, 1, ldk)
    prior[:2] /= 10.0
    beta = np.ones(B)

    def chain_set():
        tk, tv, tl, tg, tb, ts, td, to = _dev(k, voro, ll, sigma, beta, so, sd, tobs)
        if graph:
            g = chains.McmcGraph(tk, tv, tl, tg, tb, n_moves, prior, sd_prior, pk, 1, ldk, ts, td, to, seed=3)
            return (tv, tl), lambda gen: g.run(1)
        pos = torch.zeros(B, dtype=torch.int32, device="cuda")
        return (tv, tl), lambda gen: chains.mh_moves_device(tk, tv, tl, pos, n_moves, tb, tg, prior, ts, td, to,
                                                            generator=gen)

    (tv, tl), run = chain_set()
    gen = torch.Generator(device="cuda").manual_seed(5)
    try:
        rt.set_option(option, 0)
        run(gen)
        rt.set_option(option, 1)
        if fresh_capture:
            chain_set()[1](torch.Generator(device="cuda").manual_seed(6))
        run(gen)
        torch.cuda.synchronize()
    finally:
        rt.set_option(option, 0)
    return tv.cpu().numpy(), tl.cpu().numpy()


@pytest.mark.parametrize("graph", [False, True], ids=["mh_moves_device", "McmcGraph"])
@pytest.mark.parametrize("option", ["stable_lognorm", "logl_shuffle"])
def test_a_changed_option_takes_effect_on_the_next_graph_call(option, graph):
    """A replayed graph computes what a graph captured under the current options computes."""
    v_replay, l_replay = _moves_then_option_change(option, False, graph)
    v_fresh, l_fresh = _moves_then_option_change(option, True, graph)
    assert np.array_equal(v_replay.view(np.uint64), v_fresh.view(np.uint64))
    assert np.array_equal(l_replay.view(np.uint64), l_fresh.view(np.uint64))


def _entries():
    """The six chain-move entries, each called with valid arguments unless a keyword overrides one."""
    import torch
    B, ldk, nsrc, M = 8, 6, 4, 2
    f = lambda *shape: torch.zeros(shape, dtype=torch.float64, device="cuda")
    i = lambda *shape: torch.ones(shape, dtype=torch.int32, device="cuda")
    k, voro, logL, sigma, beta, so, sd, tobs = i(B), f(B, 2, ldk), f(B), f(B), f(B), f(nsrc), f(nsrc), f(nsrc)
    idxar, arpar, pos, acc = i(B), f(B), i(B), i(M, B)
    dev_m, int_m = f(M, B), i(M, B)
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    tally = torch.zeros((5, B), dtype=torch.int64, device="cuda")
    work = torch.zeros(_lib.load().rtb200_mcmc_workspace_bytes(B, M), dtype=torch.uint8, device="cuda")
    dp = C.POINTER(C.c_double)
    host = {"prior": chains.prior_array(), "sd_prior": chains.sd_prior_array(), "ar_prior": chains.ar_prior_array(),
            "pk": chains.poisson_pk(3.01, 1, ldk)}
    p = lambda t: t.data_ptr()
    base = dict(k=p(k), voro=p(voro), logL=p(logL), sigma=p(sigma), beta=p(beta), B=B, ldk=ldk, so=p(so),
                sd=p(sd), tobs=p(tobs), NSrc=nsrc, accept=p(acc), stream=None, enos=0, u=p(dev_m), iu=p(int_m),
                n_moves=M, kmin=1, kmax=ldk, idxar=p(idxar), arpar=p(arpar), pos=p(pos), counter=p(counter),
                work=p(work), tally=p(tally), **{n: a.ctypes.data_as(dp) for n, a in host.items()})
    lib = _lib.load()
    orders = {
        "rtb200_mh_step_device": (lib.rtb200_mh_step_device_ev,
            "k voro logL B ldk iu iu u u beta sigma prior so sd tobs NSrc accept stream none enos"),
        "rtb200_mh_moves_device": (lib.rtb200_mh_moves_device_ex,
            "k voro logL B ldk n_moves iu iu u u beta sigma prior so sd tobs NSrc accept stream enos"),
        "rtb200_bd_step_device": (lib.rtb200_bd_step_device_ex,
            "k voro logL B ldk u iu u u u beta sigma prior pk kmin kmax so sd tobs NSrc accept stream enos"),
        "rtb200_sd_step_device": (lib.rtb200_sd_step_device,
            "k voro logL sigma B ldk u u u beta sd_prior so sd tobs NSrc accept stream"),
        "rtb200_ar_step_device": (lib.rtb200_ar_step_device,
            "k voro logL sigma idxar arpar B ldk u u u u beta ar_prior so sd tobs NSrc accept stream"),
        "rtb200_mcmc_iterations_device": (lib.rtb200_mcmc_iterations_device,
            "k voro logL sigma beta pos B ldk n_moves prior sd_prior pk kmin kmax enos so sd tobs NSrc seed "
            "counter work tally one idxar arpar ar_prior stream"),
    }
    base.update(none=None, seed=1, one=1)
    keep = (k, voro, logL, sigma, beta, so, sd, tobs, idxar, arpar, pos, acc, dev_m, int_m, counter, tally, work, host)

    def call(name, **bad):
        fn, order = orders[name]
        args = {**base, **bad}
        return fn(*[args[a] for a in order.split()])
    call.keep_alive = keep                  # base holds raw pointers into these
    return call


_COMMON = [({"ldk": 0}, "{} supports 1..64 nodes per state"), ({"ldk": 65}, "{} supports 1..64 nodes per state"),
           ({"NSrc": 0}, "{} needs at least one source")]
_REFUSALS = {
    "rtb200_mh_step_device": [({"prior": None}, "{} needs the prior array")],
    "rtb200_mh_moves_device": [({"prior": None}, "{} needs the prior array"),
                               ({"n_moves": 513}, "{}: at most 512 moves per call")],
    "rtb200_bd_step_device": [({"prior": None}, "{} needs the prior array"),
                              ({"kmin": 0}, "{} needs 1 <= kmin <= kmax <= ldk"),
                              ({"kmin": 4, "kmax": 3}, "{} needs 1 <= kmin <= kmax <= ldk"),
                              ({"kmax": 7}, "{} needs 1 <= kmin <= kmax <= ldk")],
    "rtb200_sd_step_device": [({"sd_prior": None}, "{} needs the sd_prior array")],
    "rtb200_ar_step_device": [({"ar_prior": None}, "{} needs the ar_prior array")],
    "rtb200_mcmc_iterations_device": [
        ({"prior": None}, "{} needs the prior and sd_prior arrays"),
        ({"sd_prior": None}, "{} needs the prior and sd_prior arrays"),
        ({"kmin": 0}, "{} needs 1 <= kmin <= kmax <= ldk"),
        ({"kmax": 7}, "{} needs 1 <= kmin <= kmax <= ldk"),
        ({"n_moves": 510}, "{}: at most 509 moves per iteration"),
        ({"n_moves": -1}, "{}: at most 509 moves per iteration"),
        ({"idxar": None}, "{}: the AR move needs idxar, arpar and ar_prior together"),
        ({"arpar": None}, "{}: the AR move needs idxar, arpar and ar_prior together"),
        ({"ar_prior": None}, "{}: the AR move needs idxar, arpar and ar_prior together"),
        ({"counter": None}, "{} needs counter, workspace and pos"),
        ({"work": None}, "{} needs counter, workspace and pos"),
        ({"pos": None}, "{} needs counter, workspace and pos")],
}


@pytest.mark.parametrize("name", sorted(_REFUSALS))
def test_move_entries_refuse_bad_arguments(name):
    """Each bad argument is refused before any work, with the entry's own message."""
    call = _entries()
    for bad, message in _COMMON + _REFUSALS[name]:
        rc = call(name, **bad)
        assert rc != 0, (name, bad)
        assert _lib.last_error() == message.format(name), (name, bad)
