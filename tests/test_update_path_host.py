"""mr_dp_reduce_apply refuses bad arguments on the host, before any CUDA call.  CPU only: the pointers below are
integers that must never reach a kernel, so the test does not run where a CUDA device could execute one."""

import ctypes as C

import pytest

from movierec import _native as nat

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.skipif(torch.cuda.is_available(),
                                reason="fake device pointers: run only where a missing check cannot launch a kernel")

MR_ERR_INVALID = -1


def _peers(world, offset_rank=None, offset=4):
    return (C.c_void_p * world)(*[0x10000000 * (r + 1) + (offset if r == offset_rank else 0) for r in range(world)])


def _call(world=2, rank=0, lo=0, hi=64, grads=None, params=None, m=0x7000000, v=0x7100000, adam=True):
    grads = grads if grads is not None else _peers(max(world, 1))
    params = params if params is not None else _peers(max(world, 1))
    return nat.lib.mr_dp_reduce_apply(grads, params, world, rank, C.c_void_p(m) if m else None,
                                      C.c_void_p(v) if v else None, lo, hi, nat.OPT_ADAM if adam else nat.OPT_SGD,
                                      1e-3, 0.9, 0.999, 1e-7, 0.0, None, None, None)


@pytest.mark.parametrize("args", [
    dict(world=9, rank=0),                           # no kernel instance for 9 ranks
    dict(world=17, rank=0),
    dict(world=0, rank=0),
    dict(world=2, rank=2),                           # rank >= world
    dict(world=2, rank=-1),
    dict(lo=2),                                      # slice bounds not multiples of 4
    dict(hi=62),
    dict(lo=64, hi=60),
    dict(grads=_peers(2, offset_rank=1)),            # a peer pointer 4 bytes off
    dict(params=_peers(2, offset_rank=0)),
    dict(m=0x7000004),                               # Adam state read as float4: 16-byte alignment
    dict(v=0x7100008),
    dict(m=0),                                       # Adam without m
], ids=lambda a: "-".join("{}={}".format(k, v if isinstance(v, int) else "peers") for k, v in sorted(a.items())))
def test_dp_reduce_apply_refuses_on_the_host(args):
    assert _call(**args) == MR_ERR_INVALID
    assert "dp_reduce_apply" in nat.last_error()
