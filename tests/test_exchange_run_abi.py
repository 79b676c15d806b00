"""CPU-side checks of pf_exchange_run's ABI: the ctypes mirrors have the sizes the library was built
with, and the in-process communicator is created, handed out per rank and destroyed without a GPU."""
import ctypes

import pytest

from panfeed_b200 import capi


def test_exchange_struct_mirrors_match_the_library():
    lib = capi.load()
    assert lib.pf_struct_size(9) == ctypes.sizeof(capi.Comm)
    assert lib.pf_struct_size(10) == ctypes.sizeof(capi.ExchangeResult)
    assert ctypes.sizeof(capi.ExchangeResult) == 2 * ctypes.sizeof(capi.ExchangeNs) == 2 * 56


@pytest.mark.parametrize("world", [1, 2, 5, 32])
def test_local_comm_hands_out_every_rank(world):
    g = capi.LocalComm(world)
    users = set()
    for r in range(world):
        c = g.get(r)
        assert (c.rank, c.world) == (r, world)
        assert c.all_gather and c.all_to_all_v
        users.add(c.user)
    assert len(users) == world                   # one state per rank
    with pytest.raises(capi.PfError):
        g.get(world)
    g.abort()
    g.close()
    g.close()


@pytest.mark.parametrize("world", [0, 33])
def test_local_comm_refuses_a_bad_world(world):
    with pytest.raises(capi.PfError):
        capi.LocalComm(world)


def test_exchange_run_refuses_null_arguments():
    lib = capi.load()
    assert lib.pf_exchange_run(None, None, 0, None) == -1
    assert lib.pf_exchange_release(None, None) == -1
