"""Host-side pieces of the pixel <-> pixel losses over the global batch (no GPU needed): the C ABI's argument checks of the
bulk row exchange and the state helpers, and the size of the records the exchange carries."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from slcl import _lib
    try:
        return _lib.load()
    except _lib.SlclError:
        pytest.skip("libslcl.so not built")


def test_rows_region_and_allgather_arguments(lib):
    from slcl import _lib
    assert lib.slcl_peer_rows_region_bytes(1 << 20) == 512 + 2 * (1 << 20)
    assert lib.slcl_peer_rows_region_bytes(24) == 0                        # slots are whole 16-byte words
    peer = _lib.PeerT(16, 0, 2, 64, 1.0)
    assert lib.slcl_peer_allgather(None, 64, 16, 16, C.byref(peer), 16, 64, None) == -1
    assert lib.slcl_peer_allgather(16, 40, 16, 16, C.byref(peer), 16, 64, None) == -1       # n_bytes % 16
    assert lib.slcl_peer_allgather(16, 128, 16, 16, C.byref(peer), 16, 64, None) == -3      # record larger than the slot
    bad = _lib.PeerT(16, 2, 2, 64, 1.0)
    assert lib.slcl_peer_allgather(16, 64, 16, 16, C.byref(bad), 16, 64, None) == -1        # rank out of range


def test_state_layout_and_assemble_arguments(lib):
    off = (C.c_int64 * 7)()
    assert lib.slcl_p2p_state_layout(4096, 256, off) == 0
    assert list(off)[6] == lib.slcl_p2p_state_bytes(4096, 256)
    assert list(off)[0] == 0 and all(o % 256 == 0 for o in list(off)[:6])
    assert lib.slcl_p2p_state_layout(4096, 100, off) == -1
    assert lib.slcl_p2p_state_assemble(None, 64, 64, 4, 16, 16, 16, 16, 2, None) == -1
    assert lib.slcl_p2p_state_assemble(16, 64, 64, 9, 16, 16, 16, 16, 2, None) == -1       # n_class <= 8


def test_global_record_bytes_covers_both_records():
    from slcl.p2p import global_record_bytes
    # cfg3 per rank: 16384 contrast rows + 4096 anchors, 256 channels (bf16 rows, {label, id}, 1/|x|)
    assert global_record_bytes(4096, 16384, 256) == 32 + (16384 + 4096) * (512 + 8 + 4)
    # tiny row sets: the second record (per-anchor constants and an 8 x (d + 1) table) is the larger one
    small = global_record_bytes(16, 16, 32, same_rows=True)
    assert small >= 32 + 3 * 64 + 8 * 65 * 4


def test_pack_puts_every_part_on_a_16_byte_boundary():
    import torch
    from slcl.p2p import _pack
    rec, lay = _pack([torch.zeros(4, dtype=torch.int32), torch.ones(3, dtype=torch.int32), torch.ones(5, 2, dtype=torch.int32)])
    assert rec.dtype == torch.uint8 and rec.numel() % 16 == 0
    assert [o for o, *_ in lay] == [0, 16, 32] and rec.numel() == 32 + 48
