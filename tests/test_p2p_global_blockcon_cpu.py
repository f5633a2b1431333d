"""Host-side pieces of ``BlockConLoss(group=)`` (no GPU needed): the argument checks of the batched state assembly, the
record size of a block-diagonal problem, and the tile-major order the gathered records land in."""
import ctypes as C
import inspect

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from slcl import _lib
    try:
        return _lib.load()
    except _lib.SlclError:
        pytest.skip("libslcl.so not built")


def test_state_assemble_batched_arguments(lib):
    f = lib.slcl_p2p_state_assemble_batched
    # (state, n_anchor, dim_padded, n_class, n_batch, alpha, beta, colshift, absum_parts, n_parts, stream)
    assert f(None, 512, 64, 4, 4, 16, 16, 16, 16, 2, None) == -1                 # no state buffer
    assert f(16, 512, 64, 4, 4, None, 16, 16, 16, 2, None) == -1                 # no alpha
    assert f(16, 512, 64, 4, 4, 16, None, 16, 16, 2, None) == -1                 # no beta
    assert f(16, 512, 64, 4, 4, 16, 16, None, 16, 2, None) == -1                 # no colshift
    assert f(16, 512, 64, 4, 4, 16, 16, 16, None, 2, None) == -1                 # no ABsum parts
    assert f(16, 512, 64, 4, 0, 16, 16, 16, 16, 2, None) == -1                   # n_batch < 1
    assert f(16, 512, 64, 4, -3, 16, 16, 16, 16, 2, None) == -1
    assert f(16, 512, 64, 9, 4, 16, 16, 16, 16, 2, None) == -1                   # n_class <= 8
    assert f(16, 512, 64, 0, 4, 16, 16, 16, 16, 2, None) == -1                   # n_class >= 1
    assert f(16, 512, 64, 4, 4, 16, 16, 16, 16, 0, None) == -1                   # n_parts >= 1
    assert f(16, 512, 64, 4, 3, 16, 16, 16, 16, 2, None) == -1                   # batches of equal size
    assert f(16, 512, 64, 4, 8, 16, 16, 16, 16, 2, None) == -1                   # 64-row batches: not whole 128-row tiles
    assert f(16, 512, 100, 4, 4, 16, 16, 16, 16, 2, None) == -1                  # dim_padded a multiple of 64
    assert f(24, 512, 64, 4, 4, 16, 16, 16, 16, 2, None) == -1                   # state 16-byte aligned
    # the unbatched entry point is the n_batch = 1 case and keeps its own checks
    assert lib.slcl_p2p_state_assemble(None, 64, 64, 4, 16, 16, 16, 16, 2, None) == -1


def test_global_record_bytes_with_block_diagonal_batches():
    from slcl.p2p import AUTO_N_CLASS, global_record_bytes
    assert global_record_bytes(4096, 16384, 256, n_batch=1) == global_record_bytes(4096, 16384, 256)
    assert global_record_bytes(16, 16, 32, True, n_batch=1) == global_record_bytes(16, 16, 32, same_rows=True)
    # the reference's per-rank shape (1, 2, 32, 224, 224), block 32: 49 tiles of 2048 rows; the row record dominates
    m, dp = 1 * 2 * 49 * 32 * 32, 64
    assert global_record_bytes(m, m, 32, same_rows=True, n_batch=49) == 32 + m * (2 * dp + 8 + 4)
    # few rows, many tiles: the second record -- one [K][d + 1] ABsum table per tile -- is the larger one
    for n_batch in (1, 4, 49):
        got = global_record_bytes(16, 16, 32, same_rows=True, n_batch=n_batch)
        assert got == 32 + 3 * 64 + n_batch * AUTO_N_CLASS * (dp + 1) * 4


def _record(rank, n_tiles, rows, d):
    """One rank's record: key, bf16 rows [T R, d], {label, id} [T R, 2], norms [T R], an ABsum-like table [T, 5]."""
    from slcl.p2p import _pack
    n = n_tiles * rows
    base = torch.arange(n, dtype=torch.float32) + 1000 * rank
    parts = [torch.full((4,), 7, dtype=torch.int32),
             (base.view(-1, 1) + torch.arange(d, dtype=torch.float32) / 64).to(torch.bfloat16),
             torch.stack([base.int() % 5, base.int()], 1),
             base * 0.5,
             torch.arange(n_tiles * 5, dtype=torch.float32).view(n_tiles, 5) + 100 * rank]
    return _pack(parts)


def test_unpack_lands_rows_tile_major():
    """W = 3 ranks, T = 4 tiles of R = 6 rows: row part -> [tile][rank][row of the tile]; the table stays rank-major."""
    from slcl.p2p import _unpack
    W, T, R, d = 3, 4, 6, 64
    recs = [_record(q, T, R, d) for q in range(W)]
    lay = recs[0][1]
    gathered = torch.stack([rec for rec, _ in recs])
    per_rank = lambda i: [_unpack(rec.view(1, -1), lay, i) for rec, _ in recs]          # each rank's part on its own
    for i in (1, 2, 3):
        mine = per_rank(i)
        want = torch.cat([mine[q][t * R:(t + 1) * R] for t in range(T) for q in range(W)])      # explicit permutation
        got = _unpack(gathered, lay, i, T)
        assert got.dtype == mine[0].dtype and got.shape == (W * T * R,) + tuple(mine[0].shape[1:])
        assert torch.equal(got, want)
        # global row g = t W R + q R + k  <->  rank q's local row t R + k
        perm = torch.tensor([q * T * R + t * R + k for t in range(T) for q in range(W) for k in range(R)])
        assert torch.equal(got, torch.cat(mine)[perm])
        assert torch.equal(_unpack(gathered, lay, i), torch.cat(mine))                  # n_batch = 1: rank order
    assert torch.equal(_unpack(gathered, lay, 4), torch.cat(per_rank(4)))              # rank-major table


def test_global_self_maps_in_tile_major_order():
    """The self maps of rank r in the global [tile][rank][row] index spaces, against their definitions."""
    from slcl.p2p import _global_self_maps
    W, T, R = 3, 4, 5
    n = T * R
    ident = torch.arange(n, dtype=torch.int32)
    sparse = torch.where(ident % 3 == 0, (ident + 7) % n, torch.full_like(ident, -1)).to(torch.int32)   # a partial map
    inv = torch.full((n,), -1, dtype=torch.int32)
    inv[sparse[sparse >= 0].long()] = ident[sparse >= 0]
    for selfcol, selfrow in ((ident, ident), (sparse, inv)):
        for r in range(W):
            col_f, row_g, col_g, row_l = _global_self_maps(selfcol, selfrow, n, n, W, r, T)
            glob = lambda i: -1 if i < 0 else (i // R) * W * R + r * R + i % R
            assert col_f.tolist() == [glob(int(j)) for j in selfcol]                   # local anchor -> global column
            assert row_l.tolist() == [glob(int(i)) for i in selfrow]                   # local column -> global anchor
            want_row_g, want_col_g = [], []
            for t in range(T):
                for q in range(W):
                    for k in range(R):
                        want_row_g.append(int(selfrow[t * R + k]) if q == r else -1)
                        want_col_g.append(int(selfcol[t * R + k]) if q == r else -1)
            assert row_g.tolist() == want_row_g and col_g.tolist() == want_col_g
            assert all(t.dtype == torch.int32 for t in (col_f, row_g, col_g, row_l))
    # one tile: the rank-major offsets of the unbatched global losses
    col_f, row_g, col_g, row_l = _global_self_maps(ident, ident, n, n, W, 2, 1)
    assert torch.equal(col_f, ident + 2 * n) and torch.equal(row_l, ident + 2 * n)
    assert torch.equal(row_g[2 * n:], ident) and bool((row_g[:2 * n] == -1).all())


def test_blockcon_signature_takes_group():
    from slcl import loss
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(loss.BlockConLoss.__init__) == ["self", "temperature", "block_size", "n_class", "group"]
    assert sig(loss.BlockConLoss.forward) == ["self", "features", "labels", "group"]
    m = loss.BlockConLoss()
    assert m.supconloss.group is None and m.block_size == 32 and m.supconloss.temperature == 0.7
