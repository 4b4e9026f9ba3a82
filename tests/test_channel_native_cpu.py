"""CPU tests of the channel-sparse native step's host side: the `smt_column_ref` layout, the argument checks of
`smt_compact_adam_columns` (they run before anything touches device memory), the column-table builder's checks, and the
arena layout a channel owner asks for."""
import ctypes

import pytest
import torch


def test_column_ref_struct_layout():
    from sparse_matrix_tuning_b200._lib import ColumnRef
    assert ctypes.sizeof(ColumnRef) == 32
    assert (ColumnRef.ldw.offset, ColumnRef.off.offset, ColumnRef.col.offset, ColumnRef.n_out.offset) == (8, 16, 24, 28)


def test_compact_adam_columns_rejects_bad_arguments_without_a_gpu(built_library):
    lib = built_library
    buf = ctypes.create_string_buffer(256)
    p = (ctypes.cast(buf, ctypes.c_void_p).value + 15) // 16 * 16           # 16-byte aligned host address
    hp = (1e-3, .9, .95, 1e-8, 0., .1, .05, 1.)

    def call(master=p, grad=p, gdt=1, n=16, sq=None, n_sq=0, comp=None, cdt=1, cols=p, n_cols=2, wdt=1, bc1=.1):
        lr, b1, b2, eps, wd, _bc1, bc2, gs = hp
        return lib.smt_compact_adam_columns(master, p, p, grad, gdt, n, lr, b1, b2, eps, wd, bc1, bc2, gs, sq, n_sq,
                                            0., comp, cdt, cols, n_cols, wdt, None)

    def rejects(needle, **kw):
        assert call(**kw) == -1
        assert needle in lib.smt_last_error(), lib.smt_last_error()

    rejects(b"null pointer", master=None)
    rejects(b"bad grad dtype 7", gdt=7)
    rejects(b"multiple of 8", n=12)
    rejects(b"16-byte aligned", grad=p + 2)
    rejects(b"16-byte aligned", comp=p + 4)
    rejects(b"bias corrections", bc1=0.)
    rejects(b"n_sqnorm", sq=p, n_sq=0)
    rejects(b"bad compact dtype", comp=p, cdt=5)
    rejects(b"null column table", cols=None)
    rejects(b"bad W dtype", wdt=3)
    rejects(b"negative size", n_cols=-1)
    rejects(b"negative size", n=-8)
    # nothing to do is a no-op that needs no device, even with NULL pointers
    assert call(master=None, grad=None, cols=None, n_cols=0) == 0
    assert call(master=None, grad=None, cols=None, n=0) == 0


def test_column_table_builder_checks_its_entries():
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200._lib import SMTLibraryError
    w = torch.zeros(64, 32, dtype=torch.bfloat16)
    with pytest.raises(SMTLibraryError, match="column 32 outside"):
        ops.make_column_table([(w, 32, 0)], "cpu")
    with pytest.raises(SMTLibraryError, match="multiples of 8"):
        ops.make_column_table([(w, 3, 4)], "cpu")
    with pytest.raises(SMTLibraryError, match="multiples of 8"):
        ops.make_column_table([(torch.zeros(60, 32, dtype=torch.bfloat16), 3, 0)], "cpu")
    with pytest.raises(SMTLibraryError, match="unit column stride"):
        ops.make_column_table([(w.t(), 3, 0)], "cpu")
    t = ops.make_column_table([(w, 3, 0), (w, 31, 64)], "cpu")
    assert t.dtype == torch.uint8 and t.numel() == 64


@pytest.mark.parametrize("n,out_f,b,rows,cols", [(5, 512, 64, 1, 8), (64, 1024, 64, 1, 16), (77, 1024, 128, 1, 8),
                                                 (130, 4096, 128, 2, 32), (131, 768, 128, 2, 6), (70, 320, 64, 2, 5)])
def test_channel_tiles_and_arena_layout(n, out_f, b, rows, cols):
    """The arena reserves the ceil(n/b)*b rows the last row tile of the gradient launch stores, and two sum-of-squares
    slots per tile (the layer itself needs CUDA, so its methods run on a stand-in)."""
    from sparse_matrix_tuning_b200 import ops
    from sparse_matrix_tuning_b200.smt.smt import LinearLayer_ChannelSparsity as L

    class Stub:
        index_list = list(range(n))
        weight = torch.zeros(out_f, 8)
        _grad_tiles = L._grad_tiles

    assert ops.channel_grad_block(n, out_f) == b
    assert Stub()._grad_tiles() == (b, rows, cols)
    assert L._arena_layout(Stub()) == (rows * b * out_f, 2 * rows * cols)
