"""CPU tests of the C ABI of the scoring, top-k, block / column movement and compact-Adam entry points: every bad
argument is rejected with SMT_ERR_ARG (SMT_ERR_WORKSPACE for a workspace) and a message that names the entry point and
the argument, before any device work; zero-size calls behave as each entry point documents.

The pointers are host addresses that are never dereferenced: every call below is either rejected by the argument
checks or has nothing to do, so it returns before a kernel is launched, with or without a GPU."""
import ctypes as C

import pytest

OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -4
F32, BF16, F16 = 0, 1, 2
MEAN_ABS, L2 = 0, 3

_HOST_BUF = C.create_string_buffer(1 << 12)
P = (C.cast(_HOST_BUF, C.c_void_p).value + 15) & ~15          # a 16-byte aligned host address (only its value is used)


@pytest.fixture(scope="module")
def lib(built_library):
    return built_library


def _rejects(lib, name, args, *words, code=ERR_ARG):
    rc = getattr(lib, name)(*args)
    assert rc == code, (name, args, rc)
    msg = lib.smt_last_error().decode()
    assert msg.startswith(name), (name, msg)
    for w in words:
        assert w in msg, (name, args, w, msg)


def _variants(lib, name, good, cases, code=ERR_ARG):
    """`good` is a well-formed argument list by name; each case overrides some of it and names the words the message
    must contain."""
    keys = list(good)
    for over, words in cases:
        a = dict(good)
        a.update(over)
        _rejects(lib, name, [a[k] for k in keys] + [None], *words, code=code)


def test_score_accumulate(lib):
    good = dict(acc=P, grad=P, dtype=BF16, n=8)
    _variants(lib, "smt_score_accumulate", good, [
        ({"n": -1}, ["n < 0"]), ({"n": -(1 << 40)}, ["n < 0"]),
        ({"dtype": 3}, ["bad dtype 3"]), ({"dtype": -1}, ["bad dtype -1"]), ({"dtype": 3, "n": 0}, ["bad dtype 3"]),
        ({"acc": None}, ["null pointer", "(acc)"]), ({"grad": None}, ["null pointer", "(grad)"]),
        ({"acc": None, "grad": None}, ["(acc)"]),
    ])
    # n = 0 is a no-op that needs no data pointer: an empty CUDA tensor has data_ptr() == 0
    for dtype in (F32, BF16, F16):
        assert lib.smt_score_accumulate(None, None, dtype, 0, None) == OK
        assert lib.smt_score_accumulate(P, None, dtype, 0, None) == OK


def test_grad_sqnorm(lib):
    ws = lib.smt_grad_sqnorm_workspace_bytes()
    assert ws == 4096
    good = dict(grad=P, dtype=BF16, n=8, out=P, ws=P, ws_bytes=ws)
    _variants(lib, "smt_grad_sqnorm", good, [
        ({"dtype": 3}, ["bad dtype 3"]), ({"n": -1}, ["n < 0"]),
        ({"grad": None}, ["null pointer", "(grad)"]), ({"out": None}, ["null pointer", "(out_sqnorm)"]),
        ({"grad": P + 8}, ["grad must be 16-byte aligned"]), ({"grad": P + 2}, ["grad must be 16-byte aligned"]),
        # n = 0: the gradient pointer may be NULL, but out_sqnorm is still written (the Adam clip reads it)
        ({"grad": None, "n": 0, "out": None}, ["(out_sqnorm)"]),
    ])
    _variants(lib, "smt_grad_sqnorm", good, [
        ({"ws": None}, ["workspace"]), ({"ws_bytes": ws - 1}, ["workspace"]), ({"ws_bytes": 0}, ["workspace"]),
        ({"grad": None, "n": 0, "ws": None}, ["workspace"]),          # past the pointer checks: n = 0 needs no grad
    ], code=ERR_WORKSPACE)


def test_block_sum_accumulate_and_finalize(lib):
    good = dict(sums=P, grad=P, dtype=BF16, rows=512, cols=768, ld=768, block=256)
    _variants(lib, "smt_block_sum_accumulate", good, [
        ({"dtype": 3}, ["bad dtype 3"]),
        ({"grad": None}, ["null pointer", "(grad)"]), ({"sums": None}, ["null block_sums"]),
        ({"block": 100}, ["block size 100"]), ({"block": 32}, ["block size 32"]),
        ({"rows": 500}, ["matrix 500x768", "block 256"]), ({"cols": 700}, ["matrix 512x700"]),
        ({"rows": 512, "block": 512}, ["block size 512"]),
        ({"ld": 512}, ["ld 512 < cols 768"]),
        ({"grad": P + 2}, ["16-byte aligned"]), ({"ld": 772}, ["16-byte aligned"]),
        ({"dtype": F32, "ld": 770}, ["16-byte aligned"]),
        ({"rows": 64 * 65536, "cols": 64, "ld": 64, "block": 64}, ["too many block rows"]),
        # empty input is rejected by design: a score needs at least one block
        ({"rows": 0}, ["matrix 0x768"]), ({"cols": 0}, ["matrix 512x0"]), ({"rows": -256}, ["matrix -256x768"]),
    ])
    good = dict(sums=P, scores=P, n=6, block=256)
    _variants(lib, "smt_block_sum_finalize", good, [
        ({"sums": None}, ["null pointer", "(block_sums)"]), ({"scores": None}, ["null pointer", "(scores)"]),
        ({"block": 100}, ["bad block 100"]),
    ])
    assert lib.smt_block_sum_finalize(P, P, 0, 256, None) == OK
    assert lib.smt_block_sum_finalize(P, P, -3, 64, None) == OK


def test_block_score_reduce(lib):
    good = dict(acc=P, rows=512, cols=768, ld=768, block=256, strategy=MEAN_ABS, scores=P)
    _variants(lib, "smt_block_score_reduce", good, [
        ({"acc": None}, ["null pointer", "(acc)"]), ({"scores": None}, ["null scores"]),
        ({"strategy": 4}, ["unknown strategy 4"]), ({"strategy": -1}, ["unknown strategy -1"]),
        ({"block": 100}, ["block size 100"]), ({"rows": 320}, ["matrix 320x768"]), ({"ld": 700}, ["ld 700 < cols"]),
        ({"ld": 770}, ["16-byte aligned"]), ({"acc": P + 4}, ["16-byte aligned"]),
        ({"rows": 0}, ["matrix 0x768"]), ({"cols": 0}, ["matrix 512x0"]),
    ])


def test_activation_scoring(lib):
    good = dict(acc=P, x=P, dtype=BF16, batch=2, seq=7, channels=64)
    _variants(lib, "smt_act_score_accumulate", good, [
        ({"acc": None}, ["null pointer", "(acc)"]), ({"x": None}, ["null pointer", "(x)"]),
        ({"dtype": 3}, ["bad dtype 3"]),
        ({"channels": 12}, ["channels must be a multiple of 8"]), ({"acc": P + 4}, ["16-byte aligned"]),
        ({"x": P + 8}, ["16-byte aligned"]),
        # empty input is rejected by design (the activation hook always sees tokens)
        ({"batch": 0}, ["empty input"]), ({"seq": 0}, ["empty input"]), ({"channels": 0}, ["empty input"]),
        ({"batch": -1}, ["empty input"]),
    ])
    good = dict(acc=P, seq=7, channels=12, strategy=L2, out=P)
    _variants(lib, "smt_channel_score_reduce", good, [
        ({"acc": None}, ["null pointer", "(acc)"]), ({"out": None}, ["null pointer", "(out)"]),
        ({"channels": 6}, ["channels must be a positive multiple of 4"]),
        ({"channels": 0}, ["channels must be a positive multiple of 4"]), ({"seq": 0}, ["positive multiple of 4"]),
        ({"acc": P + 4}, ["16-byte aligned"]), ({"out": P + 8}, ["16-byte aligned"]),
        ({"strategy": 4}, ["unknown strategy 4"]),
    ])


def test_topk_blocks(lib):
    ws = lib.smt_topk_workspace_bytes(100)
    assert ws == (2 * 100 + 2) * 8 and lib.smt_topk_workspace_bytes(-5) == 16
    good = dict(scores=P, rank=None, inv=None, n=100, seg_off=P, seg_k=P, out_off=P, nseg=3, out=P, ws=P, ws_bytes=ws)
    _variants(lib, "smt_topk_blocks", good, [
        ({"nseg": -1}, ["num_segments < 0"]),
        ({"scores": None}, ["null pointer", "(scores)"]), ({"seg_off": None}, ["null pointer", "(seg_offsets)"]),
        ({"seg_k": None}, ["null pointer", "(seg_k)"]), ({"out_off": None}, ["null pointer", "(out_offsets)"]),
        ({"out": None}, ["null pointer", "(out_idx)"]),
        ({"rank": P}, ["tiebreak_rank and inv_rank"]), ({"inv": P}, ["tiebreak_rank and inv_rank"]),
        ({"n": 1 << 31, "ws_bytes": 1 << 40}, ["too many scores"]),
    ])
    _variants(lib, "smt_topk_blocks", good, [
        ({"ws": None}, ["workspace too small"]), ({"ws_bytes": ws - 1}, ["workspace too small"]),
    ], code=ERR_WORKSPACE)
    # no segment or no score: nothing to do, no pointer needed
    assert lib.smt_topk_blocks(None, None, None, 0, None, None, None, 3, None, None, 0, None) == OK
    assert lib.smt_topk_blocks(None, None, None, 100, None, None, None, 0, None, None, 0, None) == OK


@pytest.mark.parametrize("name", ["smt_block_gather", "smt_block_scatter"])
def test_block_copies(lib, name):
    good = dict(table=P, n=4, block=128, elem=2, compact=P)
    _variants(lib, name, good, [
        ({"n": -1}, ["n_blocks < 0"]),
        ({"table": None}, ["null pointer", "(table)"]), ({"compact": None}, ["null pointer", "(compact)"]),
        ({"block": 100}, ["block size 100"]), ({"elem": 3}, ["elem_bytes must be 2 or 4"]),
        ({"elem": 8}, ["elem_bytes"]), ({"compact": P + 8}, ["compact must be 16-byte aligned"]),
    ])
    assert getattr(lib, name)(None, 0, 256, 2, None, None) == OK
    assert getattr(lib, name)(None, 0, 100, 3, None, None) == OK


@pytest.mark.parametrize("name", ["smt_column_gather", "smt_column_scatter"])
def test_column_copies(lib, name):
    good = dict(W=P, ldw=100, out_f=40, in_f=90, idx=P, n=33, elem=2, compact=P)
    _variants(lib, name, good, [
        ({"n": -1}, ["negative size"]), ({"out_f": -8}, ["negative size"]),
        ({"W": None}, ["null pointer", "(W)"]), ({"idx": None}, ["null pointer", "(idx)"]),
        ({"compact": None}, ["null pointer", "(compact)"]),
        ({"elem": 3}, ["elem_bytes must be 2 or 4"]), ({"ldw": 89}, ["bad leading dimension"]),
        ({"in_f": 0, "ldw": 0}, ["bad leading dimension"]),
        ({"n": 32 * 65535 + 1}, ["too many channels"]),
    ])
    for n, out_f in ((0, 40), (33, 0), (0, 0)):
        assert getattr(lib, name)(None, 0, out_f, 0, None, n, 3, None, None) == OK


def test_channel_gather(lib):
    good = dict(x=P, T=1000, ldx=90, idx=P, n=33, elem=4, out=P)
    _variants(lib, "smt_channel_gather", good, [
        ({"T": -1}, ["negative size"]), ({"n": -1}, ["negative size"]),
        ({"x": None}, ["null pointer", "(x)"]), ({"idx": None}, ["null pointer", "(idx)"]),
        ({"out": None}, ["null pointer", "(out)"]),
        ({"elem": 1}, ["elem_bytes must be 2 or 4"]), ({"ldx": 0}, ["bad leading dimension"]),
        ({"ldx": -5}, ["bad leading dimension"]),
    ])
    for T, n in ((0, 33), (1000, 0), (0, 0)):
        assert lib.smt_channel_gather(None, T, 0, None, n, 3, None, None) == OK


HP = (1e-3, .9, .95, 1e-8, 0.01, .1, .05, 1.)                   # lr, beta1, beta2, eps, wd, bc1, bc2, grad_scale


def _adam_args(**kw):
    a = dict(master=P, m=P, v=P, grad=P, gdt=BF16, n=64 * 64 * 2, lr=HP[0], b1=HP[1], b2=HP[2], eps=HP[3], wd=HP[4],
             bc1=HP[5], bc2=HP[6], gs=HP[7], sq=None, n_sq=0, max_norm=0., comp=None, cdt=BF16)
    a.update(kw)
    return a


def test_compact_adam(lib):
    good = _adam_args()
    good.update(table=P, n_blocks=2, block=64, wdt=BF16)
    _variants(lib, "smt_compact_adam", good, [
        ({"n": -8}, ["n_elems < 0"]),
        ({"master": None}, ["null pointer", "(master)"]), ({"m": None}, ["null pointer", "(exp_avg)"]),
        ({"v": None}, ["null pointer", "(exp_avg_sq)"]), ({"grad": None}, ["null pointer", "(grad)"]),
        ({"gdt": 3}, ["bad grad dtype 3"]), ({"n": 12}, ["n_elems must be a multiple of 8"]),
        ({"grad": P + 2}, ["16-byte aligned"]), ({"master": P + 4}, ["16-byte aligned"]),
        ({"m": P + 8}, ["16-byte aligned"]), ({"v": P + 12}, ["16-byte aligned"]),
        ({"comp": P + 8}, ["16-byte aligned"]),
        ({"bc1": 0.}, ["bias corrections must be > 0"]), ({"bc2": -1.}, ["bias corrections must be > 0"]),
        ({"sq": P, "n_sq": 0}, ["n_sqnorm must be >= 1"]),
        ({"comp": P, "cdt": 5}, ["bad compact dtype 5"]),
        ({"block": 100}, ["block size 100"]), ({"n_blocks": 3}, ["n_blocks*b*b != n_elems"]),
        ({"block": 128}, ["n_blocks*b*b != n_elems"]), ({"wdt": 3}, ["bad W dtype 3"]),
    ])
    # n_elems = 0 is a no-op that needs no pointer (an empty parameter group)
    args = [None, None, None, None, BF16, 0, *HP, None, 0, 0., None, BF16, None, 0, 0, BF16, None]
    assert lib.smt_compact_adam(*args) == OK


def test_compact_adam_columns_sizes_and_names(lib):
    good = _adam_args(n=16)
    good.update(cols=P, n_cols=2, wdt=BF16)
    _variants(lib, "smt_compact_adam_columns", good, [
        ({"n": -8}, ["negative size"]), ({"n_cols": -1}, ["negative size"]),
        ({"m": None}, ["null pointer", "(exp_avg)"]), ({"v": None}, ["null pointer", "(exp_avg_sq)"]),
        ({"grad": None}, ["null pointer", "(grad)"]), ({"master": None}, ["null pointer", "(master)"]),
    ])
    for n, n_cols in ((0, 2), (16, 0), (0, 0)):
        args = [None, None, None, None, BF16, n, *HP, None, 0, 0., None, BF16, None, n_cols, BF16, None]
        assert lib.smt_compact_adam_columns(*args) == OK
