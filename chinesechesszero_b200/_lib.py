"""ctypes binding of the C ABI in include/ccz_b200.h (libccz_b200.so, built by build.py).

The library is the only compute path: loading fails loudly when the .so is missing and every
wrapper raises on a non-zero status.  Tensors own all device memory; wrappers pass raw
``data_ptr()`` values and the current torch CUDA stream.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np
import torch

from . import build as _build

BOARD_BYTES = 96
MAX_MOVES = 128
N_ACTIONS = 2086
PLANE_ELEMS = 10710
KEY_WINDOW = 128

FLAG_CHECK, FLAG_NOMOVES, FLAG_INSUFFICIENT, FLAG_FOURFOLD, FLAG_SIXTY = 1, 2, 4, 8, 16
FLAG_TIE_MASK = FLAG_INSUFFICIENT | FLAG_FOURFOLD | FLAG_SIXTY
STATUS_EXPAND_FAILED, STATUS_TREE_DROPPED = 1, 2
STATUS_NODE_OVERFLOW = STATUS_EXPAND_FAILED
ADVANCE_NEW_GAME, ADVANCE_DROP_TREE, ADVANCE_KEEP = -1, -2, -3
CTL_HEAD, CTL_TAIL, CTL_EXPAND_FAILED, CTL_TREES_DROPPED, CTL_MIN_FREE, CTL_WORDS = 0, 1, 2, 3, 4, 8
NODE_BYTES = 24  # ccz_node (16) + ccz_link (8)
MAX_CHILDREN = 119  # most legal moves of any Xiangqi position
POLICY_PROBS, POLICY_LOGITS = 0, 1
DEDUP_MAX_BOARDS = 16384  # largest leaf batch ccz_leaf_unique takes
CONV_VARIANT_1CTA, CONV_VARIANT_PAIR, CONV_VARIANT_2PAIRS, CONV_VARIANT_4PAIRS = 1, 2, 2 | 32, 2 | 64

EXPORTS = (
    "ccz_version", "ccz_last_error", "ccz_init", "ccz_action_table", "ccz_set_order_policy", "ccz_get_order_policy",
    "ccz_boards_start",
    "ccz_movegen_encode", "ccz_board_keys_init", "ccz_board_push", "ccz_mcts_pool_init", "ccz_mcts_reset",
    "ccz_mcts_reserve", "ccz_mcts_migrate", "ccz_mcts_select",
    "ccz_mcts_expand_backup", "ccz_mcts_root_visits", "ccz_mcts_advance", "ccz_replay_pack", "ccz_conv3x3_c256", "ccz_conv3x3_plan", "ccz_stem_lookup",
    "ccz_heads_pack", "ccz_conv3x3_c256_count", "ccz_stem_lookup_count", "ccz_heads_pack_rows", "ccz_leaf_unique",
)


class CczError(RuntimeError):
    pass


class ArenaStruct(ctypes.Structure):
    """Mirror of ``ccz_arena`` (include/ccz_b200.h)."""

    _fields_ = [
        ("n_games", ctypes.c_int32),
        ("n_pages", ctypes.c_int32),
        ("page_shift", ctypes.c_int32),
        ("max_pages", ctypes.c_int32),
        ("d_nodes", ctypes.c_void_p),
        ("d_links", ctypes.c_void_p),
        ("d_free_ring", ctypes.c_void_p),
        ("d_pool_ctl", ctypes.c_void_p),
        ("d_page_list", ctypes.c_void_p),
        ("d_page_fill", ctypes.c_void_p),
        ("d_n_pages", ctypes.c_void_p),
        ("d_n_pages_new", ctypes.c_void_p),
        ("d_list_sel", ctypes.c_void_p),
        ("d_alloc_page", ctypes.c_void_p),
        ("d_alloc_off", ctypes.c_void_p),
        ("d_root", ctypes.c_void_p),
        ("d_n_nodes", ctypes.c_void_p),
        ("d_status", ctypes.c_void_p),
        ("d_root_boards", ctypes.c_void_p),
        ("d_root_keys", ctypes.c_void_p),
    ]


_lib = None


def library_path() -> str:
    # CCZ_LIB points at an alternative build of the same library (debug / bisect builds)
    return os.environ.get("CCZ_LIB") or _build.OUT


def load() -> ctypes.CDLL:
    """Load libccz_b200.so (no fallback: a missing library is an error)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if path == _build.OUT and _build.is_stale():
        try:  # same image on the GPU box: nvcc is there, so a missing / outdated library is rebuilt in-tree
            _build.build()
        except Exception as e:  # noqa: BLE001 - reported below if the library is still missing
            if not os.path.exists(path):
                raise CczError(f"building {path} failed ({e}); there is no CPU fallback") from e
    if not os.path.exists(path):
        raise CczError(
            f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a); there is no CPU fallback"
        )
    lib = ctypes.CDLL(path)
    vp, i32, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    lib.ccz_version.restype = i32
    lib.ccz_last_error.restype = ctypes.c_char_p
    lib.ccz_init.restype = i32
    lib.ccz_action_table.argtypes = [vp, vp, vp]
    lib.ccz_boards_start.argtypes = [vp, i32, vp]
    lib.ccz_set_order_policy.argtypes = [vp]
    lib.ccz_get_order_policy.argtypes = [vp]
    lib.ccz_movegen_encode.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.ccz_board_keys_init.argtypes = [vp, i32, vp, vp]
    lib.ccz_board_push.argtypes = [vp, vp, i32, vp, vp]
    lib.ccz_mcts_pool_init.argtypes = [ctypes.POINTER(ArenaStruct), vp]
    lib.ccz_mcts_reset.argtypes = [ctypes.POINTER(ArenaStruct), vp, vp]
    lib.ccz_mcts_reserve.argtypes = [ctypes.POINTER(ArenaStruct), i32, vp]
    lib.ccz_mcts_migrate.argtypes = [ctypes.POINTER(ArenaStruct), ctypes.POINTER(ArenaStruct), vp]
    lib.ccz_mcts_select.argtypes = [ctypes.POINTER(ArenaStruct), f32, vp, vp, vp]
    lib.ccz_mcts_expand_backup.argtypes = [ctypes.POINTER(ArenaStruct), vp, vp, i32, vp, vp, vp, vp, vp]
    lib.ccz_mcts_root_visits.argtypes = [ctypes.POINTER(ArenaStruct), vp, vp, vp, vp]
    lib.ccz_mcts_advance.argtypes = [ctypes.POINTER(ArenaStruct), vp, vp]
    lib.ccz_replay_pack.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.ccz_conv3x3_c256.argtypes = [vp, vp, vp, vp, vp, i32, i32, vp]
    lib.ccz_stem_lookup.argtypes = [vp, i32, vp, vp, vp, vp]
    lib.ccz_conv3x3_plan.argtypes = [i32, i32, i32, vp]
    lib.ccz_heads_pack.argtypes = [vp, i32, vp, i32, i32, vp]
    lib.ccz_conv3x3_c256_count.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32, vp]
    lib.ccz_stem_lookup_count.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.ccz_heads_pack_rows.argtypes = [vp, i32, vp, vp, i32, i32, vp]
    lib.ccz_leaf_unique.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    for name in EXPORTS:
        if name not in ("ccz_last_error",):
            getattr(lib, name).restype = i32
    _lib = lib
    # generation order pinned against a real cchess (scripts/pin_cchess.py writes this file next to the library)
    pinned = os.path.join(os.path.dirname(os.path.abspath(__file__)), "order_policy.json")
    if os.path.exists(pinned):
        import json

        with open(pinned) as f:
            set_order_policy(json.load(f))
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ccz_last_error().decode("utf-8", "replace")
        raise CczError(f"{what} failed ({rc}): {msg}")


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: torch.Tensor | None) -> int | None:
    if t is None:
        return None
    if not t.is_cuda:
        raise CczError("device tensor expected (the C ABI takes device pointers)")
    if not t.is_contiguous():
        raise CczError("contiguous tensor expected")
    return t.data_ptr()


def host_action_table():
    """(id_of[90,90] int16, from_of[2086] uint8, to_of[2086] uint8) from the library (host side)."""
    id_of = np.empty(8100, dtype=np.int16)
    fr = np.empty(N_ACTIONS, dtype=np.uint8)
    to = np.empty(N_ACTIONS, dtype=np.uint8)
    n = load().ccz_action_table(id_of.ctypes.data, fr.ctypes.data, to.ctypes.data)
    if n != N_ACTIONS:
        raise CczError(f"ccz_action_table returned {n}")
    return id_of.reshape(90, 90), fr, to


PIECE_SYMBOLS = (None, "p", "c", "r", "n", "b", "a", "k")  # piece type 1..7 (ccz_rules.cuh)
DEFAULT_ORDER_POLICY = {"class_rank": {"p": 1, "c": 0, "r": 0, "n": 0, "b": 0, "a": 0, "k": 0},
                        "from_descending": 1, "to_descending": 1, "capture_mode": 0, "check_king_first": 0}


def set_order_policy(policy: dict | None = None) -> None:
    """Generation order of the legal moves K1 emits (``ccz_order_policy``; None = the default).  A dict as
    ``DEFAULT_ORDER_POLICY`` -- what ``scripts/pin_cchess.py`` stores under "order_policy" in
    tests/golden/cchess_pin.json.  Library-wide host state: set it before any search starts."""
    if policy is None:
        check(load().ccz_set_order_policy(None), "ccz_set_order_policy")
        return
    ranks = [0] * 8
    for sym, r in policy["class_rank"].items():
        ranks[PIECE_SYMBOLS.index(sym)] = int(r)
    raw = bytes(ranks + [int(policy["from_descending"]), int(policy["to_descending"]), int(policy["capture_mode"]),
                        int(policy.get("check_king_first", 0))])
    check(load().ccz_set_order_policy(ctypes.create_string_buffer(raw, 12)), "ccz_set_order_policy")


def get_order_policy() -> dict:
    buf = ctypes.create_string_buffer(12)
    check(load().ccz_get_order_policy(buf), "ccz_get_order_policy")
    b = buf.raw
    return {"class_rank": {PIECE_SYMBOLS[t]: b[t] for t in range(1, 8)}, "from_descending": b[8],
            "to_descending": b[9], "capture_mode": b[10], "check_king_first": b[11]}


# ---- tensor-level wrappers ------------------------------------------------------------------

def boards_start(n: int, device="cuda") -> torch.Tensor:
    boards = torch.empty((n, BOARD_BYTES), dtype=torch.uint8, device=device)
    with torch.cuda.device(boards.device):
        check(load().ccz_boards_start(_ptr(boards), n, stream_ptr(boards.device)), "ccz_boards_start")
    return boards


def movegen_encode(boards: torch.Tensor, planes: bool = True, out=None):
    """boards [n,96] uint8 (cuda) -> (move_ids [n,128] i16, counts [n] i16, flags [n] u8, planes [n,17,7,10,9] bf16|None).

    ``out`` may carry preallocated (move_ids, counts, flags, planes) tensors.
    """
    n = boards.shape[0]
    dev = boards.device
    _ptr(boards)  # device + contiguity check before anything is allocated
    if out is None:
        move_ids = torch.empty((n, MAX_MOVES), dtype=torch.int16, device=dev)
        counts = torch.empty((n,), dtype=torch.int16, device=dev)
        flags = torch.empty((n,), dtype=torch.uint8, device=dev)
        pl = torch.empty((n, 17, 7, 10, 9), dtype=torch.bfloat16, device=dev) if planes else None
    else:
        move_ids, counts, flags, pl = out
    with torch.cuda.device(dev):
        check(
            load().ccz_movegen_encode(_ptr(boards), n, _ptr(move_ids), _ptr(counts), _ptr(flags), _ptr(pl),
                                      stream_ptr(dev)),
            "ccz_movegen_encode",
        )
    return move_ids, counts, flags, pl


def board_keys_init(boards: torch.Tensor) -> torch.Tensor:
    n = boards.shape[0]
    keys = torch.empty((n, KEY_WINDOW), dtype=torch.int64, device=boards.device)
    with torch.cuda.device(boards.device):
        check(load().ccz_board_keys_init(_ptr(boards), n, _ptr(keys), stream_ptr(boards.device)),
              "ccz_board_keys_init")
    return keys


def board_push(boards: torch.Tensor, move_ids: torch.Tensor, keys: torch.Tensor | None = None) -> None:
    n = boards.shape[0]
    if move_ids.dtype != torch.int16 or move_ids.numel() != n:
        raise CczError("move_ids must be int16 [n]")
    with torch.cuda.device(boards.device):
        check(load().ccz_board_push(_ptr(boards), _ptr(move_ids), n, _ptr(keys), stream_ptr(boards.device)),
              "ccz_board_push")


def search_pages(n_playout: int, page_shift: int) -> int:
    """Upper bound of the pages one game can take during ``n_playout`` playouts: every playout expands
    at most one leaf into at most MAX_CHILDREN contiguous slots, a page holds at least
    ``2**page_shift // MAX_CHILDREN`` such runs, plus the partly used page the search starts in."""
    runs_per_page = max(1, (1 << page_shift) // MAX_CHILDREN)
    return -(-int(n_playout) // runs_per_page) + 1


class Arena:
    """Device arrays of one pooled MCTS arena (see ``ccz_arena`` in include/ccz_b200.h): ``n_pages``
    pages of ``2**page_shift`` nodes shared by ``n_games`` trees."""

    def __init__(self, n_games: int, n_pages: int, page_shift: int = 11, max_pages: int | None = None, device="cuda"):
        self.n_games, self.n_pages, self.page_shift = int(n_games), int(n_pages), int(page_shift)
        if not 7 <= self.page_shift <= 16:
            raise CczError("page_shift must be 7..16")
        if self.n_pages < self.n_games:
            raise CczError("the pool needs at least one page per game")
        if (self.n_pages << self.page_shift) >= 1 << 31:
            raise CczError("pool too large: n_pages << page_shift must stay below 2^31 nodes")
        self.max_pages = int(max_pages) if max_pages is not None else min(self.n_pages, 4096)
        self.device = torch.device(device)
        total = self.n_pages << self.page_shift
        g, z = self.n_games, dict(device=self.device)
        i32 = torch.int32
        self.nodes = torch.empty((total, 4), dtype=i32, **z)   # N, Q bits, P bits, first_child
        self.links = torch.empty((total, 2), dtype=i32, **z)   # parent, move | n_child << 16
        self.free_ring = torch.zeros(self.n_pages, dtype=i32, **z)
        self.pool_ctl = torch.zeros(CTL_WORDS, dtype=torch.int64, **z)
        self.page_lists = torch.zeros((2, g, self.max_pages), dtype=i32, **z)
        self.page_fill = torch.zeros((g, self.max_pages), dtype=i32, **z)
        self.n_pages_game = torch.zeros(g, dtype=i32, **z)
        self.n_pages_new = torch.zeros(g, dtype=i32, **z)
        self.list_sel = torch.zeros(g, dtype=i32, **z)
        self.alloc_page = torch.zeros(g, dtype=i32, **z)
        self.alloc_off = torch.zeros(g, dtype=i32, **z)
        self.root = torch.zeros(g, dtype=i32, **z)
        self.n_nodes = torch.zeros(g, dtype=i32, **z)
        self.status = torch.zeros(g, dtype=i32, **z)
        self.root_boards = torch.zeros((g, BOARD_BYTES), dtype=torch.uint8, **z)
        self.root_keys = torch.zeros((g, KEY_WINDOW), dtype=torch.int64, **z)
        self._tensors = (self.nodes, self.links, self.free_ring, self.pool_ctl, self.page_lists, self.page_fill,
                         self.n_pages_game, self.n_pages_new, self.list_sel, self.alloc_page, self.alloc_off, self.root,
                         self.n_nodes, self.status, self.root_boards, self.root_keys)
        self.struct = ArenaStruct(self.n_games, self.n_pages, self.page_shift, self.max_pages,
                                  *(t.data_ptr() for t in self._tensors))
        with torch.cuda.device(self.device):
            check(load().ccz_mcts_pool_init(self.ref, stream_ptr(self.device)), "ccz_mcts_pool_init")

    @property
    def ref(self):
        return ctypes.byref(self.struct)

    @property
    def page_nodes(self) -> int:
        return 1 << self.page_shift

    def bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self._tensors)

    # ---- host-side views for tests and statistics (each call synchronises) ----------------------
    def pool_stats(self) -> dict:
        c = self.pool_ctl.cpu().numpy()
        free = int(c[CTL_TAIL] - c[CTL_HEAD])
        return {"n_pages": self.n_pages, "page_nodes": self.page_nodes, "free_pages": free,
                "min_free_pages": int(c[CTL_MIN_FREE]), "expand_failed": int(c[CTL_EXPAND_FAILED]),
                "trees_dropped": int(c[CTL_TREES_DROPPED])}

    def node_fields(self, idx: torch.Tensor) -> dict:
        """visits / value (fp32) / prior (fp32) / first_child / parent / move / n_child of the pool indices ``idx``."""
        idx = idx.to(torch.int64)
        n, l = self.nodes[idx], self.links[idx]
        word = l[..., 1]
        return {"visits": n[..., 0], "value": n[..., 1].contiguous().view(torch.float32),
                "prior": n[..., 2].contiguous().view(torch.float32), "first_child": n[..., 3], "parent": l[..., 0],
                "move": ((word & 0xFFFF) ^ 0x8000) - 0x8000, "n_child": word >> 16}

    def children(self, node: int) -> dict:
        f = self.node_fields(torch.tensor([node], device=self.device))
        fc, nc = int(f["first_child"][0]), int(f["n_child"][0])
        return self.node_fields(torch.arange(fc, fc + nc, device=self.device))


def mcts_reset(a: Arena, mask: torch.Tensor | None = None) -> None:
    if mask is not None and (mask.dtype != torch.uint8 or mask.numel() != a.n_games):
        raise CczError("mask must be uint8 [n_games]")
    with torch.cuda.device(a.device):
        check(load().ccz_mcts_reset(a.ref, _ptr(mask), stream_ptr(a.device)), "ccz_mcts_reset")


def mcts_select(a: Arena, c_puct: float, leaf_boards: torch.Tensor, leaf_nodes: torch.Tensor) -> None:
    with torch.cuda.device(a.device):
        check(load().ccz_mcts_select(a.ref, float(c_puct), _ptr(leaf_boards), _ptr(leaf_nodes), stream_ptr(a.device)),
              "ccz_mcts_select")


def mcts_expand_backup(a: Arena, leaf_nodes, policy, policy_kind, values, move_ids, counts, flags) -> None:
    if policy.dtype != torch.float32 or values.dtype != torch.float32:
        raise CczError("policy and values must be float32")
    with torch.cuda.device(a.device):
        check(
            load().ccz_mcts_expand_backup(a.ref, _ptr(leaf_nodes), _ptr(policy), int(policy_kind), _ptr(values),
                                          _ptr(move_ids), _ptr(counts), _ptr(flags), stream_ptr(a.device)),
            "ccz_mcts_expand_backup",
        )


def mcts_root_visits(a: Arena, acts, visits, counts) -> None:
    with torch.cuda.device(a.device):
        check(load().ccz_mcts_root_visits(a.ref, _ptr(acts), _ptr(visits), _ptr(counts), stream_ptr(a.device)),
              "ccz_mcts_root_visits")


def mcts_advance(a: Arena, chosen: torch.Tensor) -> None:
    if chosen.dtype != torch.int16 or chosen.numel() != a.n_games:
        raise CczError("chosen must be int16 [n_games]")
    with torch.cuda.device(a.device):
        check(load().ccz_mcts_advance(a.ref, _ptr(chosen), stream_ptr(a.device)), "ccz_mcts_advance")


def mcts_reserve(a: Arena, pages_per_game: int) -> None:
    with torch.cuda.device(a.device):
        check(load().ccz_mcts_reserve(a.ref, int(pages_per_game), stream_ptr(a.device)), "ccz_mcts_reserve")


def mcts_migrate(src: Arena, dst: Arena) -> None:
    with torch.cuda.device(src.device):
        check(load().ccz_mcts_migrate(src.ref, dst.ref, stream_ptr(src.device)), "ccz_mcts_migrate")


def replay_pack(hist_boards, turn_plane, acts, probs, counts):
    """-> (states [2n,17,7,10,9] f16, pi [2n,2086] f64) on the device."""
    n = hist_boards.shape[0]
    dev = hist_boards.device
    states = torch.empty((2 * n, 17, 7, 10, 9), dtype=torch.float16, device=dev)
    pi = torch.empty((2 * n, N_ACTIONS), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(
            load().ccz_replay_pack(_ptr(hist_boards), _ptr(turn_plane), _ptr(acts), _ptr(probs), _ptr(counts), n,
                                   _ptr(states), _ptr(pi), stream_ptr(dev)),
            "ccz_replay_pack",
        )
    return states, pi


def _check_count(count: torch.Tensor, dev) -> None:
    if count.dtype != torch.int32 or count.numel() != 1 or count.device != dev:
        raise CczError("count must be a one-element int32 tensor on the boards' device")


def conv3x3_c256(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, skip: torch.Tensor | None = None,
                 out: torch.Tensor | None = None, variant: int = 0, count: torch.Tensor | None = None) -> torch.Tensor:
    """K9: relu(conv3x3_pad1(x, w) + bias [+ skip]) on the tcgen05 tensor cores.

    ``x`` / ``skip`` / ``out``: bf16 ``(n,256,10,9)`` tensors in ``torch.channels_last`` memory
    format (= NHWC rows of 256 channels); ``w``: bf16 ``(256,256,3,3)`` channels_last; ``bias`` fp32 (256,).
    ``variant`` 0 = the library default; other values select the tiling for measurements
    (``CONV_VARIANT_*``: 1 single-CTA tiles, 2 CTA pairs, 34 / 66 clusters of 2 / 4 pairs sharing weight stages).
    ``count``: int32 (1,) device tensor -- only the first ``count`` boards are convolved (``ccz_conv3x3_c256_count``);
    the later rows of ``out`` are left unspecified.
    """
    cl = torch.channels_last
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16 or bias.dtype != torch.float32:
        raise CczError("conv3x3_c256: x and w must be bfloat16, bias float32")
    if tuple(x.shape[1:]) != (256, 10, 9) or tuple(w.shape) != (256, 256, 3, 3) or bias.numel() != 256:
        raise CczError("conv3x3_c256: shapes must be x (n,256,10,9), w (256,256,3,3), bias (256,)")
    if not x.is_contiguous(memory_format=cl) or not w.is_contiguous(memory_format=cl):
        raise CczError("conv3x3_c256: x and w must be channels_last")
    if skip is not None and (skip.shape != x.shape or skip.dtype != x.dtype or not skip.is_contiguous(memory_format=cl)):
        raise CczError("conv3x3_c256: skip must match x (bf16, channels_last)")
    if out is None:
        out = torch.empty_like(x, memory_format=cl)
    elif out.shape != x.shape or out.dtype != x.dtype or not out.is_contiguous(memory_format=cl):
        raise CczError("conv3x3_c256: out must match x (bf16, channels_last)")
    if not 0 <= variant < 128:
        raise CczError("conv3x3_c256: variant out of range (see ccz_conv3x3_c256 in include/ccz_b200.h)")
    if not (x.is_cuda and w.is_cuda and bias.is_cuda and out.is_cuda):
        raise CczError("device tensor expected (the C ABI takes device pointers)")
    sk = None if skip is None else skip.data_ptr()
    with torch.cuda.device(x.device):
        if count is None:
            check(load().ccz_conv3x3_c256(x.data_ptr(), w.data_ptr(), bias.data_ptr(), sk, out.data_ptr(), int(x.shape[0]),
                                          int(variant), stream_ptr(x.device)), "ccz_conv3x3_c256")
        else:
            _check_count(count, x.device)
            check(load().ccz_conv3x3_c256_count(x.data_ptr(), w.data_ptr(), bias.data_ptr(), sk, out.data_ptr(), int(x.shape[0]),
                                                count.data_ptr(), int(variant), stream_ptr(x.device)), "ccz_conv3x3_c256_count")
    return out


def stem_lookup(boards: torch.Tensor, table: torch.Tensor, bias_turn: torch.Tensor, out: torch.Tensor | None = None,
                count: torch.Tensor | None = None) -> torch.Tensor:
    """K10: stem conv + BN + ReLU of search-time inputs straight from ``boards`` (n,96) uint8 ->
    bf16 ``(n,256,10,9)`` channels_last.  ``table`` bf16 (9,16,256), ``bias_turn`` fp32 (2,9,256)
    (built by ``net.stem_tables``).  ``count``: int32 (1,) device tensor -- only the first ``count`` boards
    are evaluated (``ccz_stem_lookup_count``), later output rows are not written."""
    n = boards.shape[0]
    if boards.dtype != torch.uint8 or boards.shape[1:] != (BOARD_BYTES,):
        raise CczError("stem_lookup: boards must be uint8 (n,96)")
    if table.dtype != torch.bfloat16 or tuple(table.shape) != (9, 16, 256) or bias_turn.dtype != torch.float32 \
            or tuple(bias_turn.shape) != (2, 9, 256):
        raise CczError("stem_lookup: table must be bf16 (9,16,256) and bias_turn fp32 (2,9,256)")
    if out is None:
        out = torch.empty((n, 256, 10, 9), dtype=torch.bfloat16, device=boards.device).contiguous(memory_format=torch.channels_last)
    elif tuple(out.shape) != (n, 256, 10, 9) or out.dtype != torch.bfloat16 or not out.is_contiguous(memory_format=torch.channels_last):
        raise CczError("stem_lookup: out must be bf16 (n,256,10,9) channels_last")
    with torch.cuda.device(boards.device):
        if count is None:
            check(load().ccz_stem_lookup(_ptr(boards), n, _ptr(table), _ptr(bias_turn), out.data_ptr(), stream_ptr(boards.device)),
                  "ccz_stem_lookup")
        else:
            _check_count(count, boards.device)
            check(load().ccz_stem_lookup_count(_ptr(boards), n, count.data_ptr(), _ptr(table), _ptr(bias_turn), out.data_ptr(),
                                               stream_ptr(boards.device)), "ccz_stem_lookup_count")
    return out


def heads_pack(h: torch.Tensor, operands: torch.Tensor, value_off: int, rows: torch.Tensor | None = None) -> torch.Tensor:
    """K11: ``h`` bf16 (n*90, 32) head-convolution outputs (bias added, before the ReLU) -> ``operands`` bf16 (n, K)
    with relu(policy) channel-major at column 0 and relu(value) at column ``value_off`` (net.py:96-97,103-104).
    ``rows``: int32 (n,) device tensor -- operand row b is packed from board ``rows[b]`` of ``h`` (``ccz_heads_pack_rows``);
    the caller guarantees every entry is below n."""
    n = operands.shape[0]
    if h.dtype != torch.bfloat16 or operands.dtype != torch.bfloat16 or tuple(h.shape) != (n * 90, 32):
        raise CczError("heads_pack: h must be bf16 (n*90, 32) and operands bf16 (n, K)")
    with torch.cuda.device(h.device):
        if rows is None:
            check(load().ccz_heads_pack(_ptr(h), n, _ptr(operands), int(operands.shape[1]), int(value_off), stream_ptr(h.device)),
                  "ccz_heads_pack")
        else:
            if rows.dtype != torch.int32 or rows.numel() != n:
                raise CczError("heads_pack: rows must be int32 (n,)")
            check(load().ccz_heads_pack_rows(_ptr(h), n, _ptr(rows), _ptr(operands), int(operands.shape[1]), int(value_off),
                                             stream_ptr(h.device)), "ccz_heads_pack_rows")
    return operands


def leaf_unique(boards: torch.Tensor, rows: torch.Tensor, uniq: torch.Tensor, n_unique: torch.Tensor,
                total: torch.Tensor | None = None) -> None:
    """K12: the distinct positions (bytes 0..90) of ``boards`` (n,96) uint8.  Writes ``uniq`` (n,96) rows 0..U-1 with the
    distinct records in order of first occurrence, ``rows`` int32 (n,) with each board's row in ``uniq``, ``n_unique``
    int32 (1,) = U, and adds U to ``total`` (int64 (1,)) when given.  No host synchronisation."""
    n = boards.shape[0]
    if boards.dtype != torch.uint8 or boards.shape[1:] != (BOARD_BYTES,) or uniq.dtype != torch.uint8 or uniq.shape != boards.shape:
        raise CczError("leaf_unique: boards and uniq must be uint8 (n,96)")
    if rows.dtype != torch.int32 or rows.numel() != n:
        raise CczError("leaf_unique: rows must be int32 (n,)")
    _check_count(n_unique, boards.device)
    if total is not None and (total.dtype != torch.int64 or total.numel() != 1):
        raise CczError("leaf_unique: total must be int64 (1,)")
    with torch.cuda.device(boards.device):
        check(load().ccz_leaf_unique(_ptr(boards), n, _ptr(rows), _ptr(uniq), _ptr(n_unique), _ptr(total),
                                     stream_ptr(boards.device)), "ccz_leaf_unique")


def conv3x3_plan(n_boards: int, variant: int = 0, resident_clusters: int = 74) -> dict:
    """Host-side work plan of K9 for ``n_boards`` (no device needed): see ``ccz_conv3x3_plan``."""
    out = (ctypes.c_int32 * 6)()
    check(load().ccz_conv3x3_plan(int(n_boards), int(variant), int(resident_clusters), out), "ccz_conv3x3_plan")
    keys = ("rows_per_tile", "n_tiles", "n_items", "n_full", "split_log2", "clusters")
    return dict(zip(keys, (int(v) for v in out)))
