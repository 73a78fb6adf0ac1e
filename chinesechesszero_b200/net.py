"""Host-side mirror of the reference's ``net.py`` for the self-play path.

``Net`` / ``ResBlock`` keep the reference architecture and ``state_dict`` keys (net.py:15-110) so
reference checkpoints (``torch.save(state_dict)``, net.py:208-209) load unchanged.  The new part
is :class:`BatchedEvaluator`: the search-time forward evaluated ONCE per lockstep step on the
whole leaf batch in bf16 through PyTorch (the only dense contraction of the path, hence the only
tensor-core user): eval-mode BatchNorm folded into the convolutions, channels_last, bias + skip
+ ReLU in cuDNN's fused epilogue, optional CUDA-graph capture.  Policy logits and the value come
back in fp32; the softmax over all 2086 actions is fused into the expand kernel's gather
(net.py:202-203 semantics: softmax then gather, no renormalisation).
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from . import _lib

PIECES = 7  # net.py:12
PLAYS = 17  # net.py:13
N_ACTIONS = _lib.N_ACTIONS
# conv + linear multiply-accumulates of one forward, x2 (SURVEY.md §6): 8.5506 GFLOP / position
FLOP_PER_POSITION = 2 * 4_275_314_716
PRECISIONS = ("bf16", "fp8")
E4M3_MAX = 448.0  # largest finite float8_e4m3fn


def e4m3_quantize(x: torch.Tensor, inv_scale) -> torch.Tensor:
    """``satfinite(x * inv_scale)`` in float8_e4m3fn: fp32 product, clamped to +-448, rounded to nearest even -- what the
    kernels' ``cvt.rn.satfinite.e4m3x2.f32`` computes (torch's cast alone turns values past 448 into NaN)."""
    q = (x.float() * inv_scale).clamp_(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)
    return q.contiguous(memory_format=torch.channels_last) if q.dim() == 4 else q


def weight_scales(w: torch.Tensor) -> torch.Tensor:
    """Per-output-channel e4m3 scales of a folded weight ``w`` (co, ...): ``amax|w[co]| / 448`` (1 for an all-zero channel)."""
    amax = w.detach().float().abs().flatten(1).amax(1)
    return torch.where(amax > 0, amax / E4M3_MAX, torch.ones_like(amax))


def activation_scale(amax: torch.Tensor) -> torch.Tensor:
    """Static per-tensor e4m3 scale from a calibration amax: ``amax / 448`` (1 where amax is 0)."""
    amax = amax.float()
    return torch.where(amax > 0, amax / E4M3_MAX, torch.ones_like(amax))


def calibration_boards(n: int = 1024, seed: int = 0, device="cuda") -> torch.Tensor:
    """Fixed seeded calibration positions for the FP8 evaluator, generated on the device with K1 / K2: half a seeded sample
    of the perft-4 leaves (the openings self-play starts from), half the ends of seeded uniform random playouts of 8..80
    plies (middle games and endgames)."""
    from . import positions

    rng = np.random.default_rng(seed)
    l4 = positions.perft_levels(4, device)[3]
    n_open = n // 2
    pick = np.sort(rng.choice(l4.shape[0], size=n_open, replace=False))
    opening = l4[torch.from_numpy(pick).to(l4.device)].contiguous()
    del l4
    boards = _lib.boards_start(n - n_open, device)
    depth = torch.from_numpy(rng.integers(8, 81, size=n - n_open)).to(boards.device)
    for ply in range(80):
        ids, counts, _, _ = _lib.movegen_encode(boards, planes=False)
        u = torch.from_numpy(rng.random(boards.shape[0], dtype=np.float32)).to(boards.device)
        active = ((counts > 0) & (depth > ply)).nonzero().view(-1)
        if active.numel() == 0:
            break
        c = counts[active].to(torch.int64)
        slot = torch.minimum((u[active] * c).to(torch.int64), c - 1)
        sub = boards[active].contiguous()
        _lib.board_push(sub, ids[active, slot].contiguous(), None)
        boards[active] = sub
    return torch.cat([opening, boards]).contiguous()


class ResBlock(nn.Module):
    """net.py:15-41 (same attribute names => same state_dict keys)."""

    def __init__(self, num_channels=256):
        super().__init__()
        self.conv1 = nn.Conv2d(num_channels, num_channels, kernel_size=(3, 3), stride=(1, 1), padding=1)
        self.conv1_bn = nn.BatchNorm2d(num_channels)
        self.conv1_act = nn.ReLU()
        self.conv2 = nn.Conv2d(num_channels, num_channels, kernel_size=(3, 3), stride=(1, 1), padding=1)
        self.conv2_bn = nn.BatchNorm2d(num_channels)
        self.conv2_act = nn.ReLU()

    def forward(self, x):
        y = self.conv1_act(self.conv1_bn(self.conv1(x)))
        y = self.conv2_bn(self.conv2(y))
        return self.conv2_act(x + y)


class Net(nn.Module):
    """net.py:46-110: 119->256 stem, 40 residual blocks, policy head (2086 log-probs), value head."""

    def __init__(self, num_channels=256, resblocks_num=40):
        super().__init__()
        self.input_channels = PLAYS * PIECES
        self.conv_block = nn.Conv2d(self.input_channels, num_channels, kernel_size=(3, 3), stride=(1, 1), padding=1)
        self.conv_block_bn = nn.BatchNorm2d(num_channels)
        self.conv_block_act = nn.ReLU()
        self.res_blocks = nn.ModuleList([ResBlock(num_channels=num_channels) for _ in range(resblocks_num)])
        self.policy_conv = nn.Conv2d(num_channels, PLAYS, kernel_size=(1, 1), stride=(1, 1))
        self.policy_bn = nn.BatchNorm2d(PLAYS)
        self.policy_act = nn.ReLU()
        self.policy_fc = nn.Linear(PLAYS * 10 * 9, N_ACTIONS)
        self.value_conv = nn.Conv2d(num_channels, PIECES, kernel_size=(1, 1), stride=(1, 1))
        self.value_bn = nn.BatchNorm2d(PIECES)
        self.value_act1 = nn.ReLU()
        self.value_fc1 = nn.Linear(PIECES * 10 * 9, 256)
        self.value_act2 = nn.ReLU()
        self.value_fc2 = nn.Linear(256, 1)

    def forward(self, x):
        x = x.view(x.shape[0], -1, 10, 9)
        x = self.conv_block_act(self.conv_block_bn(self.conv_block(x)))
        for block in self.res_blocks:
            x = block(x)
        policy = self.policy_act(self.policy_bn(self.policy_conv(x)))
        policy = self.policy_fc(torch.reshape(policy, [-1, PLAYS * 10 * 9]))
        policy = F.log_softmax(policy, dim=1)
        value = self.value_act1(self.value_bn(self.value_conv(x)))
        value = self.value_act2(self.value_fc1(torch.reshape(value, [-1, PIECES * 10 * 9])))
        value = torch.tanh(self.value_fc2(value))
        return policy, value


def _round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def _fold(conv: nn.Conv2d, bn: nn.BatchNorm2d):
    """Eval-mode BatchNorm folded into the preceding convolution (fp32 arithmetic)."""
    w = conv.weight.detach().float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(w.shape[0], device=w.device)
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return w * scale.view(-1, 1, 1, 1), (b - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()


def stem_tables(w: torch.Tensor, b: torch.Tensor):
    """Lookup tables of K10 (csrc/ccz_stem.cuh) from the folded stem weights ``w`` (256,119,3,3) -- already
    rounded to the evaluator's dtype -- and the fp32 bias ``b``: ``table[tap][code][co]`` bf16 (9,16,256) and
    ``bias_turn[turn][border class][co]`` fp32 (2,9,256).  Search-time inputs (net.py:160-177) are one-hot:
    red type t -> channel 7*7 + t-1, black -> 15*7 + t-1, the turn plane is channels 16*7..16*7+6."""
    wf = w.float()
    co = wf.shape[0]
    table = torch.zeros((9, 16, co), dtype=torch.float32, device=w.device)
    for t in range(1, 8):
        table[:, t, :] = wf[:, 7 * PIECES + t - 1].reshape(co, 9).t()
        table[:, 8 + t, :] = wf[:, 15 * PIECES + t - 1].reshape(co, 9).t()
    turn_w = wf[:, 16 * PIECES:17 * PIECES].sum(1)  # (co,3,3)
    bias_turn = torch.zeros((2, 9, co), dtype=torch.float32, device=w.device)
    for rc in range(3):
        for cc in range(3):
            rows = [r for r in range(3) if not (rc == 0 and r == 0) and not (rc == 2 and r == 2)]
            cols = [c for c in range(3) if not (cc == 0 and c == 0) and not (cc == 2 and c == 2)]
            bias_turn[0, rc * 3 + cc] = b.float()
            bias_turn[1, rc * 3 + cc] = b.float() + turn_w[:, rows][:, :, cols].sum((1, 2))
    return table.to(torch.bfloat16).contiguous(), bias_turn.contiguous()


class BatchedEvaluator:
    """bf16 lockstep-batch forward of a :class:`Net` (Net.forward, net.py:82-110).

    ``__call__(planes, leaf_boards) -> (logits fp32 (G,2086), POLICY_LOGITS, values fp32 (G,))``
    which is the evaluator protocol of :class:`search.LockstepSearch`.

    ``dedup`` (default on): when the stem runs from the board records (K10) and the whole tower on K9, K12 first
    compacts the leaf batch to its U distinct positions; K10 and K9 then run on U boards (the count stays on the
    device), the 1x1 heads GEMM on the compacted buffer, and K11 packs each game's FC operands from its position's
    row.  Results are bit-identical to ``dedup=False``: every board's forward output is independent of its row.

    ``precision="fp8"`` (opt-in; needs ``conv_impl="k9"`` and the 256-channel tower) runs the 80 tower convolutions on the
    e4m3 variant of K9: operands in float8_e4m3fn, fp32 accumulation, bf16 residual stream, heads and FC layers unchanged.
    Weights get one scale per output channel; activations one static scale per tensor from a calibration forward of the
    bf16 tower over ``calib_boards`` ((n,96) board records; default :func:`calibration_boards`).  ``refresh`` re-quantises
    and re-calibrates in place, so captured graphs replay with the new weights and scales.  Check the strength of a
    trained net in fp8 against bf16 with ``evaluate.EvaluationMatch(ev_fp8, ev_bf16, ...)``.
    """

    #: which kernel runs the 3x3 tower convolutions:
    #:   "k9"      hand-written tcgen05 / TMA-im2col kernel (csrc/ccz_conv.cuh) for every 256->256 conv
    #:   "k9_skip" K9 for the conv that ends a residual block (bias + skip + ReLU epilogue), cuDNN's fused
    #:             conv+bias+ReLU for the first conv of the block
    #:   "cudnn"   cuDNN's fused epilogues for both
    #:   "torch"   unfused F.conv2d (CPU-capable; used by the fp32 folding test)
    CONV_IMPLS = ("k9", "k9_skip", "cudnn", "torch")

    def __init__(self, net: Net, device="cuda", dtype=torch.bfloat16, fused_epilogue: bool = True,
                 conv_impl: str | None = None, chunk: int | None = None, dedup: bool = True, precision: str = "bf16",
                 calib_boards: torch.Tensor | None = None):
        self.device = torch.device(device)
        self.dtype = dtype
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {PRECISIONS}")
        self.precision = precision
        # leaves per sub-batch (0 = whole batch at once): sub-batches whose activations fit the 126 MB L2
        # keep the tower's layer-to-layer traffic out of HBM
        self.chunk = int(os.environ.get("CCZ_EVAL_CHUNK", "0")) if chunk is None else int(chunk)
        if conv_impl is None:
            conv_impl = os.environ.get("CCZ_CONV_IMPL", "k9") if fused_epilogue else "torch"
        if conv_impl not in self.CONV_IMPLS:
            raise ValueError(f"conv_impl must be one of {self.CONV_IMPLS}")
        k9_ok = self.device.type == "cuda" and dtype == torch.bfloat16 and net.conv_block.out_channels == 256
        if precision == "fp8" and not (conv_impl == "k9" and k9_ok):
            raise ValueError('precision="fp8" needs conv_impl="k9", a CUDA device, dtype bfloat16 and a 256-channel net')
        if conv_impl in ("k9", "k9_skip") and not k9_ok:
            conv_impl = "cudnn"  # K9 is specialised for the 256-channel bf16 tower of the reference net
        self.conv_impl = conv_impl
        self.fused = conv_impl != "torch"
        self.dedup = bool(dedup)
        self.n_evals = 0
        # boards the forward actually ran on: host part (calls without dedup) + device accumulator of K12's counts
        self._n_unique_host = 0
        self._unique_total = torch.zeros(1, dtype=torch.int64, device=self.device) if self.device.type == "cuda" else None
        self._dedup_buf: dict = {}
        self.use_heads_pack = os.environ.get("CCZ_HEADS_PACK", "1") != "0"  # K11; "0" = the torch copies (A/B measurements)
        # measurement hook (bench.py): when a list, every K9 launch of the next forwards is bracketed by CUDA
        # events on the launching stream and the (with_skip, start, end) triples are appended to it
        self.conv_events: list | None = None
        if precision == "fp8":
            if calib_boards is None:
                calib_boards = calibration_boards(device=self.device)
            elif calib_boards.dtype != torch.uint8 or calib_boards.dim() != 2 or calib_boards.shape[1] != _lib.BOARD_BYTES \
                    or calib_boards.shape[0] < 1:
                raise ValueError("calib_boards must be uint8 (n,96) board records, n >= 1")
            self.calib_boards = calib_boards.to(self.device).contiguous()
        self.refresh(net)

    def _keep(self, key: str, t: torch.Tensor) -> torch.Tensor:
        """First call: adopt ``t``.  Later calls: copy into the tensor adopted under ``key`` so that its
        device address never changes -- CUDA graphs captured by ``LockstepSearch.enable_graphs`` and the
        search loops of other owners of this evaluator keep reading valid (and current) weights."""
        old = self._params.get(key)
        if old is not None and old.shape == t.shape and old.dtype == t.dtype and old.stride() == t.stride():
            old.copy_(t)
            return old
        self._params[key] = t
        return t

    @torch.no_grad()
    def refresh(self, net: Net) -> None:
        """(Re)fold the weights of ``net`` (call after a training update).  In place: every folded tensor
        keeps its storage, so captured graphs stay valid; ``version`` counts the refreshes."""
        dev, dt = self.device, self.dtype
        cl = torch.channels_last
        if not hasattr(self, "_params"):
            self._params: dict[str, torch.Tensor] = {}
            self.version = 0
        self.version += 1
        keep = self._keep

        def conv_params(key, conv, bn):
            w, b = _fold(conv, bn)
            return (keep(key + ".w", w.to(dev, dt).contiguous(memory_format=cl)), keep(key + ".b", b.to(dev, dt)),
                    keep(key + ".b32", b.to(dev, torch.float32).contiguous()))

        self.stem = conv_params("stem", net.conv_block, net.conv_block_bn)
        # K10: with the tower on K9 the stem of search-time inputs is a table lookup over the board records
        if self.conv_impl in ("k9", "k9_skip"):
            table, bias_turn = stem_tables(self.stem[0], self.stem[2])
            self.stem_lookup = (keep("stem.table", table), keep("stem.bias_turn", bias_turn))
        else:
            self.stem_lookup = None
        self.blocks = [(conv_params(f"rb{i}.1", rb.conv1, rb.conv1_bn), conv_params(f"rb{i}.2", rb.conv2, rb.conv2_bn))
                       for i, rb in enumerate(net.res_blocks)]
        # both 1x1 heads in one convolution: 17 policy + 7 value channels
        pw, pb = _fold(net.policy_conv, net.policy_bn)
        vw, vb = _fold(net.value_conv, net.value_bn)
        self.heads_w = keep("heads.w", torch.cat([pw, vw], 0).to(dev, dt).contiguous(memory_format=cl))
        self.heads_b = keep("heads.b", torch.cat([pb, vb], 0).to(dev, dt))
        self.policy_fc = (keep("pfc.w", net.policy_fc.weight.detach().to(dev, dt).clone()),
                          keep("pfc.b", net.policy_fc.bias.detach().to(dev, torch.float32).clone()))
        self.value_fc1 = (keep("vfc1.w", net.value_fc1.weight.detach().to(dev, dt).clone()),
                          keep("vfc1.b", net.value_fc1.bias.detach().to(dev, dt).clone()))
        # 16-byte-aligned GEMM operands for the two FC layers: K = 17*90 = 1530 and 7*90 = 630 give row strides that
        # are not multiples of 16 bytes, which sends cuBLAS to a legacy sm80 kernel (113 us for the policy FC at 4096
        # leaves).  Zero-padded copies: K -> 1536 / 640, policy N -> 2088.
        self._kp, self._kv, self._np = _round_up(PLAYS * 90, 8), _round_up(PIECES * 90, 8), _round_up(N_ACTIONS, 8)
        wp = torch.zeros((self._np, self._kp), dtype=dt, device=dev)
        wp[:N_ACTIONS, :PLAYS * 90] = self.policy_fc[0]
        wv = torch.zeros((self.value_fc1[0].shape[0], self._kv), dtype=dt, device=dev)
        wv[:, :PIECES * 90] = self.value_fc1[0]
        self._fc_pad = (keep("pfc.pad", wp), keep("vfc1.pad", wv))
        if not hasattr(self, "_head_buf"):
            self._head_buf = {}
        # the fused 1x1 heads as one GEMM over the NHWC pixel rows: [g*90, C] x [C, 24 -> 32] (+ bias)
        hw = torch.zeros((32, self.heads_w.shape[1]), dtype=dt, device=dev)
        hw[:PLAYS + PIECES] = self.heads_w.reshape(PLAYS + PIECES, -1)
        hb = torch.zeros((32,), dtype=dt, device=dev)
        hb[:PLAYS + PIECES] = self.heads_b
        self._heads_gemm = (keep("heads.gemm_w", hw), keep("heads.gemm_b", hb))
        self.value_fc2 = (keep("vfc2.w", net.value_fc2.weight.detach().to(dev, torch.float32).clone()),
                          keep("vfc2.b", net.value_fc2.bias.detach().to(dev, torch.float32).clone()))
        if self.precision == "fp8":
            self._refresh_fp8(net)

    def _refresh_fp8(self, net: Net) -> None:
        """e4m3 tower operands: per-channel weight scales on the fp32 folded weights, static activation scales from a
        calibration forward of the bf16 tower (K10 + K9) over ``calib_boards``."""
        keep, dev, cl = self._keep, self.device, torch.channels_last
        amax_x, amax_y = [], []  # block inputs x_l and conv1 outputs y_l (post-ReLU, so amax = max)
        for i in range(0, self.calib_boards.shape[0], 4096):
            x = _lib.stem_lookup(self.calib_boards[i:i + 4096], *self.stem_lookup)
            ax, ay = [], []
            for (w1, _, b1), (w2, _, b2) in self.blocks:
                ax.append(x.amax())
                y = _lib.conv3x3_c256(x, w1, b1)
                ay.append(y.amax())
                x = _lib.conv3x3_c256(y, w2, b2, skip=x, out=x)
            amax_x.append(torch.stack(ax).float())
            amax_y.append(torch.stack(ay).float())
        s_x = activation_scale(torch.stack(amax_x).amax(0))
        s_y = activation_scale(torch.stack(amax_y).amax(0))
        self.fp8_scales = {"x": keep("fp8.s_x", s_x), "y": keep("fp8.s_y", s_y)}
        self._inv_sx, self._inv_sy = keep("fp8.inv_sx", 1.0 / s_x), keep("fp8.inv_sy", 1.0 / s_y)
        self.qblocks = []
        for i, rb in enumerate(net.res_blocks):
            convs = []
            for j, (conv, bn, s_in) in enumerate(((rb.conv1, rb.conv1_bn, s_x[i]), (rb.conv2, rb.conv2_bn, s_y[i])), 1):
                w, _ = _fold(conv, bn)
                w = w.to(dev)
                s_w = weight_scales(w)
                wq = e4m3_quantize(w, (1.0 / s_w).view(-1, 1, 1, 1))
                convs.append((keep(f"rb{i}.{j}.wq", wq.contiguous(memory_format=cl)), keep(f"rb{i}.{j}.deq", (s_in * s_w).contiguous()),
                              self.blocks[i][j - 1][2]))
            self.qblocks.append(tuple(convs))

    def _tower_fp8(self, x, xq, count=None):
        """The residual tower on e4m3 K9: conv1 reads xq_l and writes yq_l only; conv2 reads yq_l and the bf16 skip x_l and
        writes x_{l+1} over x_l plus (except in the last block) xq_{l+1} over xq_l."""
        yq = torch.empty_like(xq, memory_format=torch.channels_last)
        last = len(self.qblocks) - 1
        for i, (c1, c2) in enumerate(self.qblocks):
            _lib.conv3x3_c256_e4m3(xq, *c1, y=False, out_q=yq, inv_s_out=self._inv_sy[i:i + 1], count=count)
            _lib.conv3x3_c256_e4m3(yq, *c2, skip=x, out=x, out_q=None if i == last else xq,
                                   inv_s_out=None if i == last else self._inv_sx[i + 1:i + 2], count=count)
        return x

    def _k9(self, x, w, b32, skip, out, count=None):
        if self.conv_events is None:
            return _lib.conv3x3_c256(x, w, b32, skip=skip, out=out, count=count)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y = _lib.conv3x3_c256(x, w, b32, skip=skip, out=out, count=count)
        e1.record()
        self.conv_events.append((skip is not None, e0, e1))
        return y

    def _conv_relu(self, x, wb, k9=False, count=None):
        w, b, b32 = wb
        if k9:
            return self._k9(x, w, b32, None, None, count)
        if self.fused:
            return torch.cudnn_convolution_relu(x, w, b, (1, 1), (1, 1), (1, 1), 1)
        return F.relu_(F.conv2d(x, w, b, padding=1))

    def _conv_add_relu(self, x, wb, skip, k9=False, count=None):
        w, b, b32 = wb
        if k9:  # the block's output overwrites its input (each tile reads its skip rows before storing them)
            return self._k9(x, w, b32, skip, skip, count)
        if self.fused:
            return torch.cudnn_convolution_add_relu(x, w, skip, 1.0, b, (1, 1), (1, 1), (1, 1), 1)
        return F.relu_(F.conv2d(x, w, b, padding=1).add_(skip))

    @property
    def needs_planes(self) -> bool:
        """False when ``__call__`` evaluates the stem from the board records (K10) and ignores ``planes``."""
        return self.stem_lookup is None

    @torch.no_grad()
    def forward(self, planes: torch.Tensor | None, boards: torch.Tensor | None = None):
        """(logits fp32 (g,2086), values fp32 (g,)).  ``planes``: any (g,17,7,10,9) net input.  ``boards``:
        (g,96) board records of SEARCH-TIME positions (no history planes, net.py:160-177); when given and the
        tower runs on K9, the stem is evaluated from them by K10 and ``planes`` is not read."""
        use_boards = boards is not None and self.stem_lookup is not None
        g = boards.shape[0] if use_boards else planes.shape[0]
        if self.chunk and g > self.chunk:
            parts = [self._forward(None if use_boards else planes[i:i + self.chunk],
                                   boards[i:i + self.chunk] if use_boards else None) for i in range(0, g, self.chunk)]
            return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])
        return self._forward(None if use_boards else planes, boards if use_boards else None)

    @property
    def n_unique(self) -> int:
        """Boards the forwards so far ran on (distinct leaves where dedup applied); reading it synchronises."""
        dev = int(self._unique_total.item()) if self._unique_total is not None else 0
        return self._n_unique_host + dev

    def _dedup_buffers(self, g: int):
        """(rows int32 (g,), uniq boards uint8 (g,96), n_unique int32 (1,)) kept per batch size: fixed addresses for
        captured graphs."""
        buf = self._dedup_buf.get(g)
        if buf is None:
            z = dict(device=self.device)
            buf = self._dedup_buf[g] = (torch.zeros(g, dtype=torch.int32, **z), torch.zeros((g, _lib.BOARD_BYTES), dtype=torch.uint8, **z),
                                        torch.zeros(1, dtype=torch.int32, **z))
            if len(self._dedup_buf) > 8:
                self._dedup_buf.pop(next(iter(self._dedup_buf)))
        return buf

    def _forward(self, planes, boards=None):
        row_map = count = None
        if boards is not None:
            g = boards.shape[0]
            if self.dedup and self.conv_impl == "k9" and g <= _lib.DEDUP_MAX_BOARDS:
                # K12: forward the distinct positions only (rows 0..U-1); rows >= U of every activation are don't-care
                row_map, uniq, count = self._dedup_buffers(g)
                _lib.leaf_unique(boards, row_map, uniq, count, self._unique_total)
                boards = uniq
            else:
                self._n_unique_host += g
            if self.precision == "fp8":
                x, xq = _lib.stem_lookup_e4m3(boards, *self.stem_lookup, self._inv_sx[0:1], count=count)
            else:
                x = _lib.stem_lookup(boards, *self.stem_lookup, count=count)
        else:
            g = planes.shape[0]
            x = planes.view(g, PLAYS * PIECES, 10, 9).contiguous(memory_format=torch.channels_last)
            x = self._conv_relu(x, self.stem)
            if self.precision == "fp8":
                xq = e4m3_quantize(x, self._inv_sx[0:1])
            self._n_unique_host += g
        if self.precision == "fp8":
            x = self._tower_fp8(x, xq, count)
        else:
            k9_plain, k9_skip = self.conv_impl == "k9", self.conv_impl in ("k9", "k9_skip")
            for c1, c2 in self.blocks:
                y = self._conv_relu(x, c1, k9_plain, count)
                x = self._conv_add_relu(y, c2, x, k9_skip, count)
        if self.device.type == "cuda":
            # 1x1 heads = a GEMM over the (g*90, C) NHWC pixel rows (a view of the channels_last activations)
            rows = x.permute(0, 2, 3, 1).reshape(g * 90, x.shape[1])
            h = F.linear(rows, *self._heads_gemm)
            buf = self._head_buf.get(g)  # [policy operand | value operand], pad columns stay zero
            if buf is None:
                buf = self._head_buf[g] = torch.zeros((g, self._kp + self._kv), dtype=h.dtype, device=h.device)
                if len(self._head_buf) > 8:
                    self._head_buf.pop(next(iter(self._head_buf)))
            if self.dtype == torch.bfloat16 and self.use_heads_pack:
                # K11: ReLU + NHWC -> NCHW flatten order (channel-major within a board, net.py:97) in one launch;
                # with dedup, game b's operands come from its position's compacted row row_map[b]
                _lib.heads_pack(h, buf, self._kp, rows=row_map)
            else:
                h = F.relu_(h).view(g, 90, 32)
                if row_map is not None:
                    h = h.index_select(0, row_map)
                buf[:, :PLAYS * 90].view(g, PLAYS, 90).copy_(h[:, :, :PLAYS].transpose(1, 2))
                buf[:, self._kp:self._kp + PIECES * 90].view(g, PIECES, 90).copy_(h[:, :, PLAYS:PLAYS + PIECES].transpose(1, 2))
            logits = F.linear(buf[:, :self._kp], self._fc_pad[0])[:, :N_ACTIONS].float() + self.policy_fc[1]
            v = F.relu_(F.linear(buf[:, self._kp:], self._fc_pad[1], self.value_fc1[1])).float()
        else:
            h = F.relu_(F.conv2d(x, self.heads_w, self.heads_b))  # (g, 24, 10, 9)
            hp = h[:, :PLAYS].reshape(g, PLAYS * 90)               # NCHW flatten order, net.py:97
            hv = h[:, PLAYS:].reshape(g, PIECES * 90)
            logits = F.linear(hp, self.policy_fc[0]).float() + self.policy_fc[1]
            v = F.relu_(F.linear(hv, *self.value_fc1)).float()
        v = torch.tanh(F.linear(v, *self.value_fc2)).view(g)
        return logits, v

    def __call__(self, planes, leaf_boards=None):
        logits, v = self.forward(planes, leaf_boards)
        self.n_evals += logits.shape[0]
        return logits, _lib.POLICY_LOGITS, v


class PolicyValueNet:
    """Same constructor, attributes and methods as the reference class (net.py:113-247) for the
    self-play path: ``policy_value_net`` (an nn.Module with the reference state_dict keys),
    ``policy_value(state_batch)``, ``policy_value_fn(board)``, ``save_model(path)``."""

    def __init__(self, model=None, use_gpu=True, num_channels=256, resblocks_num=40):
        self.use_gpu = use_gpu
        self.l2_const = 2e-3
        self.device = torch.device("cuda") if (use_gpu and torch.cuda.is_available()) else torch.device("cpu")
        self.policy_value_net = Net(num_channels, resblocks_num).to(self.device)
        self.optimizer = torch.optim.Adam(self.policy_value_net.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                                          weight_decay=self.l2_const)
        if model:
            self.policy_value_net.load_state_dict(torch.load(model, map_location=self.device))
        self._evaluator = None

    def evaluator(self, **kw) -> BatchedEvaluator:
        """The lockstep-batch evaluator over the current weights (CUDA only, no fallback); ``precision="fp8"`` for the
        e4m3 tower (see :class:`BatchedEvaluator`)."""
        if self.device.type != "cuda":
            raise _lib.CczError("BatchedEvaluator needs a CUDA device; there is no CPU fallback")
        if self._evaluator is None:
            self.policy_value_net.eval()
            self._evaluator = BatchedEvaluator(self.policy_value_net, self.device, **kw)
        return self._evaluator

    def policy_value(self, state_batch):
        """net.py:138-148: (act_probs ndarray (N,2086), value ndarray (N,1)) for a state batch."""
        self.policy_value_net.eval()
        if not isinstance(state_batch, torch.Tensor):
            state_batch = torch.tensor(np.asarray(state_batch), dtype=torch.float)
        state_batch = state_batch.to(self.device, torch.float32)
        with torch.no_grad():
            log_act_probs, value = self.policy_value_net(state_batch)
        return np.exp(log_act_probs.cpu().numpy()), value.cpu().numpy()

    def policy_value_fn(self, board, red_states=None, black_states=None):
        """net.py:151-205 for ONE position given as a 96-byte board record (or an object with
        ``.record()``): ``(zip(legal_ids, probs[legal_ids]), value ndarray (1,1))``.  Legal ids and
        the input planes come from the CUDA kernel (ccz_movegen_encode); the forward runs in bf16."""
        rec = board.record() if hasattr(board, "record") else board
        boards = torch.as_tensor(np.ascontiguousarray(rec, dtype=np.uint8).reshape(1, 96)).to(self.device)
        ids, counts, _, planes = _lib.movegen_encode(boards)
        logits, v = self.evaluator().forward(planes)
        probs = torch.softmax(logits, dim=1)[0].cpu().numpy()
        legal = ids[0, : int(counts[0])].cpu().numpy().astype(np.int64)
        return zip(legal.tolist(), probs[legal]), v.cpu().numpy().reshape(1, 1)

    def save_model(self, model_file):
        torch.save(self.policy_value_net.state_dict(), model_file)
