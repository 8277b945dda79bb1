"""Host-side mirror of `model.score.ScoreUNet` (reference model/score.py:37-70, model/nn.py:88-242).

Same constructor signature, same parameter names / shapes / initialisation order as the reference module, so
reference state_dicts and pickled snapshots load unchanged; the arithmetic is done by the CUDA library
(climate2weather_b200/csrc via include/c2w_b200.h).  There is no torch-op forward and no CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor, nn

from . import _lib

NOISE_FEATURES = 32  # model/score.py:53


def _layer_specs(channels: int, embedding_dim: int, hidden_channels: Sequence[int], hidden_blocks: Sequence[int],
                 attention_levels: Sequence[int], ks: int, forcing_dim: int = 0) -> List[Tuple[str, Tuple[int, ...]]]:
    """state_dict prefixes and weight shapes in the reference's construction order (model/nn.py:165-218;
    `tails` / `ascent` are stored reversed, :216,218), followed by the time MLP (model/score.py:56-57)."""
    nl = len(hidden_blocks)
    ch = list(hidden_channels)
    specs: List[Tuple[str, Tuple[int, ...]]] = []
    if forcing_dim > 0:  # model/score.py:49-51: the forcing Linear is constructed before the UNet
        specs.append(("map_forcing", (embedding_dim, forcing_dim)))
    for lvl in range(nl):
        rev = nl - 1 - lvl
        if lvl == 0:
            specs.append(("unet.heads.0", (ch[0], channels, ks, ks)))
            specs.append((f"unet.tails.{rev}", (channels, ch[0], ks, ks)))
        else:
            specs.append((f"unet.heads.{lvl}.0", (ch[lvl], ch[lvl - 1], ks, ks)))
            specs.append((f"unet.tails.{rev}.2", (ch[lvl - 1], ch[lvl], ks, ks)))
        has_attn = lvl in attention_levels
        step = 2 if has_attn else 1
        for b in range(hidden_blocks[lvl]):
            sides = (("descent", lvl), ("ascent", rev))
            for side, idx in sides:
                p = f"unet.{side}.{idx}.{b * step}"
                specs.append((p + ".project.0", (ch[lvl], embedding_dim)))
                specs.append((p + ".residue.1", (ch[lvl], ch[lvl], ks, ks)))
                specs.append((p + ".residue.3", (ch[lvl], ch[lvl], ks, ks)))
            if has_attn:
                for side, idx in sides:
                    p = f"unet.{side}.{idx}.{b * step + 1}"
                    specs.append((p + ".qkv", (3 * ch[lvl], ch[lvl], 1)))
                    specs.append((p + ".proj_out", (ch[lvl], ch[lvl], 1)))
    specs.append(("map_layer0", (embedding_dim, NOISE_FEATURES)))
    specs.append(("map_layer1", (embedding_dim, embedding_dim)))
    return specs


#: id(parameter) -> (weakref(parameter), weakref(ScoreUNet that owns it))
_PARAM_OWNER: Dict[int, tuple] = {}


def owner_of(p: nn.Parameter):
    hit = _PARAM_OWNER.get(id(p))
    return hit[1]() if hit is not None and hit[0]() is p else None


class _Node(nn.Module):
    """Anonymous container: gives parameters the dotted names of the reference module tree."""


def _register(root: nn.Module, dotted: str, param: nn.Parameter) -> None:
    parts = dotted.split(".")
    node = root
    for part in parts[:-1]:
        if part not in node._modules:
            node.add_module(part, _Node())
        node = node._modules[part]
    node.register_parameter(parts[-1], param)


class Engine:
    """One c2w handle: packed weights + workspace for a fixed (frame_channels, window, H, W)."""

    def __init__(self, net: "ScoreUNet", frame_channels: int, window: int, height: int, width: int,
                 device: torch.device, max_windows: int, vjp: bool = False, per_sample_t: bool = False,
                 train: bool = False, tile_windows: int = 0):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.C2WError("climate2weather_b200 runs on CUDA devices only (no CPU path)")
        cfg = _lib.Config()
        cfg.frame_channels, cfg.window, cfg.height, cfg.width = frame_channels, window, height, width
        cfg.embedding_dim, cfg.noise_features = net.embedding_dim, NOISE_FEATURES
        cfg.n_levels = len(net.hidden_blocks)
        if cfg.n_levels > _lib.MAX_LEVELS:
            raise _lib.C2WError("too many UNet levels")
        for i, (c, b) in enumerate(zip(net.hidden_channels, net.hidden_blocks)):
            cfg.hidden_channels[i], cfg.hidden_blocks[i] = c, b
        cfg.attention_mask = sum(1 << l for l in net.attention_levels)
        cfg.forcing_dim = int(getattr(net, "forcing_dim", 0))
        self.frame_channels, self.window, self.height, self.width = frame_channels, window, height, width
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_create(ctypes.byref(cfg), ctypes.byref(self.handle)), "c2w_create")
            for name, p in net.state_dict().items():
                w = p.detach().to(device="cpu", dtype=torch.float32).contiguous()
                _lib.check(self.lib.c2w_load_weight(self.handle, name.encode(), w.data_ptr(), w.numel()),
                           f"c2w_load_weight({name})")
            _lib.check(self.lib.c2w_finalize_weights(self.handle), "c2w_finalize_weights")
            self.max_windows = 0
            self.tile_windows = 0
            self.workspace = None
            self.vjp = bool(vjp) or bool(train)
            self.per_sample_t = bool(per_sample_t) or bool(train)
            self.train = bool(train)
            self.param_total = int(self.lib.c2w_param_total(self.handle))
            self.layout: Dict[str, Tuple[int, int]] = {}
            off, num = ctypes.c_int64(), ctypes.c_int64()
            for name in net.state_dict():
                _lib.check(self.lib.c2w_param_layout(self.handle, name.encode(), ctypes.byref(off), ctypes.byref(num)),
                           f"c2w_param_layout({name})")
                self.layout[name] = (int(off.value), int(num.value))
            self._flat_scratch: Optional[Tensor] = None
            self._train_token = None
            self.bind(max_windows, tile_windows)

    def bind(self, max_windows: int, tile_windows: int = 0) -> None:
        """Binds a workspace of max_windows windows.  tile_windows > 0 (an ensemble, plain workspace only): the convs are
        planned (tile width, CTA pair, main loop) as for tile_windows windows, a member's own workspace
        (c2w_bind_workspace_members)."""
        flags = _lib.WS_TRAIN if self.train else ((_lib.WS_VJP if self.vjp else 0) |
                                                  (_lib.WS_PER_SAMPLE_T if self.per_sample_t else 0))
        with torch.cuda.device(self.device):
            nbytes = self.lib.c2w_workspace_bytes_ex(self.handle, max_windows, flags)
            if nbytes < 0:
                _lib.check(-1, "c2w_workspace_bytes")
            self.workspace = None  # release the old arena before taking the new one
            self.workspace = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
            if tile_windows:
                if flags:
                    raise _lib.C2WError("an ensemble workspace is a plain one (no VJP / per-sample times)")
                _lib.check(self.lib.c2w_bind_workspace_members(self.handle, max_windows, tile_windows,
                                                               self.workspace.data_ptr(), self.workspace.numel()),
                           "c2w_bind_workspace_members")
            else:
                _lib.check(self.lib.c2w_bind_workspace_ex(self.handle, max_windows, self.workspace.data_ptr(),
                                                          self.workspace.numel(), flags), "c2w_bind_workspace")
            self.max_windows, self.tile_windows = max_windows, tile_windows

    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def unet_forward(self, x: Tensor, t: float) -> Tensor:
        """x: fp32 NCHW [n, C*window, H, W] on self.device."""
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_unet_forward(self.handle, x.data_ptr(), x.shape[0], float(t), out.data_ptr(),
                                                 self.stream), "c2w_unet_forward")
        return out

    def set_forcing(self, forcing: Optional[Tensor]) -> None:
        """Forcing rows [n, forcing_dim] (device fp32) of the next per-sample forward / training calls, or None."""
        self._forcing_keepalive = forcing
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_set_forcing(self.handle, forcing.data_ptr() if forcing is not None else None),
                       "c2w_set_forcing")

    def unet_forward_t(self, x: Tensor, t: Tensor) -> Tensor:
        """x: fp32 NCHW [n, C*window, H, W]; t: fp32 [n] on self.device (one diffusion time per sample)."""
        assert self.per_sample_t, "engine was built without per-sample modulation"
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_unet_forward_t(self.handle, x.data_ptr(), x.shape[0], t.data_ptr(), out.data_ptr(),
                                                   self.stream), "c2w_unet_forward_t")
        return out

    # ------------------------------------------------------------------------------------------ training step
    def refresh_weights(self, net: "ScoreUNet") -> None:
        """Re-packs the weights from the module's CURRENT parameters on the device (after an optimiser step): no host
        round trip, the workspace stays bound.  Zero-copy when the parameters are views of one flat buffer in the
        library's layout (optim.AdamW); gathered into a scratch buffer otherwise."""
        params = dict(net.state_dict(keep_vars=True))
        first = next(iter(self.layout))
        base = params[first].data_ptr() - 4 * self.layout[first][0]
        aliased = all(p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and
                      p.data_ptr() == base + 4 * self.layout[k][0] for k, p in params.items())
        with torch.cuda.device(self.device):
            if aliased:
                ptr = base
            else:
                if self._flat_scratch is None:
                    self._flat_scratch = torch.zeros(self.param_total, dtype=torch.float32, device=self.device)
                for k, p in params.items():
                    o, n = self.layout[k]
                    self._flat_scratch[o:o + n].copy_(p.detach().reshape(-1))
                ptr = self._flat_scratch.data_ptr()
            _lib.check(self.lib.c2w_refresh_weights(self.handle, ptr, self.stream), "c2w_refresh_weights")

    def train_forward(self, x: Tensor, t: Tensor) -> Tensor:
        """net(x, t) with one diffusion time per sample, stashing for train_backward.  x: fp32 NCHW [n <= max_windows]."""
        assert self.train, "engine was built without the training workspace"
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_train_forward(self.handle, x.data_ptr(), x.shape[0], t.data_ptr(), out.data_ptr(),
                                                  self.stream), "c2w_train_forward")
        self._t_keepalive = t  # the backward re-reads the diffusion times
        return out

    def train_backward(self, gout: Tensor, grad_flat: Tensor, want_gin: bool = False, accumulate: bool = False):
        """All parameter gradients of the last train_forward into grad_flat (fp32, library layout); returns the input
        gradient if asked."""
        gin = torch.empty_like(gout) if want_gin else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_train_backward(self.handle, gout.data_ptr(), gout.shape[0],
                                                   gin.data_ptr() if gin is not None else None, grad_flat.data_ptr(),
                                                   int(accumulate), self.stream), "c2w_train_backward")
        return gin

    def unet_vjp(self, x: Tensor, t: float, gout: Tensor):
        """(out, gin): forward and (d out / d x)^T gout for x, gout: fp32 NCHW [n, C*window, H, W], chunked."""
        assert self.vjp, "engine was built without a VJP workspace"
        out, gin = torch.empty_like(x), torch.empty_like(x)
        with torch.cuda.device(self.device):
            for i in range(0, x.shape[0], self.max_windows):
                xs, gs = x[i:i + self.max_windows], gout[i:i + self.max_windows]
                _lib.check(self.lib.c2w_unet_vjp(self.handle, xs.data_ptr(), xs.shape[0], float(t), gs.data_ptr(),
                                                 out[i:].data_ptr(), gin[i:].data_ptr(), self.stream), "c2w_unet_vjp")
        return out, gin

    def window_score_backward(self, cot: Tensor, frame_global0: int, win_first: int, n_win: int, n_win_global: int,
                              vjp: Tensor) -> None:
        """Adjoint of the last window_score call (same window range, one chunk); accumulates into vjp."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_window_score_backward(self.handle, cot.data_ptr(), cot.shape[0], frame_global0,
                                                          win_first, n_win, n_win_global, vjp.data_ptr(), self.stream),
                       "c2w_window_score_backward")

    def window_score_sel(self, traj: Tensor, frame_global0: int, win_list: Tensor, t: float, n_win_global: int = 0,
                         eps: Optional[Tensor] = None) -> None:
        """Forward of the selected windows (global indices, int32 device tensor): stashing on a VJP workspace, chunked
        on a plain one; with `eps` their part of the composed score is written into it."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_window_score_sel(self.handle, traj.data_ptr(), traj.shape[0], frame_global0,
                                                     win_list.data_ptr(), win_list.numel(), n_win_global, float(t),
                                                     eps.data_ptr() if eps is not None else None, self.stream),
                       "c2w_window_score_sel")

    def window_score_backward_sel(self, cot: Tensor, frame_global0: int, win_list: Tensor, pos: Tensor, n_win_global: int,
                                  vjp: Tensor) -> None:
        """Adjoint of the last window_score_sel call (same list); accumulates into vjp."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_window_score_backward_sel(self.handle, cot.data_ptr(), cot.shape[0], frame_global0,
                                                              win_list.data_ptr(), pos.data_ptr(), win_list.numel(),
                                                              n_win_global, vjp.data_ptr(), self.stream),
                       "c2w_window_score_backward_sel")

    def window_score(self, traj: Tensor, frame_global0: int, win_first: int, n_win: int, n_win_global: int, t: float,
                     eps: Tensor) -> None:
        """traj / eps: fp32 [frames_local, H, W, C] device layout."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_window_score(self.handle, traj.data_ptr(), traj.shape[0], frame_global0, win_first,
                                                 n_win, n_win_global, float(t), eps.data_ptr(), self.stream),
                       "c2w_window_score")

    def window_score_members(self, traj: Tensor, n_members: int, member_frames: int, win_first: int, n_win: int,
                             t: float, eps: Tensor) -> None:
        """Windows [win_first, win_first + n_win) of an ensemble stored member-major: traj / eps fp32
        [n_members * member_frames, H, W, C] (c2w_window_score_members)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_window_score_members(self.handle, traj.data_ptr(), n_members, member_frames,
                                                         win_first, n_win, float(t), eps.data_ptr(), self.stream),
                       "c2w_window_score_members")

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                self.lib.c2w_destroy(self.handle)
                self.handle = ctypes.c_void_p()
        except Exception:
            pass


class ScoreUNet(nn.Module):
    r"""Drop-in for `model.score.ScoreUNet(channels, embedding_dim, forcing_dim=0, **unet_kwargs)`.

    Arguments mirror model/score.py:46 and model/nn.py:108-121.  Supported: kernel_size=3, stride=2, spatial=2,
    SiLU activation, zero padding, forcing_dim=0 — i.e. configs/sda_unet.yml with train.py:164-173 — with any
    hidden_channels (multiples of 64, <= 512), hidden_blocks and attention_levels.

    Geometry: every level l (H_l x W_l, halved from the patch per level) must have W_l >= 8 and either W_l a power
    of two <= 128 whose rows tile into 128-pixel row blocks, or W_l a multiple of 128 (e.g. 128 x 256, 256 x 256,
    512 x 512); H_l and W_l are even below the last level.  Other widths (96, 160, 192, ...) are refused when the
    engine is created.
    """

    DEFAULT_MAX_WINDOWS = 16

    def __init__(self, channels: int, embedding_dim: int, forcing_dim: int = 0,
                 hidden_channels: Sequence[int] = (32, 64, 128), hidden_blocks: Sequence[int] = (2, 3, 5),
                 attention_levels: Sequence[int] = (), kernel_size=3, stride=2, activation=None, spatial: int = 2,
                 padding_mode: str = "zeros", **kwargs):
        super().__init__()
        if activation is None:
            # the reference's own default is torch.nn.ReLU (model/nn.py:118); every config passes SiLU (train.py:171).
            # Falling back to either silently would build a different network than the caller may expect.
            raise NotImplementedError("climate2weather_b200.ScoreUNet: pass activation=torch.nn.SiLU explicitly (the "
                                      "reference default, ReLU, is not built; train.py:171 configures SiLU)")
        ks = kernel_size if isinstance(kernel_size, int) else kernel_size[0]
        st = stride if isinstance(stride, int) else stride[0]
        unsupported = []
        if ks != 3 or st != 2 or spatial != 2:
            unsupported.append("kernel_size/stride/spatial other than 3/2/2")
        if padding_mode != "zeros":
            unsupported.append(f"padding_mode={padding_mode!r}")
        if activation is not nn.SiLU and not isinstance(activation, nn.SiLU):
            unsupported.append("activation other than SiLU")
        if kwargs:
            unsupported.append(f"extra conv kwargs {sorted(kwargs)}")
        if unsupported:
            raise NotImplementedError("climate2weather_b200.ScoreUNet: " + "; ".join(unsupported))
        self.channels = int(channels)
        self.embedding_dim = int(embedding_dim)
        self.noise_features = NOISE_FEATURES
        self.hidden_channels = [int(c) for c in hidden_channels]
        self.hidden_blocks = [int(b) for b in hidden_blocks]
        self.attention_levels = sorted(int(a) for a in attention_levels)
        self.forcing_dim = int(forcing_dim)
        # Parameters are created by torch's own Conv/Linear initialisers in the reference's construction order, so
        # `torch.manual_seed(s); ScoreUNet(...)` yields the same weights as the reference module.
        for prefix, shape in _layer_specs(self.channels, self.embedding_dim, self.hidden_channels, self.hidden_blocks,
                                          self.attention_levels, ks, self.forcing_dim):
            w = torch.empty(shape)
            nn.init.kaiming_uniform_(w, a=math.sqrt(5))
            bound = 1.0 / math.sqrt(w[0].numel())
            b = torch.empty(shape[0]).uniform_(-bound, bound)
            _register(self, prefix + ".weight", nn.Parameter(w))
            _register(self, prefix + ".bias", nn.Parameter(b))
        self._engines: Dict[tuple, Engine] = {}
        self._weights_epoch = 0
        self._tag_parameters()

    def _tag_parameters(self) -> None:
        """Lets an optimiser built from `net.parameters()` alone find the module whose engines it must invalidate."""
        ref = weakref.ref(self)
        for p in self.parameters():
            # a side table keyed by identity, not an attribute: parameters must stay picklable
            _PARAM_OWNER[id(p)] = (weakref.ref(p, lambda _, k=id(p): _PARAM_OWNER.pop(k, None)), ref)

    def invalidate_engines(self) -> None:
        """Declare the parameters changed behind autograd's back (raw-pointer optimiser / EMA updates do not bump
        `Tensor._version`): the next forward re-packs the weights instead of serving the cached engine."""
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_engines"] = {}  # device handles are rebuilt lazily after unpickling / deepcopy
        state["_direct_grad"] = None  # an optimiser's buffer: never shared with copies (EMA) or pickled
        return state

    def __setstate__(self, state):
        """Also accepts the pickled state of a REFERENCE `model.score.ScoreUNet` (a network snapshot,
        training_loop.py:250-266, unpickled through `compat.install()`): the module tree keeps the reference's
        parameter names, and the architecture description is read off their shapes."""
        super().__setstate__(state)  # also restores the hook dictionaries older pickles lack
        self._engines = {}
        self._weights_epoch = 0
        self._tag_parameters()
        if "hidden_blocks" not in state:
            _validate_reference_tree(self)
            arch = _arch_from_state_dict(self.state_dict())
            self.channels, self.embedding_dim = arch["channels"], arch["embedding_dim"]
            self.noise_features = NOISE_FEATURES
            self.hidden_channels, self.hidden_blocks = arch["hidden_channels"], arch["hidden_blocks"]
            self.attention_levels = arch["attention_levels"]
            mf = self.state_dict().get("map_forcing.weight")
            self.forcing_dim = int(mf.shape[1]) if mf is not None else 0

    # ---------------------------------------------------------------------------------------------- engines
    def _fingerprint(self) -> tuple:
        return (getattr(self, "_weights_epoch", 0),) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def engine(self, frame_channels: int, window: int, height: int, width: int, device, max_windows: Optional[int] = None,
               vjp: bool = False, per_sample_t: bool = False, train: bool = False, tile_windows: int = 0) -> Engine:
        """Packed-weight engine for this geometry; if the parameters changed since it was packed (and still live on its
        device) the weights are re-packed in place on the device, otherwise the engine is rebuilt.  tile_windows: see
        Engine.bind (an ensemble's workspace); 0 plans the tiles for the bound window count."""
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if frame_channels * window != self.channels:
            raise ValueError(f"frame_channels*window = {frame_channels * window} != channels = {self.channels}")
        # an ensemble's engine (tile_windows > 0) is kept apart from the plain one: alternating ensemble and single runs
        # then rebind neither
        key = (frame_channels, window, height, width, str(device), bool(vjp), bool(per_sample_t), bool(train),
               bool(tile_windows))
        fp = self._fingerprint()
        hit = self._engines.get(key)
        want = max_windows or self.DEFAULT_MAX_WINDOWS
        if hit is not None:
            eng = hit[0]
            if hit[1] != fp:
                if not all(p.is_cuda and p.device == eng.device for p in self.parameters()):
                    hit = None  # the module moved: rebuild below
                else:
                    eng.refresh_weights(self)
                    self._engines[key] = (eng, fp)
            if hit is not None:
                if (max_windows is not None and eng.max_windows != max_windows) or eng.tile_windows != tile_windows:
                    eng.bind(max_windows or eng.max_windows, tile_windows)
                return eng
        eng = Engine(self, frame_channels, window, height, width, device, want, vjp=vjp, per_sample_t=per_sample_t,
                     train=train, tile_windows=tile_windows)
        self._engines[key] = (eng, fp)
        return eng

    def from_reference(self, module: nn.Module) -> "ScoreUNet":
        """Copies the weights of a reference `model.score.ScoreUNet` (any dtype; snapshots are fp16)."""
        self.load_state_dict({k: v.float() for k, v in module.state_dict().items()})
        return self

    # ---------------------------------------------------------------------------------------------- forward
    def forward(self, x: Tensor, t: Tensor, forcing: Optional[Tensor] = None) -> Tensor:
        """model/score.py:59-70.  x: [B, channels, H, W] on a CUDA device; t: one diffusion time for the batch."""
        fdim = int(getattr(self, "forcing_dim", 0))
        assert (forcing is None) or fdim > 0  # model/score.py:60
        if fdim > 0 and forcing is None:
            raise ValueError("this ScoreUNet has a forcing branch (forcing_dim > 0): pass forcing=")
        if not x.is_cuda:
            raise _lib.C2WError("ScoreUNet.forward: input must live on a CUDA device (no CPU path); "
                                "BatchedScoreFunction moves window batches for you")
        tt = torch.as_tensor(t).reshape(-1).float()
        B, Cc, H, W = x.shape
        training = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if tt.numel() not in (1, B):
            raise ValueError(f"t has {tt.numel()} entries for a batch of {B}")
        f_dev = None
        if forcing is not None:  # [B, forcing_dim] (a single row is broadcast like the reference's emb + Linear(forcing))
            f_dev = torch.as_tensor(forcing, dtype=torch.float32).reshape(-1, fdim).to(x.device)
            f_dev = (f_dev if f_dev.shape[0] == B else f_dev.expand(B, fdim)).contiguous()
        if not training and (f_dev is not None or (tt.numel() != 1 and not bool((tt == tt[0]).all()))):
            # one diffusion time per sample (model/score.py:61; the DSM objective, src/thor/pipelines.py:27-35)
            if torch.is_grad_enabled() and x.requires_grad:
                raise NotImplementedError("input gradients with per-sample diffusion times need trainable parameters "
                                          "(the training workspace); freeze nothing or use one diffusion time")
            eng = self.engine(Cc, 1, H, W, x.device, per_sample_t=True)
            eng.set_forcing(f_dev)
            t_all = (tt if tt.numel() == B else tt.expand(B)).to(x.device).contiguous()
            out = eng.unet_forward_t(x.detach().float().contiguous(), t_all)
            eng.set_forcing(None)
            return out.to(x.dtype).reshape(x.shape)
        B, Cc, H, W = x.shape
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training (training_loop.py:372-378): forward with stashing now, all parameter gradients in backward
            t_dev = (tt if tt.numel() == B else tt.expand(B)).to(device=x.device, dtype=torch.float32).contiguous()
            params = [p for p in self.parameters()]
            return _UNetTrainFn.apply(x, t_dev, self, f_dev, *params)
        if torch.is_grad_enabled() and x.requires_grad:
            # input gradients only (the weights are frozen in sampling, training_loop.py:257)
            return _UNetInputVJP.apply(x, self, float(tt[0]))
        eng = self.engine(Cc, 1, H, W, x.device)
        out = eng.unet_forward(x.detach().float().contiguous(), float(tt[0]))
        return out.to(x.dtype).reshape(x.shape)


class _UNetTrainFn(torch.autograd.Function):
    """ScoreUNet.forward with trainable parameters under autograd (the reference's training step,
    training_loop.py:372-378: `loss = pipeline.loss(net, x).mean(); fabric.backward(loss)`): the forward stashes on a
    training workspace, the backward is c2w_train_backward — input-gradient convs, weight-gradient GEMMs, bias /
    modulation / time-MLP sums — and hands autograd one gradient per parameter (views of one flat buffer), so gradient
    accumulation, DDP hooks and any torch optimiser work unchanged."""

    @staticmethod
    def forward(ctx, x, t_dev, net, forcing, *params):
        B, Cc, H, W = x.shape
        eng = net.engine(Cc, 1, H, W, x.device, train=True)
        if eng.max_windows < B:
            eng.bind(B)
        eng.set_forcing(forcing)  # stays set until this step's backward (map_forcing's gradients need the rows)
        out = eng.train_forward(x.detach().float().contiguous(), t_dev)
        token = object()
        eng._train_token = token
        ctx.eng, ctx.net, ctx.token, ctx.want_gin, ctx.dtype = eng, net, token, x.requires_grad, x.dtype
        ctx.n_params = len(params)
        ctx.needs = [p.requires_grad for p in params]
        return out.to(x.dtype).reshape(x.shape)

    @staticmethod
    def backward(ctx, gout):
        eng = ctx.eng
        if eng._train_token is not ctx.token:
            raise RuntimeError("another forward ran on this network's training workspace before this backward(): the "
                               "stashed activations are gone (one forward -> one backward per accumulation round)")
        direct = getattr(ctx.net, "_direct_grad", None)
        if direct is not None and direct.numel() == eng.param_total and direct.device == gout.device:
            # the optimiser's flat gradient buffer has the library's layout (optim.AdamW(direct_grads=True)): the kernels
            # ACCUMULATE into it in place and autograd gets nothing to add (no per-parameter hooks fire on this route)
            gin = eng.train_backward(gout.detach().float().contiguous(), direct, want_gin=ctx.want_gin, accumulate=True)
            eng._train_token = None
            eng.set_forcing(None)
            return (gin.to(ctx.dtype) if gin is not None else None, None, None, None, *([None] * ctx.n_params))
        flat = torch.empty(eng.param_total, dtype=torch.float32, device=gout.device)
        gin = eng.train_backward(gout.detach().float().contiguous(), flat, want_gin=ctx.want_gin)
        grads = []
        for (name, p), need in zip(ctx.net.state_dict(keep_vars=True).items(), ctx.needs):
            o, n = eng.layout[name]
            grads.append(flat[o:o + n].view_as(p) if need else None)
        eng._train_token = None
        eng.set_forcing(None)
        return (gin.to(ctx.dtype) if gin is not None else None, None, None, None, *grads)


class _UNetInputVJP(torch.autograd.Function):
    """ScoreUNet.forward under autograd: the backward is c2w_unet_vjp (forward recomputed with stashing + the
    input-gradient pass on tensor cores).  Gradients flow to x only."""

    VJP_WINDOWS = 8

    @staticmethod
    def forward(ctx, x, net, t):
        B, Cc, H, W = x.shape
        eng = net.engine(Cc, 1, H, W, x.device)
        ctx.save_for_backward(x)
        ctx.net, ctx.t = net, t
        out = eng.unet_forward(x.detach().float().contiguous(), t)
        return out.to(x.dtype).reshape(x.shape)

    @staticmethod
    def backward(ctx, gout):
        (x,) = ctx.saved_tensors
        B, Cc, H, W = x.shape
        eng = ctx.net.engine(Cc, 1, H, W, x.device, max_windows=min(B, _UNetInputVJP.VJP_WINDOWS), vjp=True)
        _, gin = eng.unet_vjp(x.detach().float().contiguous(), ctx.t, gout.detach().float().contiguous())
        return gin.to(x.dtype), None, None


def _arch_from_state_dict(sd) -> dict:
    """Architecture keyword arguments of the ScoreUNet that owns this state_dict (SURVEY.md §8(b) naming)."""
    nl = 1 + max(int(k.split(".")[2]) for k in sd if k.startswith("unet.heads."))
    ch, blocks, attn = [], [], []
    for lvl in range(nl):
        wkey = "unet.heads.0.weight" if lvl == 0 else f"unet.heads.{lvl}.0.weight"
        ch.append(int(sd[wkey].shape[0]))
        idxs = sorted({int(k.split(".")[3]) for k in sd if k.startswith(f"unet.descent.{lvl}.")})
        has_attn = any(k.startswith(f"unet.descent.{lvl}.") and ".qkv." in k for k in sd)
        if has_attn:
            attn.append(lvl)
            blocks.append(len(idxs) // 2)
        else:
            blocks.append(len(idxs))
    out = dict(channels=int(sd["unet.heads.0.weight"].shape[1]), embedding_dim=int(sd["map_layer1.weight"].shape[0]),
               hidden_channels=ch, hidden_blocks=blocks, attention_levels=attn)
    if "map_forcing.weight" in sd:
        out["forcing_dim"] = int(sd["map_forcing.weight"].shape[1])
    return out


def _validate_reference_tree(module: nn.Module) -> None:
    """A reference module tree (a snapshot's `ema`, or a live model.score.ScoreUNet) must be the network this package
    builds: SiLU activations (model/nn.py:156 `residue.2`) and zero padding; anything else would run silently wrong."""
    for name, m in module.named_modules():
        leaf = name.rsplit(".", 1)[-1]
        if ".residue" in name and leaf == "2" and not list(m.children()):
            if type(m).__name__ != "SiLU":
                raise NotImplementedError(f"{name} is {type(m).__name__}: only SiLU activations are built")
        pm = getattr(m, "padding_mode", None)
        if pm is not None and pm != "zeros":
            raise NotImplementedError(f"{name} has padding_mode={pm!r}: only zero padding is built")


def build_from_reference(module: nn.Module) -> ScoreUNet:
    """New ScoreUNet with the architecture and weights of a reference `model.score.ScoreUNet` instance."""
    _validate_reference_tree(module)
    net = ScoreUNet(activation=nn.SiLU, **_arch_from_state_dict(module.state_dict()))
    return net.from_reference(module)
