"""Host-side mirror of the reference model class for the CIST-GCN hot path.

``CISTGCN(arch, learn)`` keeps the reference constructor (models/CISTGCN/CISTGCN.py:491-557), its
``forward(x) -> (pred,)`` signature (:567-597), its class name (routed on by environment/test.py:98-99
and environment/model_loader.py:18) and its ``state_dict`` layout (SURVEY.md App. B) so checkpoints
load unchanged.  The module tree below is *only a parameter container*: no submodule has a forward.
The arithmetic runs in the hand-written sm_100a kernels behind the C-ABI (include/cistgcn_b200.h).

The tree is produced from a flat, ordered listing of leaves (``_Listing``) rather than nested layer
classes.  The listing follows the reference's creation order and re-initialisation passes, so that
``torch.manual_seed(s); CISTGCN(arch, learn)`` yields the same initial weights as the reference does
under the same seed (checked in tests/test_module_contract.py when /root/reference is mounted).
"""
from __future__ import annotations

import copy
import ctypes
import operator
import time
import warnings
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _cabi
from .pack import F, ModelGeometry, PackedModel, pack_state_dict


_TREE_EPOCH = [0]     # bumped by every attribute assignment on a container: cached tensor lists are rebuilt


class _Node(nn.Module):
    """Anonymous container; children are attached by (possibly numeric) name."""

    def __setattr__(self, name, value):
        _TREE_EPOCH[0] += 1
        super().__setattr__(name, value)

    def forward(self, *a, **k):  # pragma: no cover - containers are never called
        raise RuntimeError("cistgcn_b200: parameter container, not a callable layer")


class _Listing:
    """Ordered listing of parameter leaves + deferred init passes."""

    def __init__(self, root: nn.Module):
        self.root = root
        self.linears: Dict[str, List[nn.Linear]] = {}
        self.prelus: Dict[str, List[nn.PReLU]] = {}

    def _attach(self, path: str, leaf: nn.Module) -> nn.Module:
        node = self.root
        parts = path.split(".")
        for p in parts[:-1]:
            nxt = node._modules.get(p)
            if nxt is None:
                nxt = _Node()
                node.add_module(p, nxt)
            node = nxt
        node.add_module(parts[-1], leaf)
        return leaf

    def conv(self, path, cin, cout, k=(1, 1), bias=True):
        return self._attach(path, nn.Conv2d(cin, cout, kernel_size=k, bias=bias))

    def conv1d(self, path, cin, cout):
        return self._attach(path, nn.Conv1d(cin, cout, 1, bias=False))

    def bn2(self, path, n):
        return self._attach(path, nn.BatchNorm2d(n))

    def bn1(self, path, n):
        return self._attach(path, nn.BatchNorm1d(n))

    def prelu(self, path, n=1, group=None):
        m = self._attach(path, nn.PReLU(n))
        if group is not None:
            self.prelus.setdefault(group, []).append(m)
        return m

    def linear(self, path, cin, cout, group=None):
        m = self._attach(path, nn.Linear(cin, cout, bias=False))
        if group is not None:
            self.linears.setdefault(group, []).append(m)
        return m

    def static_adj(self, path, shape):
        # ConvTemporalGraphical with interpretable=False: U(-1/sqrt(size), 1/sqrt(size))  (CISTGCN.py:106-120)
        holder = _Node()
        holder.A = nn.Parameter(torch.empty(*shape))
        holder.A.data.uniform_(-1.0 / shape[1] ** 0.5, 1.0 / shape[1] ** 0.5)
        return self._attach(path, holder)


def _xavier_normal(convs, gain):
    for m in convs:
        nn.init.xavier_normal_(m.weight, gain=gain)


def _list_map2adj(L: _Listing, p: str, ci: int, T: int, V: int, domain: str):
    """Map2Adj leaves (CISTGCN.py:127-181); convs re-drawn xavier-normal(gain .05) per sub-sequence."""
    ch = ci // 2
    tc = [L.conv(f"{p}.time_compress.0", ci, ch, bias=False)]
    L.bn2(f"{p}.time_compress.1", ch)
    L.prelu(f"{p}.time_compress.2")
    tc.append(L.conv(f"{p}.time_compress.3", ch, ch, (T, 1), bias=False))
    L.bn2(f"{p}.time_compress.4", ch)
    tc.append(L.conv(f"{p}.time_compress.6", ch, T, bias=False))
    jc = [L.conv(f"{p}.joint_compress.0", ci, ch, bias=False)]
    L.bn2(f"{p}.joint_compress.1", ch)
    L.prelu(f"{p}.joint_compress.2")
    jc.append(L.conv(f"{p}.joint_compress.3", ch, ch, (1, V), bias=False))
    L.bn2(f"{p}.joint_compress.4", ch)
    jc.append(L.conv(f"{p}.joint_compress.6", ch, V, bias=False))
    n = V if domain == "space" else T
    ex = [L.conv(f"{p}.expansor.0", n, n, bias=False)]
    L.bn2(f"{p}.expansor.1", n)
    L.prelu(f"{p}.expansor.3")
    ex.append(L.conv(f"{p}.expansor.4", n, n, bias=False))
    for group in (tc, jc, ex):
        _xavier_normal(group, 0.05)


def _list_domain_layer(L: _Listing, p: str, ci: int, co: int, T: int, V: int, domain: str, interp: bool):
    """Domain_GCNN_layer leaves (CISTGCN.py:208-257)."""
    if not interp:
        L.static_adj(f"{p}.gcn", (T, V, V) if domain == "time" else (V, T, T))
    L.conv(f"{p}.tcn.0", ci, co)
    L.bn2(f"{p}.tcn.1", co)
    if ci != co:
        L.conv(f"{p}.residual.0", ci, co)
        L.bn2(f"{p}.residual.1", co)
    if interp:
        _list_map2adj(L, f"{p}.map_to_adj", ci, T, V, domain)
    L.prelu(f"{p}.prelu", group=p.split(".")[0])


def _list_dstd(L: _Listing, p: str, ci: int, co: int, T: int, V: int, interp: bool, reduction: int):
    """DSTD_GC leaves (CISTGCN.py:289-358)."""
    grp = p.split(".")[0]
    _list_domain_layer(L, f"{p}.dsgn", ci, co, T, V, "space", interp)
    _list_domain_layer(L, f"{p}.tsgn", ci, co, T, V, "time", interp)
    L.conv(f"{p}.compressor.0", 2 * co, co, bias=False)
    L.bn2(f"{p}.compressor.1", co)
    L.prelu(f"{p}.compressor.2", group=grp)
    hs = max(co // reduction, 1)
    L.linear(f"{p}.compressor.3.excitation.0", co, hs, group=grp)
    L.linear(f"{p}.compressor.3.excitation.2", hs, co, group=grp)
    if ci != co:
        L.conv(f"{p}.residual.0", ci, co)
        L.bn2(f"{p}.residual.1", co)
    L.bn2(f"{p}.global_norm", ci)
    cg = max(co // 2, 1)
    for k in ("conv_s", "conv_t"):
        L.conv(f"{p}.{k}.0", ci, cg, (T, 1), bias=False)
        L.bn2(f"{p}.{k}.1", cg)
        L.prelu(f"{p}.{k}.3", group=grp)
        L.conv(f"{p}.{k}.4", cg, co, (1, V), bias=False)
        L.bn2(f"{p}.{k}.5", co)
        L.prelu(f"{p}.{k}.7", group=grp)
    for k in ("map_s", "map_t"):
        L.linear(f"{p}.{k}.0", co + 2 + 2 * T, co, group=grp)
        L.bn1(f"{p}.{k}.1", co)
        L.prelu(f"{p}.{k}.3", group=grp)
        L.linear(f"{p}.{k}.4", co, co, group=grp)
    for k in ("prelu1", "prelu2"):
        L.bn2(f"{p}.{k}.0", co)
        L.prelu(f"{p}.{k}.1", group=grp)


def _list_context(L: _Listing, p: str, hid: int, Tout: int, V: int, reduction: int):
    """ContextLayer leaves (CISTGCN.py:394-461)."""
    for i, k in ((1, (1, 1)), (2, (Tout, 1)), (3, (1, 1))):
        L.conv(f"{p}.context_conv{i}.0", 1, hid, k, bias=False)
        L.bn2(f"{p}.context_conv{i}.1", hid)
        L.prelu(f"{p}.context_conv{i}.2")
    for i in (1, 2, 3):
        L.linear(f"{p}.map{i}.0", hid, Tout)
        L.prelu(f"{p}.map{i}.2")
    L.linear(f"{p}.fmap_s.0", 3 * Tout, V)
    L.bn1(f"{p}.fmap_s.1", V)
    L.linear(f"{p}.fmap_t.0", 3 * Tout, Tout)
    L.bn1(f"{p}.fmap_t.1", Tout)
    L.conv1d(f"{p}.norm_map.0", Tout, Tout)
    L.bn1(f"{p}.norm_map.1", Tout)
    L.prelu(f"{p}.norm_map.3")
    L.linear(f"{p}.norm_map.4.excitation.0", Tout, Tout // reduction)          # SE.py:10 (no max(.,1))
    L.linear(f"{p}.norm_map.4.excitation.2", Tout // reduction, Tout)
    L.conv1d(f"{p}.norm_map.5", Tout, Tout)
    L.bn1(f"{p}.norm_map.6", Tout)
    L.prelu(f"{p}.norm_map.8")
    L.conv(f"{p}.fconv.0", 1, 3, bias=False)
    L.bn2(f"{p}.fconv.1", 3)
    L.prelu(f"{p}.fconv.2")
    L.conv(f"{p}.fconv.3", 3, 3, bias=False)
    L.bn2(f"{p}.fconv.4", 3)
    L.prelu(f"{p}.fconv.5")
    hs = max(Tout // reduction, 1)
    L.linear(f"{p}.SE.excitation.0", Tout, hs)
    L.linear(f"{p}.SE.excitation.2", hs, Tout)


def _list_fpn(L: _Listing, p: str, cin: int, cout: int, k: int):
    """FPN leaves (CISTGCN.py:39-72)."""
    for i in (1, 2, 3):
        L.conv(f"{p}.block{i}.0", cin, cout, (k, k))
        L.bn2(f"{p}.block{i}.1", cout)
        L.prelu(f"{p}.block{i}.3", group="txcnns")
    L.conv(f"{p}.compress", 3 * cout + cin, cout)


class CISTGCN(nn.Module):
    """Drop-in for the reference ``CISTGCN`` (eval-mode inference on sm_100a).

    forward(x): x (B, input_n, joints, 3) float32 contiguous CUDA tensor -> 1-tuple (pred,) with pred
    (B, output_n, joints, 3).  Raises ValueError on wrong shape / dtype / device, RuntimeError if the
    CUDA extension is missing (there is no CPU or eager fallback)."""

    IN_CH = 10  # 3 pos + 3 acc + 3 vel + speed (CISTGCN.py:512)

    def __init__(self, arch, learn=None):
        super().__init__()
        mp = arch.model_params
        self.clipping = getattr(mp, "clipping", None)        # read and never used, like the reference (:493)
        self.n_input = int(mp.input_n)
        self.n_output = int(mp.output_n)
        self.n_joints = int(mp.joints)
        self.n_txcnn_layers = int(mp.n_txcnn_layers)
        self.txc_kernel_size = [mp.txc_kernel_size] * 2
        self.reduction = int(mp.reduction)
        self.hidden_dim = int(mp.hidden_dim)
        self.in_ch = self.IN_CH
        # The reference mutates the caller's lists (:516-517, :548); we copy instead, so the same
        # config object can construct any number of models.
        self._in_chain = [self.in_ch] + [int(c) for c in mp.input_gcn.model_complexity] + [self.in_ch]
        self._out_chain = [3] + [int(c) for c in mp.output_gcn.model_complexity]
        self._in_interp = [bool(v) for v in mp.input_gcn.interpretable][: len(self._in_chain) - 1]
        self._out_interp = [bool(v) for v in mp.output_gcn.interpretable][: len(self._out_chain) - 1]
        if len(self._in_interp) != len(self._in_chain) - 1 or len(self._out_interp) != len(self._out_chain) - 1:
            raise IndexError("interpretable list shorter than the block chain")
        self.dropout = float(getattr(learn, "dropout", 0.0)) if learn is not None else 0.0
        if mp.txc_kernel_size != 3:
            raise ValueError("cistgcn_b200: only txc_kernel_size=3 is implemented (all shipped configs)")

        T, V, To = self.n_input, self.n_joints, self.n_output
        L = _Listing(self)
        for name in ("st_gcnns", "txcnns", "se", "in_conv", "context_layer", "trans"):
            self.add_module(name, _Node())                   # registration order of the reference (:505-511)
        for i in range(len(self._in_chain) - 1):
            _list_dstd(L, f"st_gcnns.{i}", self._in_chain[i], self._in_chain[i + 1], T, V,
                       self._in_interp[i], self.reduction)
        _list_context(L, "context_layer", self.hidden_dim, To, V, self.reduction)
        _list_fpn(L, "txcnns.0", T, To, 3)
        for i in range(1, self.n_txcnn_layers):
            _list_fpn(L, f"txcnns.{i}", To, To, 3)
        self.add_module("prelus", _Node())
        for i in range(self.n_txcnn_layers):
            L.prelu(f"prelus.{i}")
        L.conv("dim_conversor.0", self.in_ch, 3, bias=False)
        L.bn2("dim_conversor.1", 3)
        L.prelu("dim_conversor.2")
        L.conv("dim_conversor.3", 3, 3, bias=False)
        L.prelu("dim_conversor.4", 3)
        self.add_module("st_gcnns_o", _Node())
        for i in range(len(self._out_chain) - 1):
            _list_dstd(L, f"st_gcnns_o.{i}", self._out_chain[i], self._out_chain[i + 1], V, To,
                       self._out_interp[i], self.reduction)
        # re-initialisation passes in the reference's order (:555-565): Linear -> xavier-uniform(.1)
        for grp in ("st_gcnns_o", "st_gcnns", "txcnns"):
            for m in L.linears.get(grp, []):
                nn.init.xavier_uniform_(m.weight, gain=0.1)
            for m in L.prelus.get(grp, []):
                nn.init.constant_(m.weight, 0.25)

        self._packed: Optional[PackedModel] = None
        self._packed_key = None
        self._tensor_cache = None
        self._tree_epoch = -1
        self.check_weights = False      # True: checksum the state on the device before every forward (synchronises)
        self.kernel_flags = 0           # CISTGCN_FLAG_* kernel choices, travels with every call (CP_FLAGS of the plan)
        self.act_dtype = torch.float32  # torch.bfloat16: cistgcn_forward_bf16 (bf16 activation storage + bf16 FPN tensor-core operands)
        self.pack_count = 0
        self.last_pack_ms = 0.0
        self._warned_fpn_fallback = False
        # load_state_dict(assign=True) swaps Parameter objects: drop the cached tensor list afterwards
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate_pack())
        self._taps_enabled = False
        self.last_taps: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------ geometry / packing
    def geometry(self) -> ModelGeometry:
        return ModelGeometry(input_n=self.n_input, output_n=self.n_output, joints=self.n_joints,
                             in_chain=list(self._in_chain), out_chain=list(self._out_chain),
                             in_interp=list(self._in_interp), out_interp=list(self._out_interp),
                             n_fpn=self.n_txcnn_layers, hidden_dim=self.hidden_dim,
                             reduction=self.reduction, feat_ch=self.in_ch)

    def _state_tensors(self):
        # state_dict() rebuilds 1 178 prefixed keys per call (~1 ms).  What is cached instead is the list of SLOTS
        # (owning module's _parameters / _buffers dict + name), read afresh on every call, so a replaced Parameter
        # object (`conv.weight = nn.Parameter(...)`) is seen.  The slot list itself is rebuilt whenever the module
        # tree could have changed: _apply (.to / .cuda), load_state_dict, attribute assignment on a container.
        if self._tensor_cache is None or self._tree_epoch != _TREE_EPOCH[0]:
            slots = []
            for mod in self.modules():
                slots += [(mod._parameters, n) for n, v in mod._parameters.items() if v is not None]
                slots += [(mod._buffers, n) for n, v in mod._buffers.items()
                          if v is not None and v.is_floating_point() and n not in mod._non_persistent_buffers_set]
            self._tensor_cache = slots
            self._tree_epoch = _TREE_EPOCH[0]
        return [d[n] for d, n in self._tensor_cache]

    def _invalidate_pack(self):
        self._tensor_cache = None
        self._packed = None

    def invalidate_pack(self):
        """Forget the packed device weights; the next forward re-packs from the current parameters.  Call this
        (or ``repack()``) after writes that PyTorch's version counters cannot see, i.e. through ``.data``
        (``p.data.copy_()``, EMA / weight averaging, ``gcn.A.data.uniform_()`` as in CISTGCN.py:120), unless
        ``check_weights`` is on."""
        self._invalidate_pack()
        return self

    def repack(self, device=None) -> PackedModel:
        """Unconditionally re-pack from the current parameters / buffers (see ``invalidate_pack``)."""
        self._invalidate_pack()
        return self.pack(device)

    def _apply(self, fn, *args, **kwargs):
        self._invalidate_pack()
        return super()._apply(fn, *args, **kwargs)

    def _state_key(self, device):
        # (storage address, version) per tensor: catches in-place updates through the autograd-visible API
        # (optimizer steps, load_state_dict, p.mul_()) and storage swaps (p.data = other).  Writes *through*
        # p.data keep both unchanged; those need invalidate_pack() or check_weights.
        ts = self._state_tensors()
        return (str(device),) + tuple((t.data_ptr(), t._version) for t in ts)

    def _state_checksum(self):
        """Order-sensitive checksum of every floating-point state entry, computed on the tensors' device
        (check_weights mode only: the comparison synchronises the stream)."""
        ts = self._state_tensors()
        flat = torch.cat([t.detach().reshape(-1).to(torch.float32) for t in ts])
        bits = flat.view(torch.int32).to(torch.int64)
        idx = torch.arange(1, bits.numel() + 1, device=bits.device, dtype=torch.int64)
        return int(((bits * (idx % 65521 + 1)).sum() ^ bits.sum()).item())

    def pack(self, device=None) -> PackedModel:
        """Fold eval-mode BatchNorm + biases and lay the weights out in one device blob
        (re-run automatically whenever a parameter / buffer changed since the last forward)."""
        device = torch.device(device) if device is not None else next(self.parameters()).device
        key = self._state_key(device)
        if self.check_weights:
            key = key + (self._state_checksum(),)
        if self._packed is None or key != self._packed_key:
            t0 = time.perf_counter()
            sd = {k: v.detach() for k, v in self.state_dict().items()}
            self._packed = pack_state_dict(sd, self.geometry(), device)
            self._packed_key = key
            self.pack_count += 1
            self.last_pack_ms = 1e3 * (time.perf_counter() - t0)
            if not self._packed.fpn_tc and not self._warned_fpn_fallback:
                self._warned_fpn_fallback = True
                warnings.warn("cistgcn_b200: the FPN stack runs on the FP32-FMA kernel for these weights "
                              f"({self._packed.fpn_tc_reason}); the tcgen05 kernel is ~2.5x faster", RuntimeWarning)
        return self._packed

    def enable_taps(self, on: bool = True):
        """Interpretability outputs (Adj, w1, w2, ContextLayer maps; environment/test.py:146-157)
        are written to ``self.last_taps`` by the next forward when enabled."""
        self._taps_enabled = bool(on)
        return self

    # ------------------------------------------------------------------ forward
    def _check_input(self, x):
        if not isinstance(x, torch.Tensor):
            raise ValueError("cistgcn_b200: x must be a torch.Tensor")
        if x.dim() != 4 or x.shape[1] != self.n_input or x.shape[2] != self.n_joints or x.shape[3] != 3:
            raise ValueError(f"cistgcn_b200: expected x of shape (B, {self.n_input}, {self.n_joints}, 3), "
                             f"got {tuple(x.shape)}")
        if x.dtype != torch.float32:
            raise ValueError(f"cistgcn_b200: expected float32 input, got {x.dtype}")
        if not x.is_cuda:
            raise ValueError("cistgcn_b200: input must live on a CUDA device (no CPU fallback exists)")

    def forward(self, x) -> Tuple[torch.Tensor]:
        pred, _ = self._run(x, None)
        return pred,                                         # 1-tuple, like CISTGCN.py:597

    def forward_mpjpe(self, x, target, groups=None, n_groups=None):
        """Forward + fused MPJPE partial sums.  Returns (pred, frame_sums) where frame_sums is a
        float64 (output_n,) tensor: sum over samples and joints of ||pred - target||_2 per frame.
        mpjpe(reduce_axis=[]) = frame_sums.sum() / (B*T*V); (0,2) = frame_sums / (B*V).

        With ``groups`` (a (B,) integer tensor of per-sample group ids, e.g. the action of every window) and
        ``n_groups``: returns (pred, sums, counts) instead, sums a float64 (n_groups, output_n) tensor of the same frame
        sums per group and counts an int64 (n_groups,) tensor of samples per group, so group g's per-frame MPJPE is
        sums[g] / (counts[g] * joints).  ``pred`` is ``forward(x)[0]``; the sums come from one extra pass over pred and
        target.  A CPU ``groups`` tensor is range-checked here (ValueError); ids of a CUDA ``groups`` tensor are not
        (that would synchronise): samples whose id is outside [0, n_groups) are left out of sums and counts."""
        if target.shape != (x.shape[0], self.n_output, self.n_joints, 3) or target.dtype != torch.float32 \
                or target.device != x.device:
            raise ValueError("cistgcn_b200: target must be (B, output_n, joints, 3) float32 on x's device")
        if groups is None and n_groups is None:
            return self._run(x, target.contiguous())
        groups = self._check_groups(groups, n_groups, x)
        pred = self._run(x, None)[0]
        return (pred,) + self._grouped_mpjpe(pred, target, groups, n_groups)

    def rollout(self, x, horizon) -> torch.Tensor:
        """Autoregressive forecast past output_n, eval mode only: ceil(horizon / output_n) forwards, each fed the last
        input_n frames of the previous prediction (the first one x).  Returns (B, horizon, joints, 3) = the concatenated
        predictions cut to `horizon`, bit-identical to that loop over ``model(...)`` at the same batch size."""
        return self._rollout(x, horizon, None)[0]

    def rollout_mpjpe(self, x, target, groups=None, n_groups=None):
        """``rollout(x, target.shape[1])`` + fused MPJPE partial sums: returns (pred, frame_sums), frame_sums a float64
        (horizon,) tensor with the meaning of ``forward_mpjpe``'s, so it plugs into ``dist.sharded_eval_mpjpe``.
        With ``groups`` / ``n_groups``: returns (pred, sums (n_groups, horizon), counts (n_groups,)) as ``forward_mpjpe``
        does, so it plugs into ``dist.sharded_eval_grouped``."""
        if not isinstance(target, torch.Tensor) or target.dim() != 4:
            raise ValueError("cistgcn_b200: target must be a (B, horizon, joints, 3) tensor")
        if groups is None and n_groups is None:
            return self._rollout(x, target.shape[1], target)
        B = x.shape[0] if isinstance(x, torch.Tensor) else None
        if target.shape != (B, target.shape[1], self.n_joints, 3) or target.dtype != torch.float32 \
                or target.device != getattr(x, "device", None):
            raise ValueError("cistgcn_b200: target must be (B, horizon, joints, 3) float32 on x's device")
        groups = self._check_groups(groups, n_groups, x)
        pred = self._rollout(x, target.shape[1], None)[0]
        return (pred,) + self._grouped_mpjpe(pred, target, groups, n_groups)

    def _check_groups(self, groups, n_groups, x):
        """Validates per-sample group ids before the library is reached; returns them as int32 on x's device."""
        if isinstance(n_groups, bool):
            n_groups = None
        try:
            n_groups = operator.index(n_groups)
        except TypeError:
            n_groups = None
        if n_groups is None or not 1 <= n_groups < 2**31:
            raise ValueError("cistgcn_b200: n_groups must be an integer >= 1 when groups are given")
        B = x.shape[0] if isinstance(x, torch.Tensor) else None
        if not isinstance(groups, torch.Tensor) or groups.shape != (B,) or groups.is_floating_point() \
                or groups.is_complex() or groups.dtype == torch.bool:
            raise ValueError("cistgcn_b200: groups must be a (B,) integer tensor of group ids")
        if groups.is_cuda:
            if groups.device != x.device:
                raise ValueError("cistgcn_b200: groups must live on the CPU or on x's device")
        elif groups.numel() and (int(groups.min()) < 0 or int(groups.max()) >= n_groups):
            raise ValueError(f"cistgcn_b200: group ids must lie in [0, {n_groups})")
        return groups.to(x.device, torch.int32).contiguous()

    def _grouped_mpjpe(self, pred, target, groups, n_groups):
        """(sums (G, T) float64, counts (G,) int64) of cistgcn_mpjpe_grouped_f32 over pred / target."""
        B, T, V, _ = pred.shape
        sums = torch.zeros(n_groups, T, device=pred.device, dtype=torch.float64)
        counts = torch.zeros(n_groups, device=pred.device, dtype=torch.int64)
        if B == 0:
            return sums, counts
        lib = _cabi.lib()
        pred_c, target = pred.detach().contiguous(), target.contiguous()
        stream = torch.cuda.current_stream(pred.device).cuda_stream
        with torch.cuda.device(pred.device):
            rc = lib.cistgcn_mpjpe_grouped_f32(pred_c.data_ptr(), target.data_ptr(), groups.data_ptr(), n_groups, B, T, V,
                                               sums.data_ptr(), counts.data_ptr(), stream)
        _cabi.check(rc, "cistgcn_mpjpe_grouped_f32")
        return sums, counts

    def _rollout(self, x, horizon, target):
        if self.training:
            raise ValueError("cistgcn_b200: rollout runs in eval mode only (call model.eval())")
        if torch.is_grad_enabled() and getattr(x, "requires_grad", False):
            raise ValueError("cistgcn_b200: rollout is not differentiable; loop forward() for input gradients")
        if isinstance(horizon, bool):
            horizon = None
        try:
            horizon = operator.index(horizon)
        except TypeError:
            horizon = None
        if horizon is None or not 1 <= horizon < 2**31:
            raise ValueError("cistgcn_b200: horizon must be an integer >= 1")
        if target is not None:
            B = x.shape[0] if isinstance(x, torch.Tensor) else None
            if target.shape != (B, horizon, self.n_joints, 3) or target.dtype != torch.float32 \
                    or target.device != getattr(x, "device", None):
                raise ValueError("cistgcn_b200: target must be (B, horizon, joints, 3) float32 on x's device")
            target = target.contiguous()
        self._check_input(x)
        lib = _cabi.lib()
        x = x.contiguous()
        B = x.shape[0]
        packed = self.pack(x.device)
        packed.plan_c[F["CP_FLAGS"]] = int(self.kernel_flags)
        out = torch.empty(B, horizon, self.n_joints, 3, device=x.device, dtype=torch.float32)
        sums = torch.zeros(horizon, device=x.device, dtype=torch.float64) if target is not None else None
        if B == 0:
            return out, sums
        workspace = torch.empty(lib.cistgcn_rollout_workspace_bytes(packed.plan_c, B), device=x.device, dtype=torch.uint8)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        name = "cistgcn_rollout_bf16" if self.act_dtype == torch.bfloat16 else "cistgcn_rollout_f32"
        with torch.cuda.device(x.device):
            rc = getattr(lib, name)(packed.plan_c, len(packed.plan), packed.blob.data_ptr(), x.data_ptr(), horizon,
                                    out.data_ptr(), target.data_ptr() if target is not None else None,
                                    sums.data_ptr() if sums is not None else None,
                                    workspace.data_ptr(), workspace.numel(), B, stream)
        _cabi.check(rc, name)
        return out, sums

    def _run(self, x, target):
        self._check_input(x)
        if self.training or (torch.is_grad_enabled() and x.requires_grad):
            return self._run_differentiable(x, target)
        lib = _cabi.lib()                                    # raises loudly if the extension is missing
        x = x.contiguous()
        B = x.shape[0]
        packed = self.pack(x.device)
        packed.plan_c[F["CP_FLAGS"]] = int(self.kernel_flags)
        pred = torch.empty(B, self.n_output, self.n_joints, 3, device=x.device, dtype=torch.float32)
        if B == 0:
            return pred, torch.zeros(self.n_output, device=x.device, dtype=torch.float64)
        # per-call scratch from the caching allocator: stream-ordered, so two forwards of one module on different
        # streams never share a buffer (a cached per-module buffer would race)
        need = lib.cistgcn_workspace_bytes(packed.plan_c, B)
        workspace = torch.empty(need, device=x.device, dtype=torch.uint8)
        sums = None
        if target is not None:
            sums = torch.zeros(self.n_output, device=x.device, dtype=torch.float64)
        taps_struct, holders = None, {}
        if self._taps_enabled:
            taps_struct, holders = _cabi.make_taps(self.geometry(), B, x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        with torch.cuda.device(x.device):
            entry = lib.cistgcn_forward_bf16 if self.act_dtype == torch.bfloat16 else lib.cistgcn_forward_f32
            rc = entry(packed.plan_c, len(packed.plan), packed.blob.data_ptr(),
                                         x.data_ptr(), pred.data_ptr(),
                                         target.data_ptr() if target is not None else None,
                                         sums.data_ptr() if sums is not None else None,
                                         workspace.data_ptr(), workspace.numel(), B,
                                         taps_struct, stream)
        _cabi.check(rc, "cistgcn_forward_bf16" if self.act_dtype == torch.bfloat16 else "cistgcn_forward_f32")
        if self._taps_enabled:
            self.last_taps = holders
            self._publish_taps(holders)
        return pred, sums

    # ------------------------------------------------------------------ differentiable path (train mode / input gradients)
    def _diff_state(self):
        """(FlatParams, DiffGraph) of the layer-by-layer differentiable path (cistgcn_b200/train.py), rebuilt when the
        parameters were moved (.to / .cuda replaces their storage)."""
        from .train import DiffGraph, FlatParams
        st = getattr(self, "_diff", None)
        first = next(self.parameters())
        if st is None or st[0].flat.device != first.device or first.data_ptr() != st[0].flat.data_ptr():
            flat = FlatParams(self)
            st = (flat, DiffGraph(self, flat), torch.zeros(flat.numel, device=flat.device),
                  torch.zeros(1, device=flat.device, requires_grad=True))
            object.__setattr__(self, "_diff", st)
        return st

    def _run_differentiable(self, x, target):
        """Train-mode forward (environment/train.py:59: batch-statistics BatchNorm, dropout, parameter gradients through
        autograd) and eval-mode forward with gradients w.r.t. the input (environment/adversarial_attacks.py:184, 422,
        495-511).  Runs the hand-written layer kernels of csrc/train_ops.cu behind a torch.autograd.Function."""
        flat, graph, fresh, anchor = self._diff_state()
        pred = _DiffForward.apply(self, x, anchor)
        if target is None:
            return pred, None
        from .losses import mpjpe
        with torch.no_grad():
            B, V = x.shape[0], self.n_joints
            sums = mpjpe(pred.detach(), target, reduce_axis=(0, 2)).double() * (B * V)
        return pred, sums

    def _publish_taps(self, taps: Dict[str, torch.Tensor]):
        """Expose the interpretability outputs as attributes on the same dotted paths the reference sets
        in its forward (CISTGCN.py:262, 381-382, 469-473), so `getattr`-walking callers such as
        environment/test.py:146-157 (predict.yaml:162-195) keep working."""
        taps = dict(taps)
        if "context_layer.joints" in taps and "context_layer.displacements" in taps:      # CISTGCN.py:471
            taps["context_layer.seq_joints"] = taps["context_layer.displacements"].unsqueeze(2) * \
                taps["context_layer.joints"].unsqueeze(1)
        for key, value in taps.items():
            node = self
            parts = key.split(".")
            try:
                for k in parts[:-1]:
                    node = getattr(node, k)
            except AttributeError:
                continue
            object.__setattr__(node, parts[-1], value)
            if parts[-1] == "Adj":                           # the reference also aliases it as gcn.A (CISTGCN.py:264)
                gcn = node._modules.get("gcn")
                if gcn is None:
                    gcn = _Node()
                    object.__setattr__(node, "gcn", gcn)     # plain attribute: keeps state_dict / module tree unchanged
                if "A" not in gcn._parameters:
                    object.__setattr__(gcn, "A", value)


class _DiffForward(torch.autograd.Function):
    """autograd bridge of the differentiable path.  Parameter gradients do not travel through autograd's return values
    (1 018 tensors): the backward kernels write them into one flat buffer and ``.grad`` of every Parameter is a view of
    the flat accumulator, so `loss.backward(); optimizer.step()` of environment/train.py:80-106 works unchanged."""

    @staticmethod
    def forward(ctx, model, x, anchor):
        flat, graph, fresh, _ = model._diff_state()
        training = model.training
        want_dx = bool(x.requires_grad) and torch.is_grad_enabled()
        with torch.no_grad():
            pred = graph.forward(x.detach(), training=training, input_grad=want_dx, param_grads=training)
        ctx.model, ctx.training, ctx.want_dx = model, training, want_dx
        if model._taps_enabled:
            model.last_taps = dict(graph.taps)
            model._publish_taps(model.last_taps)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        model = ctx.model
        flat, graph, fresh, _ = model._diff_state()
        lib = graph.lib
        with torch.no_grad():
            graph.grad_target = fresh if ctx.training else None
            dx = graph.backward(dpred.contiguous())
            if ctx.training:
                params = list(model.parameters())
                have = [p.grad is not None for p in params]
                stream = torch.cuda.current_stream(flat.device).cuda_stream if flat.flat.is_cuda else None
                ours = all(p.grad is None or p.grad.data_ptr() == flat.grad.data_ptr() + 4 * flat.offsets[n][0]
                           for (n, _), p in zip(model.named_parameters(), params))
                if ours:
                    # accumulate (or set, after zero_grad(set_to_none=True)) in ONE flat launch
                    beta = 1.0 if any(have) else 0.0
                    _cabi.check(lib.cistgcn_axpby(ctypes.c_float(1.0), fresh.data_ptr(), ctypes.c_float(beta), flat.grad.data_ptr(),
                                                  flat.numel, stream), "axpby", lib)
                    for (n, _), p in zip(model.named_parameters(), params):
                        if p.grad is None:
                            p.grad = flat.grad_view(n)
                else:                                                    # foreign .grad tensors: per-parameter accumulation
                    for (n, _), p in zip(model.named_parameters(), params):
                        off, k, shape = flat.offsets[n]
                        g = fresh[off: off + k].view(shape)
                        p.grad = g.clone() if p.grad is None else p.grad + g
                model._invalidate_pack()
        return None, (dx if ctx.want_dx else None), None


def choose_net(architecture: str, opt):
    """models/choose_net.py:4-11 equivalent: registry name -> model on the current CUDA device."""
    if architecture not in ("CISTGCN_0", "CISTGCN_eval"):
        raise ValueError(f"unknown architecture {architecture!r}")
    return CISTGCN(copy.deepcopy(opt.architecture_config), opt.learning_config).cuda()
