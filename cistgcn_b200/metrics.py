"""Fused evaluation metrics on the GPU (reference: environment/test.py:65-94 ``Metrics.compute`` and :125-129 the
scatter of the predicted joints into the full skeleton; losses/losses.py).  One kernel (csrc/eval_metrics.cu) reads the
prediction and the target once and accumulates every metric per output frame; the reference launches ~10 chains of
ATen kernels with a ``.cpu()`` sync each."""
from __future__ import annotations

import operator
from typing import Dict, Optional, Sequence

import torch

from . import _cabi
from .pack import F as _F

METRICS = ("mpjpe", "pa_mpjpe", "n_mpjpe", "velocity", "bone_length", "weighted0", "weighted1")
# loaders/h36m_motion_3d.py:55-56: joints of the 22-joint prediction that are copied onto ignored joints of the 32-joint skeleton
H36M_DIM_REPEAT_22 = (9, 9, 14, 16, 19, 21)
H36M_DIM_REPEAT_32 = (16, 24, 20, 23, 28, 31)


def source_map(n_full: int, dim_used: Sequence[int], dim_repeat_full: Sequence[int] = (), dim_repeat_used: Sequence[int] = ()) -> torch.Tensor:
    """[n_full] int32 table: which predicted joint lands on each joint of the full skeleton (-1: keep the target's joint).
    Mirrors ``mygt[:, :, dim_used] = outputs; mygt[:, :, dim_repeat_32] = outputs[:, :, dim_repeat_22]`` (test.py:125-129)."""
    m = torch.full((n_full,), -1, dtype=torch.int32)
    for k, j in enumerate(dim_used):
        m[j] = k
    for j, k in zip(dim_repeat_full, dim_repeat_used):
        m[j] = k
    return m


class EvalMetrics:
    """Accumulates the evaluation metrics of ``Metrics.compute`` over batches, entirely on the device, optionally split
    into ``n_groups`` groups (one per action or sub-dataset).

    compute(outputs, target, weights0=None, weights1=None, groups=None): outputs (B, To, Vu, 3) from the model, target
    (B, To, Vf, 3), groups an optional (B,) integer tensor of per-sample group ids in [0, n_groups) (default: group 0).
    values(): dict name -> float32 (To,) tensor = the reference's ``reduce_axis=(0, 2)`` means over all groups
    (velocity: To - 1 entries).  values_by_group(): the same per group, (n_groups, To) (velocity (n_groups, To - 1)), NaN
    rows for groups without samples.  counts: int64 (n_groups,) samples per group.  all_reduce(): sums and counts over
    the ranks of a process group, for sharded evaluation.

    Ids of a CUDA ``groups`` tensor are not checked in compute() (that would synchronise); samples with ids outside
    [0, n_groups) are left out of the sums and counts, and values() / values_by_group() then raise ValueError."""

    def __init__(self, output_n: int, src_map: torch.Tensor, bones: Optional[Sequence[Sequence[int]]] = None, device="cuda",
                 n_groups: int = 1):
        self.To = int(output_n)
        try:
            self.n_groups = operator.index(n_groups) if not isinstance(n_groups, bool) else 0
        except TypeError:
            self.n_groups = 0
        if self.n_groups < 1:
            raise ValueError("EvalMetrics: n_groups must be an integer >= 1")
        self.device = torch.device(device)
        self.src_map = src_map.to(self.device, torch.int32).contiguous()
        self.Vf = int(src_map.numel())
        self.bones = torch.tensor(bones, dtype=torch.int32, device=self.device).contiguous() if bones is not None and len(bones) else None
        self.n_bones = 0 if self.bones is None else int(self.bones.shape[0])
        self.group_sums = torch.zeros(self.n_groups, len(METRICS), self.To, dtype=torch.float64, device=self.device)
        self.counts = torch.zeros(self.n_groups, dtype=torch.int64, device=self.device)
        self.count = 0

    @property
    def sums(self) -> torch.Tensor:
        """(len(METRICS), To) float64 metric sums over all groups."""
        return self.group_sums[0] if self.n_groups == 1 else self.group_sums.sum(0)

    def compute(self, outputs: torch.Tensor, target: torch.Tensor, weights0: Optional[torch.Tensor] = None,
                weights1: Optional[torch.Tensor] = None, want_assembled: bool = False,
                groups: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        if outputs.dim() != 4 or target.dim() != 4 or outputs.shape[:2] != target.shape[:2] or target.shape[2] != self.Vf \
                or outputs.shape[1] != self.To or outputs.shape[3] != 3 or target.shape[3] != 3:
            raise ValueError("EvalMetrics.compute: outputs (B, To, Vu, 3) / target (B, To, Vf, 3) expected")
        B = outputs.shape[0]
        if groups is not None:
            if not isinstance(groups, torch.Tensor) or groups.shape != (B,) or groups.is_floating_point() \
                    or groups.is_complex() or groups.dtype == torch.bool:
                raise ValueError("EvalMetrics.compute: groups must be a (B,) integer tensor of group ids")
            if groups.is_cuda:
                if groups.device != outputs.device:
                    raise ValueError("EvalMetrics.compute: groups must live on the CPU or on the outputs' device")
            elif groups.numel() and (int(groups.min()) < 0 or int(groups.max()) >= self.n_groups):
                raise ValueError(f"EvalMetrics.compute: group ids must lie in [0, {self.n_groups})")
        if not outputs.is_cuda or outputs.dtype != torch.float32 or target.dtype != torch.float32:
            raise ValueError("EvalMetrics.compute: float32 CUDA tensors required (no CPU fallback)")
        if groups is not None:
            groups = groups.to(outputs.device, torch.int32).contiguous()
        if B == 0:                  # nothing to accumulate (and empty tensors have no data pointer to hand to the library)
            return torch.empty_like(target) if want_assembled else None
        lib = _cabi.lib()
        o, t = outputs.detach().contiguous(), target.detach().contiguous()
        Vu = o.shape[2]
        w0 = weights0.contiguous() if weights0 is not None else None
        w1 = weights1.contiguous() if weights1 is not None else None
        asm = torch.empty_like(t) if want_assembled else None
        stream = torch.cuda.current_stream(o.device).cuda_stream
        bones = self.bones.data_ptr() if self.bones is not None else None
        w0p, w1p = (w0.data_ptr() if w0 is not None else None), (w1.data_ptr() if w1 is not None else None)
        asmp = asm.data_ptr() if asm is not None else None
        if self.n_groups == 1 and groups is None and self.To <= 32:
            # the ungrouped kernel: the numbers of earlier releases, bit for bit
            with torch.cuda.device(o.device):
                rc = lib.cistgcn_eval_metrics_f32(o.data_ptr(), t.data_ptr(), self.src_map.data_ptr(), bones, self.n_bones,
                                                  w0p, w1p, asmp, self.group_sums.data_ptr(), B, self.To, Vu, self.Vf, stream)
            _cabi.check(rc, "cistgcn_eval_metrics_f32")
            self.counts += B
        else:
            with torch.cuda.device(o.device):
                rc = lib.cistgcn_eval_metrics_grouped_f32(o.data_ptr(), t.data_ptr(),
                                                          groups.data_ptr() if groups is not None else None, self.n_groups,
                                                          self.src_map.data_ptr(), bones, self.n_bones, w0p, w1p, asmp,
                                                          self.group_sums.data_ptr(), self.counts.data_ptr(), B, self.To, Vu,
                                                          self.Vf, stream)
            _cabi.check(rc, "cistgcn_eval_metrics_grouped_f32")
        self.count += B
        return asm

    def _check_counts(self) -> torch.Tensor:
        counts = self.counts.cpu()
        if int(counts.sum()) < self.count:
            raise ValueError(f"EvalMetrics: {self.count - int(counts.sum())} of {self.count} samples had group ids outside "
                             f"[0, {self.n_groups}) and were not accumulated")
        return counts

    def values(self) -> Dict[str, torch.Tensor]:
        self._check_counts()
        sums = self.sums
        out = {}
        for i, name in enumerate(METRICS):
            den = self.count * (self.n_bones if name == "bone_length" else self.Vf)
            v = (sums[i] / max(den, 1)).to(torch.float32)
            out[name] = v[:-1] if name == "velocity" else v
        return out

    def values_by_group(self) -> Dict[str, torch.Tensor]:
        counts = self._check_counts().to(self.device, torch.float64)[:, None]
        out = {}
        for i, name in enumerate(METRICS):
            den = counts * (self.n_bones if name == "bone_length" else self.Vf)
            v = torch.where(counts > 0, self.group_sums[:, i] / den.clamp(min=1), float("nan")).to(torch.float32)
            out[name] = v[:, :-1] if name == "velocity" else v
        return out

    def all_reduce(self, group=None) -> "EvalMetrics":
        """Sums the metric sums, the per-group counts and the sample count over the ranks of `group` in ONE
        ``torch.distributed.all_reduce`` (NCCL for CUDA accumulators), after which values() / values_by_group() are the
        global results on every rank."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return self
        n = self.group_sums.numel()
        buf = torch.cat([self.group_sums.reshape(-1), self.counts.to(torch.float64),
                         self.group_sums.new_tensor([float(self.count)])])
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        self.group_sums.copy_(buf[:n].view_as(self.group_sums))
        self.counts.copy_(buf[n:n + self.n_groups].round().to(torch.int64))
        self.count = int(round(float(buf[-1])))
        return self
