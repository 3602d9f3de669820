"""Training slices resident on the device (SURVEY section 8(f) N3).

The reference keeps a Python list of per-index tensor slices and feeds it through a
``torch.utils.data.DataLoader`` (dataset_management.py:17-67); at ~1e9 samples/s that loader is the
bottleneck.  Here every trajectory is sliced once with the same index arithmetic
(``add_slices_from_trajectory``, dataset_management.py:43-59) into two dense device tensors, and an
epoch is one on-device permutation plus gathers, so batches never touch the host.

On-disk format of the reference: one ``torch.save``d ``(T, n_x)`` float64 tensor per trajectory,
named ``<index>.pt`` (file_utils.py:16,168-176).
"""
import os
from dataclasses import dataclass
from typing import Iterator, List, Optional, Tuple

import torch
from torch import Tensor


@dataclass
class TrajectorySliceConfig:
    """Same fields and checks as the reference's ``data_config.TrajectorySliceConfig`` (data_config.py:5-19)."""
    t_skip: int = 0
    t_history: int = 1
    t_prediction: int = 1

    def __post_init__(self):
        assert self.t_skip + 1 >= self.t_history
        assert self.t_history >= 1
        assert self.t_prediction >= 1


class DeviceTrajectorySliceDataset:
    """(previous states, future states) transition pairs of a set of trajectories, as two dense tensors
    ``(N, t_history, n_x)`` and ``(N, t_prediction, n_x)`` on ``device``; indexable like the reference's
    ``TrajectorySliceDataset`` and iterable in shuffled device batches."""

    def __init__(self, config: TrajectorySliceConfig, device: torch.device = torch.device('cpu'),
                 dtype: torch.dtype = torch.float64) -> None:
        self.config = config
        self.device = torch.device(device)
        self.dtype = dtype
        self._previous: List[Tensor] = []
        self._future: List[Tensor] = []
        self._dense: Optional[Tuple[Tensor, Tensor]] = None
        self._cost: Optional[Tensor] = None      # (N,) int32 per-slice cost hint (last epoch's Newton counts)
        self._usol: Optional[Tensor] = None      # (N, 6) cube / (N, 7) elbow: last epoch's QP optima, next epoch's warm starts

    def add_slices_from_trajectory(self, trajectory: Tensor) -> None:
        """``trajectory``: (T, n_x).  Slice i predicts from time index ``t_skip + i``
        (dataset_management.py:49-59): previous = traj[idx+1-t_history : idx+1], future = traj[idx+1 : idx+1+t_prediction]."""
        cfg = self.config
        T = trajectory.shape[0]
        first, last = cfg.t_skip, T - cfg.t_prediction
        assert first <= last
        if last == first:
            return
        traj = trajectory.to(device=self.device, dtype=self.dtype)
        # unfold gives (windows, n_x, window) views: window w starts at time index w
        prev = traj.unfold(0, cfg.t_history, 1)[first + 1 - cfg.t_history:last + 1 - cfg.t_history]
        fut = traj.unfold(0, cfg.t_prediction, 1)[first + 1:last + 1]
        self._previous.append(prev.transpose(1, 2).contiguous())
        self._future.append(fut.transpose(1, 2).contiguous())
        self._dense = None
        self._cost = None
        self._usol = None

    def add_trajectories_from_directory(self, trajectory_dir: str, indices: Optional[List[int]] = None) -> int:
        """Loads ``<index>.pt`` trajectories (all whole-number-named files when ``indices`` is None)."""
        if indices is None:
            indices = sorted(int(f[:-3]) for f in os.listdir(trajectory_dir) if f.endswith('.pt') and f[:-3].isdigit())
        for i in indices:
            self.add_slices_from_trajectory(torch.load(os.path.join(trajectory_dir, f'{i}.pt'), map_location='cpu'))
        return len(indices)

    def tensors(self) -> Tuple[Tensor, Tensor]:
        """(previous (N, t_history, n_x), future (N, t_prediction, n_x)), device-resident."""
        if self._dense is None:
            if not self._previous:
                raise ValueError('empty dataset')
            self._dense = (torch.cat(self._previous, 0), torch.cat(self._future, 0))
            self._previous, self._future = [self._dense[0]], [self._dense[1]]
        return self._dense

    def __len__(self) -> int:
        return sum(p.shape[0] for p in self._previous)

    def __getitem__(self, idx) -> Tuple[Tensor, Tensor]:
        prev, fut = self.tensors()
        return prev[idx], fut[idx]

    # -- cost hints -------------------------------------------------------------------------------------
    # The loss kernel's run time per sample is its Newton count (0 for free flight, up to ~45), and training
    # revisits the same slices every epoch while the parameters move slowly: last epoch's counts predict this
    # epoch's.  A batch handed to the kernel in order of decreasing cost (with ``system.dynamic_schedule``)
    # starts its longest solves first and ends on the cheap samples, which removes the serial tail of the
    # launch (DESIGN.md section 4).  The hint only orders the batch; results do not depend on it.
    def update_costs(self, indices: Optional[Tensor], newton_iters: Tensor) -> None:
        """Records ``BatchLoss.newton_iters`` of the slices ``indices`` (None: all slices, in storage order)."""
        n = len(self)
        if self._cost is None:
            self._cost = torch.zeros(n, dtype=torch.int32, device=self.device)
        it = newton_iters.reshape(-1).to(device=self.device, dtype=torch.int32)
        if indices is None:
            assert it.numel() == n
            self._cost.copy_(it)
        else:
            self._cost[indices.reshape(-1).to(self.device)] = it

    def update_solutions(self, indices: Optional[Tensor], qp_solution: Tensor) -> None:
        """Records ``BatchLoss.qp_solution`` (the cone QPs' optima) of the slices ``indices`` (None: all).  The width of a
        solution (6 for the cube, 7 for the elbow) is taken from the first one recorded; a later one of another width
        raises."""
        n = len(self)
        width = qp_solution.shape[-1]
        if self._usol is None:
            self._usol = torch.zeros((n, width), dtype=self.dtype, device=self.device)
        elif width != self._usol.shape[1]:
            raise ValueError(f'QP solutions of width {width}, but this data set records width {self._usol.shape[1]}')
        u = qp_solution.reshape(-1, width).to(device=self.device, dtype=self.dtype)
        if indices is None:
            assert u.shape[0] == n
            self._usol.copy_(u)
        else:
            self._usol[indices.reshape(-1).to(self.device)] = u

    def warm_start(self, indices: Optional[Tensor] = None) -> Optional[Tensor]:
        """(len(indices), width) warm starts for ``system.qp_warm_start`` (zeros for slices not recorded yet); None if no
        solution has been recorded yet."""
        if self._usol is None:
            return None
        return self._usol if indices is None else self._usol.index_select(0, indices.reshape(-1).to(self.device))

    def cost_order(self, indices: Optional[Tensor] = None, rank: int = 0, world: int = 1) -> Tensor:
        """Slice indices (of ``indices``, default all) by decreasing cost hint (stable), dealt round-robin to the
        ranks of a data-parallel step so that every shard is itself ordered and equally expensive."""
        if indices is None:
            indices = torch.arange(len(self), device=self.device)
        if self._cost is not None:
            indices = indices[torch.argsort(self._cost[indices], descending=True, stable=True)]
        return indices[rank::world]

    def batches(self, batch_size: int, shuffle: bool = True, generator: Optional[torch.Generator] = None,
                drop_last: bool = False, cost_ordered: bool = False, return_indices: bool = False,
                rank: int = 0, world: int = 1) -> Iterator[Tuple[Tensor, ...]]:
        """One epoch: a permutation drawn on the device and one gather per batch.  ``cost_ordered``: every batch
        is handed out by decreasing cost hint (see above); ``rank`` / ``world``: this rank's share of every batch;
        ``return_indices``: also yield the slice indices (to feed ``update_costs``)."""
        prev, fut = self.tensors()
        n = prev.shape[0]
        order = torch.randperm(n, device=self.device, generator=generator) if shuffle else None
        for lo in range(0, n, batch_size):
            hi = min(lo + batch_size, n)
            if drop_last and hi - lo < batch_size:
                return
            if order is None and not cost_ordered and world == 1:
                out = (prev[lo:hi], fut[lo:hi])
                idx = None
            else:
                idx = order[lo:hi] if order is not None else torch.arange(lo, hi, device=self.device)
                idx = self.cost_order(idx, rank, world) if cost_ordered else idx[rank::world]
                out = (prev.index_select(0, idx), fut.index_select(0, idx))
            if return_indices:
                out = out + (idx if idx is not None else torch.arange(lo, hi, device=self.device),)
            yield out
