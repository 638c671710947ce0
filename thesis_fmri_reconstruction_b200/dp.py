"""Host-side logic of batch data parallelism (SURVEY.md section 8e): sharding, flat gradient buckets, SUM all-reduce and
the globally consistent equilibrium gate. Device-agnostic (the GPU engine uses it over NCCL, the CPU tests over gloo).

The reference is single-device (its device2/device3 settings are never used, train_vgan_stage1.py:118-119); this is the
one parallelism the B200 build adds. Semantics: every rank holds a full replica, BatchNorm statistics stay per rank (each
rank is a reference-sized training step on its shard), losses are batch SUMS (train_vgan_stage1.py:369-372) so gradients
are all-reduced with SUM and never divided, and the gate (train_vgan_stage1.py:396-404) is evaluated from the all-reduced
BCE sums over the GLOBAL batch so that all ranks take the same train_dis / train_dec branch.
"""
from __future__ import annotations

from collections import OrderedDict

import torch


def shard_range(global_batch, rank, world):
    """Samples [lo, hi) of the global batch owned by `rank` (equal shards; the global batch must divide evenly)."""
    if global_batch % world:
        raise ValueError(f"global batch {global_batch} is not divisible by {world} ranks")
    per = global_batch // world
    return rank * per, (rank + 1) * per


class FlatBucket:
    """Flat fp32 parameter / gradient / optimizer-state buffers of one sub-network; the named tensors are views, so one
    all-reduce and one multi-tensor optimizer launch cover the whole bucket."""

    def __init__(self, prefix, named_params, n_states, device):
        self.prefix = prefix
        self.names = list(named_params)
        sizes = [named_params[k].numel() for k in self.names]
        offs, o = [], 0
        for s in sizes:
            offs.append(o)
            o += (s + 3) // 4 * 4  # keep every tensor 16-byte aligned inside the flat buffer
        self.numel = o
        self.flat_p = torch.zeros(o, dtype=torch.float32, device=device)
        self.flat_g = torch.zeros(o, dtype=torch.float32, device=device)
        self.states = [torch.zeros(o, dtype=torch.float32, device=device) for _ in range(n_states)]
        self.P, self.G = OrderedDict(), OrderedDict()
        for k, off, s in zip(self.names, offs, sizes):
            shape = named_params[k].shape
            self.P[k] = self.flat_p[off:off + s].view(shape)
            self.G[k] = self.flat_g[off:off + s].view(shape)
            self.P[k].copy_(named_params[k])
        self.offsets = dict(zip(self.names, zip(offs, sizes)))

    def state_view(self, i, name):
        off, s = self.offsets[name]
        return self.states[i][off:off + s].view(self.P[name].shape)


def allreduce_sum_(tensors, group=None):
    """In-place SUM all-reduce of each tensor over `group` (no averaging: the losses are sums over the batch)."""
    import torch.distributed as td

    if not td.is_available() or not td.is_initialized() or td.get_world_size(group) == 1:
        return
    for t in tensors:
        td.all_reduce(t, op=td.ReduceOp.SUM, group=group)


def gate_from_sums(sum_bce_o, sum_bce_p, global_batch, margin, equilibrium, train_dis_in=True):
    """Host restatement of the gate (train_vgan_stage1.py:396-404) on globally reduced sums; the engine evaluates the same
    rule on the device (fmri_vgan_gate_mix). train_dis_in: train_dis as the loss-mix block leaves it before the gate (False
    in mode 'vae', :387). Returns (train_dis, train_dec)."""
    mo, mp = sum_bce_o / global_batch, sum_bce_p / global_batch
    dis, dec = bool(train_dis_in), True
    if mo < equilibrium - margin or mp < equilibrium - margin:
        dis = False
    if mo > equilibrium + margin or mp > equilibrium + margin:
        dec = False
    if not dis and not dec:
        dis = dec = True
    return dis, dec
