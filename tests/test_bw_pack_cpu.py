"""The backward-pack cache of framework/layer_grads.py: one entry per (weight, tag), replaced when the weight changes in place (a torch
optimizer's update bumps its version counter), when one of the tensors the pack also depends on changes, or when TrainStep's AdamW
kernel bumps _PackedCache.epoch; entries go with their weight.  Host-side logic only: runs on CPU tensors."""
import gc

import torch


def test_bw_pack_one_entry_per_weight_and_tag():
    from timbre_trap_b200.framework import layer_grads as LG
    from timbre_trap_b200.framework.packing import _PackedCache
    w, dep = torch.ones(4), torch.zeros(2)
    builds = []

    def build():
        builds.append(float(w.sum() + dep.sum()))
        return torch.full((1,), builds[-1])

    def entries():
        return len(LG._BW_PACKS.get(w, {}))

    first = LG._bw_pack(w, 'a', build, deps=(dep,))
    assert LG._bw_pack(w, 'a', build, deps=(dep,)) is first and builds == [4.0]
    for step in range(5):                               # optimizer steps: in-place updates
        with torch.no_grad():
            w.add_(1.0)
        assert float(LG._bw_pack(w, 'a', build, deps=(dep,))) == 4.0 * (step + 2)
        LG._bw_pack(w, ('b', 1), build)
        assert entries() == 2
    with torch.no_grad():
        dep.add_(1.0)
    assert float(LG._bw_pack(w, 'a', build, deps=(dep,))) == 24.0 + 2.0
    n = len(builds)
    _PackedCache.epoch += 1                             # TrainStep's AdamW kernel: weights changed behind the version counter
    LG._bw_pack(w, 'a', build, deps=(dep,))
    assert len(builds) == n + 1 and entries() == 2
    before = LG._bw_pack_entries()
    del w, first
    gc.collect()
    assert LG._bw_pack_entries() == before - 2
