"""The kernel launcher's argument check that needs no GPU: a CPU tensor is refused before the library is loaded."""
import pytest
import torch


def test_launch_refuses_cpu_tensors_without_loading_the_library(monkeypatch):
    from timbre_trap_b200 import _lib
    from timbre_trap_b200.framework import ops

    def no_library():
        raise AssertionError('the library was loaded')
    monkeypatch.setattr(_lib, 'lib', no_library)
    x = torch.zeros(8, dtype=torch.bfloat16)
    with pytest.raises(_lib.TimbreTrapB200Error, match='CUDA tensor'):
        _lib.launch('tt_add_scaled_bf16', x, x, torch.ones(1), x, x.numel())
    with pytest.raises(_lib.TimbreTrapB200Error, match='CUDA tensor'):
        _lib.launch('tt_multipitch_counts', None, x, 1, 8, 1, 0, None)
    with pytest.raises(_lib.TimbreTrapB200Error, match='CUDA tensor'):
        ops.add_scaled(x, x, torch.ones(()))
