"""The many-clip calls' argument checks that need no GPU: an empty list, and CPU clips (there is no CPU path)."""
import pytest
import torch


def test_many_empty_list_and_cpu_clips():
    from timbre_trap_b200._lib import TimbreTrapB200Error
    from timbre_trap_b200.framework import TimbreTrap, TimbreTrapMag
    for cls in (TimbreTrap, TimbreTrapMag):
        model = cls(8000, 6, 12, 0.5, latent_size=16, model_complexity=1)
        assert model.transcribe_many([]) == [] and model.reconstruct_many([]) == []
        assert model.transcribe_and_reconstruct_many(iter([])) == ([], [])
        for call in (model.transcribe_many, model.reconstruct_many, model.transcribe_and_reconstruct_many):
            with pytest.raises(TimbreTrapB200Error):
                call([torch.zeros(4000)])
