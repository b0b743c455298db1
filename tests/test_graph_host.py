"""CPU checks of the graphed train step's plumbing: the library speaks ABI 5 (device step counters) and a graphed step of a module that is not
on the GPU raises the no-CPU-fallback error instead of running anything."""

import pytest

import pseudo_speaker_vae_b200 as P
from pseudo_speaker_vae_b200 import _lib as L


def test_abi_version_5_and_counter_block_layout():
    assert L.lib().psvae_abi_version() == 5 == L.PSVAE_ABI_VERSION
    # psvae_step_counters: uint64 rng_offset, int64 adam_step, 2 reserved int64 -> the int64 slots the Python side writes
    assert (L.COUNTER_RNG_OFFSET, L.COUNTER_ADAM_STEP, L.COUNTER_SLOTS) == (0, 1, 4)
    assert L.lib().psvae_step_counters_advance(None, None) != 0          # NULL block or no device: an error code, never a crash


def test_graphed_step_on_a_cpu_module_raises():
    m = P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=8, hidden_dim=64), classifier=dict(input_dim=8, num_classes=2),
                           optimizer=dict(lr=1e-3), scheduler=dict(T_max=10))
    tr = P.DataParallelTrainer(m, local_only=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.GraphedTrainStep(tr, rows=32)
