"""pseudo_speaker_vae_b200 -- the VAE train step and latent sampling path of nmehlman/pseudo_speaker_VAE,
rebuilt for B200 (sm_100a): hand-written CUDA kernels behind a C-ABI (include/psvae_b200.h), driven from the
reference's own module API.  Nothing here falls back to PyTorch or the CPU for compute."""
from .data import PackedEmbeddingStore, PinnedBatchLoader, get_packed_dataloaders
from .embedding_classifier import EmbeddingClassifier
from .graphs import GraphedTrainStep
from .inference import conditional_synthesis, latent_transformation, sample_on_device, save_samples, shard_rows, unconditional_synthesis
from .latent_classifier import LatentClassifier
from .lightning import PseudoSpeakerVAE
from .model import VAEModel
from .optim import FusedAdam
from .parallel import DataParallelTrainer
from .search import cosine_topk
from .utils import map_cv_age_to_label, map_cv_gender_to_label, map_vctk_gender_to_label, parse_classifier_target, sample_filename

__all__ = [
    "VAEModel", "LatentClassifier", "EmbeddingClassifier", "PseudoSpeakerVAE", "FusedAdam", "DataParallelTrainer", "GraphedTrainStep", "unconditional_synthesis",
    "conditional_synthesis", "latent_transformation", "PackedEmbeddingStore", "PinnedBatchLoader", "get_packed_dataloaders", "sample_on_device", "save_samples", "shard_rows", "cosine_topk", "map_cv_age_to_label", "map_cv_gender_to_label",
    "map_vctk_gender_to_label", "parse_classifier_target", "sample_filename",
]
