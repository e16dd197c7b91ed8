"""B200-native SDF auto-decoder and latent-DDPM sampler (hot path only).

Python mirror of the API that BASELINE.json's north_star names - there is no upstream
source to mirror (`/root/reference/README.md:1` is a title):

    Decoder(latent, xyz) -> sdf      decode_grid(z, res)      sample_latents(n)

Everything numeric runs in hand-written sm_100a CUDA inside libsdfb200.so (C ABI:
include/sdfb200.h) and is reached through ctypes; torch supplies device memory,
streams and torch.distributed.  There is no CPU fallback.

The directory name contains hyphens, so import it with
``importlib.import_module("latent-diffusion-models-for-shape-sdfs_b200")``
(``__graft_entry__.load_package()`` does exactly that).
"""
from ._lib import PRECISIONS, SdfbError, load as load_library  # noqa: F401
from .api import (Decoder, LatentDDPM, DDPMTrainer, DecoderTrainer, Comm, decode_grid, sample_latents, grid_points, sign_change_mask, philox_normal,  # noqa: F401
                  ddim_schedule,
                  extract_surface, weld, unpack_mask_blocks, DDPM_LATENT_SCALE)
from .sharding import (slab_range, batch_range, decode_grid_sharded, decode_batch_sharded, sample_latents_sharded,  # noqa: F401
                       fit_latents_sharded)
from . import synthetic  # noqa: F401
from .training import bench_training_legs  # noqa: F401
