"""B200-native topological loss: the one hot path of philippendres/DILabHelmholtzOCT's
``training.py --top`` (``octsam/models/topological_loss.py``) rebuilt as sm_100a CUDA kernels
behind the reference's ``topo_loss`` signature, and its pieces -- differentiable persistence diagrams and
Wasserstein distances -- as batched GPU ops (``diagrams``; torch_topological-compatible layer in ``tda``), and the
Betti matching loss (``betti``) and the topological prior loss (``prior``); an exact distance transform and the
Hausdorff distance-transform loss, the signed distance map and the boundary loss, and surface-distance metrics of
mask pairs (``distance``)."""
from .betti import BettiMatching, betti_matching  # noqa: F401
from .distance import (SurfaceDistances, boundary_loss, distance_transform_edt, hausdorff_dt_loss,  # noqa: F401
                       signed_distance_map, surface_distances)
from .diagrams import Diagrams, cubical_persistence, total_persistence, wasserstein_distance  # noqa: F401
from .prior import topological_prior  # noqa: F401
from .topological_loss import (check_status, dice_ce_loss, pack_mask_bits, persistence_pairs, postprocess_masks, resample,  # noqa: F401
                               set_arena_factor, topo_loss, topo_loss_from_host, topo_loss_from_logits,
                               wasserstein_cost)

__all__ = ["topo_loss", "topo_loss_from_logits", "topo_loss_from_host", "resample", "postprocess_masks", "persistence_pairs",
           "wasserstein_cost", "check_status", "set_arena_factor", "dice_ce_loss", "pack_mask_bits",
           "cubical_persistence", "wasserstein_distance", "total_persistence", "Diagrams",
           "betti_matching", "BettiMatching", "topological_prior",
           "distance_transform_edt", "hausdorff_dt_loss", "surface_distances", "SurfaceDistances",
           "signed_distance_map", "boundary_loss"]
