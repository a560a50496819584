"""B200-native (sm_100a) implementation of the RotatE toolkit's scoring / loss / evaluation hot path,
behind the reference's own `KGEModel` API.  See DESIGN.md and INTEGRATION.md."""
from .model import KGEModel, ranks_from_statistics, shard_bounds  # noqa: F401
from .filter_index import FilterIndex  # noqa: F401

__all__ = ["KGEModel", "FilterIndex", "shard_bounds", "ranks_from_statistics"]
