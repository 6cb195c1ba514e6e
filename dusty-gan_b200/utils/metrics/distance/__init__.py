from .cd.chamfer_distance import *  # noqa: F401,F403
from .cd.chamfer_distance import ChamferDistance, ChamferDistanceFunction, chamfer_distance  # noqa: F401
from .emd.earth_mover_distance import *  # noqa: F401,F403
from .emd.earth_mover_distance import EarthMoverDistanceFunction, earth_mover_distance  # noqa: F401
