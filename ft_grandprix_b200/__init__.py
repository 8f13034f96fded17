"""B200-native batched replacement for the hot path of FT-Autonomous/ft_grandprix:
track compiler -> lidar -> driver -> vehicle step -> lap logic, for fleets of cars on device.

Everything numeric lives in libftgp.so (csrc/*.cu, C ABI in include/ftgp.h).  Importing this
package loads that library and fails loudly if it has not been built."""
from . import _lib
from .drivers import BatchedFastDriver, BatchedLobotomyDriver, BatchedNidcDriver, LobotomyDriver
from .policy import PolicyNet, policy_inputs
from .track import Geometry, Track, centreline
from .vehicle import VehicleStateSnapshot

_lib.load()
from . import fleet
from .fleet import Fleet
