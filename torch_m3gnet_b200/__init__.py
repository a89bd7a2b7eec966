"""torch_m3gnet_b200 — B200-native (sm_100a) energy+forces inference path of M3GNet behind the model API of
lan496/torch-m3gnet.  All arithmetic runs in hand-written CUDA kernels behind a C ABI
(include/m3gnet_b200.h); there is no CPU or eager-PyTorch fallback."""

__version__ = "0.1.0"

from torch_m3gnet_b200.data.material_graph import Batch, MaterialGraph  # noqa: E402,F401
from torch_m3gnet_b200.model.build import build_model  # noqa: E402,F401
from torch_m3gnet_b200.data.verlet import VerletList  # noqa: E402,F401
from torch_m3gnet_b200.calculator import Fire, M3GNetCalculator, VelocityVerlet  # noqa: E402,F401
from torch_m3gnet_b200.relax import BatchFire  # noqa: E402,F401
from torch_m3gnet_b200.md import BatchMD  # noqa: E402,F401
from torch_m3gnet_b200.neb import BatchNEB  # noqa: E402,F401
from torch_m3gnet_b200.phonon import BatchPhonon  # noqa: E402,F401
