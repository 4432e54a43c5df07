"""autoforce_b200 -- B200-native SGPR prediction path for AutoForce (theforce).

Drop-in for the hot path  ActiveCalculator.calculate -> neighbour list -> SOAP-type
descriptors -> (p.z)^xi kernel -> E / F / stress  of amirhajibabaei/AutoForce, executed
by hand-written sm_100a CUDA kernels behind the C ABI in include/sgpr_b200.h.
There is no CPU fallback: every compute entry point raises if the CUDA library or a
CUDA device is missing.
"""
from .model import SgprModel  # noqa: F401
from .engine import SgprEngine, library_path, load_library  # noqa: F401
from .calculator import B200Calculator  # noqa: F401
from .md import DeviceMD  # noqa: F401
from .relax import DeviceRelax  # noqa: F401
from .kernels import SeSoapKernel, SubSeSoapKernel, HeterogeneousSoapKernel, UniversalSoapKernel, DefaultRadii  # noqa: F401

__version__ = "0.1.0"
