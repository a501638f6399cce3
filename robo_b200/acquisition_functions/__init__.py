from .ei import EI  # noqa: F401
from .log_ei import LogEI  # noqa: F401
from .pi import PI  # noqa: F401
from .lcb import LCB  # noqa: F401
from .marginalization import MarginalizationGPMCMC  # noqa: F401
from .information_gain import InformationGain  # noqa: F401
from .information_gain_per_unit_cost import InformationGainPerUnitCost  # noqa: F401
