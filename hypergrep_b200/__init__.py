"""gpugrep: B200-native multi-pattern log scanning behind hypergrep's Python API.

Drop-in for the names exported by the reference package (reference hypergrep/__init__.py:3-14): the same
functions, constants and ctypes types, backed by ``lib/libgpugrep.so`` instead of libhyperscanner/libhs.
"""

from hypergrep_b200.utils import CALLBACK_TYPE
from hypergrep_b200.utils import CONTEXT_ID
from hypergrep_b200.utils import HS_FLAG_CASELESS
from hypergrep_b200.utils import HS_FLAG_DOTALL
from hypergrep_b200.utils import HS_FLAG_MULTILINE
from hypergrep_b200.utils import HS_FLAG_SINGLEMATCH
from hypergrep_b200.utils import RC_INVALID_FILE
from hypergrep_b200.utils import Result
from hypergrep_b200.utils import check_compatibility
from hypergrep_b200.utils import configure_libraries
from hypergrep_b200.utils import count_patterns
from hypergrep_b200.utils import grep
from hypergrep_b200.utils import prepare_patterns
from hypergrep_b200.utils import scan
from hypergrep_b200.utils import scan_literals

__version__ = "0.1.0"
__all__ = [
    "CALLBACK_TYPE",
    "CONTEXT_ID",
    "HS_FLAG_CASELESS",
    "HS_FLAG_DOTALL",
    "HS_FLAG_MULTILINE",
    "HS_FLAG_SINGLEMATCH",
    "RC_INVALID_FILE",
    "Result",
    "check_compatibility",
    "configure_libraries",
    "count_patterns",
    "grep",
    "prepare_patterns",
    "scan",
    "scan_literals",
]
