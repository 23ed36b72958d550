from .base import MergeTensorsBase  # noqa: F401
from .fast_fourier import FourierMerge  # noqa: F401
from .addition import AdditionMerge  # noqa: F401
from .taskaddition import TaskAdditionMerge  # noqa: F401
from .ties import DareLinearMerge, DareTiesMerge, TiesMerge  # noqa: F401
from .fourier import FourierMerge as LegacyFourierMerge  # noqa: F401  (shard/merge/fourier.py: the in-RAM variant)
