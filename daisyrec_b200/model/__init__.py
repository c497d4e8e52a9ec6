from .MFRecommender import MF  # noqa: F401
from .FMRecommender import FM  # noqa: F401
from .NeuMFRecommender import NeuMF  # noqa: F401
from .LightGCNRecommender import LightGCN  # noqa: F401
from .NGCFRecommender import NGCF  # noqa: F401
from .NFMRecommender import NFM  # noqa: F401
from .Item2VecRecommender import Item2Vec  # noqa: F401
