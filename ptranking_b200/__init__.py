"""ptranking_b200 -- B200-native (sm_100a) scoring-and-loss hot path behind PTRanking's plugin API.

    import ptranking_b200
    ptranking_b200.install()           # swap the loss classes into ptranking.ltr_adhoc.eval.ltr
    LTREvaluator(cuda=0).run(model_id='LambdaRank', ...)   # the unmodified reference driver

Importing the package never touches the GPU; the first kernel call loads
lib/libptranking_b200.so and raises if it (or an sm_100 device) is missing.
"""
from .ltr_adhoc.pairwise.ranknet import RankNet
from .ltr_adhoc.listwise.lambdarank import LambdaRank
from .ltr_adhoc.listwise.lambdaloss import LambdaLoss
from .ltr_adhoc.listwise.listnet import ListNet
from .ltr_adhoc.listwise.listmle import ListMLE
from .ltr_adhoc.listwise.approxNDCG import ApproxNDCG
from .ltr_adhoc.pointwise.rank_mse import RankMSE
from .ltr_adhoc.listwise.rank_cosine import RankCosine
from .ltr_adhoc.listwise.st_listnet import STListNet
from .ltr_adhoc.listwise.softrank import SoftRank
from .ltr_adhoc.listwise.wassrank import WassRank
from .base.ranker import LABEL_TYPE

MODELS = {c.__name__: c for c in (RankNet, LambdaRank, LambdaLoss, ListNet, ListMLE, ApproxNDCG,
                                  RankMSE, RankCosine, STListNet, SoftRank, WassRank)}
__version__ = "0.1.0"


def install(module=None):
    """Register the B200 classes where the reference resolves model ids by name:
    ``globals()[model_id]`` in ptranking/ltr_adhoc/eval/ltr.py:166-171."""
    if module is None:
        import ptranking.ltr_adhoc.eval.ltr as module  # the reference package must be importable
    previous = {}
    for name, cls in MODELS.items():
        previous[name] = getattr(module, name, None)
        setattr(module, name, cls)
    return previous
