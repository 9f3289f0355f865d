"""WassRank (mirror of ptranking/ltr_adhoc/listwise/wassrank/wassRank.py:22-86, mode 'SinkhornOT')."""
from ...base.adhoc_ranker import AdhocNeuralRanker
from ... import ops

# WassRankParameter.default_para_dict, wassRank.py:102-103
DEFAULT_WASS_PARA = dict(model_id='WassRank', mode='SinkhornOT', sh_itr=20, lam=0.1, smooth_type='ST', norm_type='BothST',
                         cost_type='eg', non_rele_gap=100, var_penalty=2.718281828459045, gain_base=4)


class WassRank(AdhocNeuralRanker):
    """Entropic optimal transport between the softmax (or normalised-gain) histograms of scores and labels, under a cost
    matrix built from the labels, as one fused kernel per batch.

    ``dict_cost_mats`` / ``dict_std_dists`` are accepted and ignored: the kernel rebuilds the cost matrix and the label
    histogram on the device every call, with the values the reference would cache.  Batches of B > 1 queries are
    evaluated per query with the loss and gradient scaled by 1/B (the reference runs at B=1 only: its
    torch.squeeze(cost, 0) fails otherwise).  ``wass_para_dict=None`` means WassRankParameter's defaults."""

    def __init__(self, sf_para_dict=None, wass_para_dict=None, dict_cost_mats=None, dict_std_dists=None, gpu=False, device=None):
        super().__init__(id='WassRank', sf_para_dict=sf_para_dict, gpu=gpu, device=device)
        self.wass_para_dict = dict(DEFAULT_WASS_PARA) if wass_para_dict is None else wass_para_dict
        self.dict_cost_mats, self.dict_std_dists = dict_cost_mats, dict_std_dists
        ops.wassrank_settings(self.wass_para_dict)     # unsupported modes and settings raise here, not at the first batch

    def custom_loss_function(self, batch_preds, batch_std_labels, **kwargs):
        """wassRank.py:43-86 without the per-call print; ``batch_ids`` is accepted and not needed."""
        batch_loss = ops.rank_loss('WassRank', batch_preds, batch_std_labels, **self.wass_para_dict, **self.ragged_kwargs(kwargs))
        self.backward_and_step(batch_loss)
        return batch_loss
