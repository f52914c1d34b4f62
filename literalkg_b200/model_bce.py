"""Drop-in for the reference's ``model_bce.py`` (the variant ``main_pretraining_BCE.py`` / ``main_finetuning_BCE.py``
drive -- the self-consistent entry path at the reference's HEAD, SURVEY.md fact 8).

Same trunk as ``model.LiteralKG`` (gate, aggregators, ``linear_gat``, attention update), different heads:
  * no ``gat_trans_M``; ``calc_triplet_loss`` is TransE on rows of the final embeddings (model_bce.py:329-368), which
    needs ``relation_dim == scale_gat_dim`` exactly like the reference (it adds the two); the triple score of
    ``evaluate_ranking(score="triple")`` is TransE likewise;
  * the MLP head (``fc1 / norm1 / fc2 / norm2 / fc3``) is built by the constructor (model_bce.py:254-258) and mode
    ``'mlp'`` returns its sigmoid output for ``nn.BCELoss`` (main_finetuning_BCE.py:117-120).
"""
from __future__ import annotations

from .model import Aggregator, LiteralKG as _Base, _TransELossFn   # noqa: F401 -- Aggregator re-exported like upstream


class LiteralKG(_Base):
    """model_bce.py:166-447."""

    def __init__(self, args, n_entities, n_relations, A_in=None, numerical_literals=None, text_literals=None):
        super().__init__(args, n_entities, n_relations, A_in, numerical_literals, text_literals)
        del self.gat_trans_M                       # the BCE variant has no TransR projection (state-dict parity)
        self.initialize_MLP()                      # model_bce.py:254-258

    def triplet_loss_from(self, all_embed, h, r, pos_t, neg_t):
        """TransE loss (model_bce.py:329-368) of one minibatch on a given embedding matrix."""
        return _TransELossFn.apply(all_embed, self.relation_embed.weight, h, r, pos_t, neg_t,
                                   float(self.kg_l2loss_lambda))

    def _triple_projection(self):
        return None                                # TransE: the triple score needs no projection
