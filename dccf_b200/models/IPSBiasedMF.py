"""IPSBiasedMF with the reference's model protocol (src/models/IPSBiasedMF.py): BiasedMF divided by the clamped
propensity of the item,

    pred = (<p_u, q_i> + b_u + b_i + g) / max(propensity_i, M)

the exposure model whose U x I prediction is DCCF's `<dataset>.ips_expo_prob.npy` (README.md:27-29 of the reference;
tools/export_exposure.py writes it).  The propensity [I] is read from `<path>/<dataset>.propensity.npy`; it is a plain
attribute, not part of the state dict, like the reference's.  Same parameters, initial values and training step as
BiasedMF."""
import os

import numpy as np
import torch

from ..utils import global_p
from .BiasedMF import BiasedMF


class IPSBiasedMF(BiasedMF):
    @staticmethod
    def parse_model_args(parser, model_name='IPSBiasedMF'):
        parser.add_argument('--M', type=float, default=0.1, help='lower clamp of the propensity (SURVEY.md row 9)')
        return BiasedMF.parse_model_args(parser, model_name)

    def __init__(self, path, dataset, M, label_min, label_max, feature_num, user_num, item_num, u_vector_size,
                 i_vector_size, random_seed, model_path, propensity=None):
        """Reference constructor arguments; `propensity` (an [I] array) is an addition: used instead of the file."""
        self.path, self.dataset, self.M = path, dataset, float(M)
        if propensity is None:
            propensity = np.load(os.path.join(path, dataset + global_p.PROPENSITY_SUFFIX))
        propensity = torch.as_tensor(np.asarray(propensity, dtype=np.float32)).contiguous()
        if propensity.shape != (item_num,):
            raise ValueError('propensity must have shape [%d] (one value per item), got %s'
                             % (item_num, tuple(propensity.shape)))
        self.propensity = propensity
        BiasedMF.__init__(self, label_min=label_min, label_max=label_max, feature_num=feature_num, user_num=user_num,
                          item_num=item_num, u_vector_size=u_vector_size, i_vector_size=i_vector_size,
                          random_seed=random_seed, model_path=model_path)

    def _scale(self):
        dev = self.uid_embeddings.weight.device
        if self.propensity.device != dev:
            self.propensity = self.propensity.to(dev)
        return self.propensity, self.M
