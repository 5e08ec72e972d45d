"""Drop-in `VectorQuantizer2` (taming's ldm/tamming/quantize.py:213-329, imported as `VectorQuantizer` by
ldm/models/autoencoder.py): the codebook lookup of the VQ-regularised first stage (`VQModel`, `VQModelInterface`).

Same constructor kwargs, state-dict key (`embedding.weight`, [n_e, e_dim]) and return values as the reference; the
arithmetic runs in one nearest-codebook kernel pair (sdb_vq_quantize) that never forms the [M, n_e] distance matrix.
The codebook is read from `embedding.weight` on every call (nothing is packed), so an in-place update of the weight
(EMA copy_, load_state_dict) is seen by the next call.  Built: eval-mode forward with legacy=True or False (the two give
the same loss bits), sane_index_shape, get_codebook_entry.  Not built: `remap` and codebook dimensions above 16.
"""
import torch
from torch import nn

from . import ops

MAX_E_DIM = 16


class VectorQuantizer2(nn.Module):
    def __init__(self, n_e, e_dim, beta, remap=None, unknown_index="random", sane_index_shape=False, legacy=True):
        super().__init__()
        if remap is not None:
            raise NotImplementedError("sdb200 VectorQuantizer2: remap is not built")
        if not 1 <= e_dim <= MAX_E_DIM:
            raise NotImplementedError("sdb200 VectorQuantizer2: codebook dimension e_dim=%d is outside [1, %d]" % (e_dim, MAX_E_DIM))
        self.n_e = n_e
        self.e_dim = e_dim
        self.beta = beta
        self.legacy = legacy
        self.embedding = nn.Embedding(self.n_e, self.e_dim)
        self.embedding.weight.data.uniform_(-1.0 / self.n_e, 1.0 / self.n_e)
        self.remap = remap
        self.re_embed = n_e
        self.unknown_index = unknown_index
        self.sane_index_shape = sane_index_shape

    def _codebook(self):
        w = self.embedding.weight.detach()
        return w if (w.dtype == torch.float32 and w.is_contiguous()) else w.float().contiguous()

    def _quantize(self, z, z_layout="nchw", zq_layout="nchw", want_idx=True, want_loss=True):
        """(z_q, loss, idx) of the fp32 kernel; z in z_layout, z_q in zq_layout (see ops.vq_quantize)."""
        from ._lib import require_cuda
        require_cuda(z)
        with torch.cuda.device(z.device):
            return ops.vq_quantize(z.float().contiguous(), self._codebook(), beta=self.beta, z_layout=z_layout,
                                   zq_layout=zq_layout, want_idx=want_idx, want_loss=want_loss)

    @torch.no_grad()
    def forward(self, z, temp=None, rescale_logits=False, return_logits=False):
        """z [B, e_dim, H, W] -> (z_q [B, e_dim, H, W], loss, (None, None, indices)); indices [B*H*W] int64, or
        [B, H, W] with sane_index_shape."""
        assert temp is None or temp == 1.0, "Only for interface compatible with Gumbel"
        assert rescale_logits == False, "Only for interface compatible with Gumbel"    # noqa: E712 (the reference's assert)
        assert return_logits == False, "Only for interface compatible with Gumbel"     # noqa: E712
        z_q, idx, loss = self._quantize(z)
        if self.sane_index_shape:
            idx = idx.reshape(z_q.shape[0], z_q.shape[2], z_q.shape[3])
        if z.dtype != torch.float32:
            z_q = z_q.to(z.dtype)
        return z_q, loss, (None, None, idx)

    @torch.no_grad()
    def get_codebook_entry(self, indices, shape):
        """embedding(indices); with shape = (batch, height, width, channel) the result is returned as NCHW."""
        from ._lib import require_cuda
        require_cuda(indices)
        with torch.cuda.device(indices.device):
            idx = indices.reshape(-1).long().contiguous()
            if shape is not None:
                B, H, W_, Cc = shape
                assert Cc == self.e_dim and B * H * W_ == idx.numel(), "shape %s does not match %d indices" % (tuple(shape), idx.numel())
                return ops.vq_codebook_gather(idx, self._codebook(), (B, H, W_), out_layout="nchw")
            out = ops.vq_codebook_gather(idx, self._codebook(), (1, 1, idx.numel()), out_layout="nhwc")
            return out.reshape(*indices.shape, self.e_dim)
