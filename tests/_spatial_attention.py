"""fp64 reference of the text-to-location attention maps of a spatial-embedding model (test infrastructure).

The reference has no function that returns these maps.  They are the per-location terms of its own spatial
similarity (multimodal.py:771-780): the einsum of `oracle.similarity_spatial_max` without the max / mean
reductions, taken for every image against its own label row.  Formula-only, like `oracle.classify_ncat`."""
import torch
import torch.nn.functional as F


def spatial_attention_maps(u, ids, lens, table, normalize=True):
    """u [M, E, H, W] head outputs; ids / lens [M, L] / [M] the label row of every image; table [V, E].
    -> (token maps [M, L, H, W], utterance maps [M, H, W]) in fp64.  Token rows at or past the length are 0 (the
    reference's <pad> rows are the zero embedding row; the mask makes it so for any id); the utterance map is the
    sum over the tokens divided by the length (0 / 0 = NaN for an empty label)."""
    u = u.double()
    tok = table.double()[ids]
    if normalize:
        u = F.normalize(u, dim=1)
        tok = F.normalize(tok, dim=-1)
    live = torch.arange(ids.shape[1], device=ids.device)[None, :] < lens[:, None]
    tok = tok * live[..., None]
    token_maps = torch.einsum("mehw,mle->mlhw", u, tok)
    return token_maps, token_maps.sum(dim=1) / lens.double()[:, None, None]
