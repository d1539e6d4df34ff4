"""The multi-head SDDMM restated on the C oracle, with no new C code:

    out[e, h] = < mat_1[dst_index[e], h, :] , mat_2[src_index[e], h, :] >

is ``oracle.sddmm_coo`` on the ``[N*H, F]`` views with the indices expanded to ``row*H + h`` / ``col*H + h``
(f64 accumulation, rounded once).  ``[E, H]``, or ``[H, E]`` with ``head_major``."""
import torch

import oracle


def sddmm_mh(src_index, dst_index, mat_1, mat_2, head_major=False):
    E, H, F = dst_index.numel(), mat_1.shape[1], mat_1.shape[2]
    heads = torch.arange(H)
    row = (dst_index.detach().cpu().long().view(E, 1) * H + heads).reshape(-1)
    col = (src_index.detach().cpu().long().view(E, 1) * H + heads).reshape(-1)
    out = oracle.sddmm_coo(col, row, mat_1.detach().cpu().reshape(-1, F), mat_2.detach().cpu().reshape(-1, F)).view(E, H)
    return out.t().contiguous() if head_major else out
