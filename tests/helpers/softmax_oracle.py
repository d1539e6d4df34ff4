"""fp64 restatement of the segment softmax and its backward, the test graph of the exact check, and the error bounds
that follow from the kernels' accumulation order (geot_b200/csrc/kernels/softmax.cuh)."""
import torch

CHUNK = 8          # kSmChunk: edges a thread sums in sequence
THREADS = 256      # threads per CTA: a tile holds THREADS // min(H, THREADS) chunks


def softmax(src, index):
    """out[e, h] = exp(src[e, h] - m[r, h]) / sum_row exp(src - m), in fp64 on the CPU; src [E] or [E, H]."""
    x = src.detach().cpu().double()
    idx = index.detach().cpu().long()
    x2 = x.view(x.shape[0], -1)
    S = int(idx.max()) + 1 if idx.numel() else 0
    ix = idx.view(-1, 1).expand_as(x2)
    m = torch.full((S, x2.shape[1]), float("-inf"), dtype=torch.float64).scatter_reduce(0, ix, x2, "amax")
    ex = (x2 - m[idx]).exp()
    den = torch.zeros(S, x2.shape[1], dtype=torch.float64).index_add(0, idx, ex)
    return (ex / den[idx]).view_as(x)


def argument_terms(src, index):
    """|x - m| per element and sum_row out * |x - m| (fp64): the accumulator rounds the argument x - m of every exp,
    which costs |x - m| u relative on that term, and on the row sum at most the out-weighted mean of those.  Elements
    whose exp is exactly 0 (x = -inf) carry no such error."""
    x = src.detach().cpu().double()
    idx = index.detach().cpu().long()
    x2 = x.view(x.shape[0], -1)
    S = int(idx.max()) + 1
    m = torch.full((S, x2.shape[1]), float("-inf"), dtype=torch.float64).scatter_reduce(
        0, idx.view(-1, 1).expand_as(x2), x2, "amax")
    arg = (x2 - m[idx]).abs()
    arg = torch.where(torch.isfinite(arg), arg, 0.0)
    out = softmax(src, index).view_as(x2)
    spread = torch.zeros(S, x2.shape[1], dtype=torch.float64).index_add(0, idx, torch.nan_to_num(out) * arg)
    return arg.view_as(x), spread[idx].view_as(x)


def softmax_backward(out, grad_out, index):
    """grad_src = out * (grad_out - sum_row out * grad_out), in fp64 on the CPU; also returns sum_row |out * grad_out|
    per edge (the scale of the row sum's rounding error)."""
    y = out.detach().cpu().double()
    g = grad_out.detach().cpu().double()
    idx = index.detach().cpu().long()
    y2, g2 = y.view(y.shape[0], -1), g.view(g.shape[0], -1)
    S = int(idx.max()) + 1
    dot = torch.zeros(S, y2.shape[1], dtype=torch.float64).index_add(0, idx, y2 * g2)
    mag = torch.zeros(S, y2.shape[1], dtype=torch.float64).index_add(0, idx, (y2 * g2).abs())
    return (y2 * (g2 - dot[idx])).view_as(y), mag[idx].view_as(y), (g2 - dot[idx]).view_as(y)


def degrees(index):
    """Per-edge degree of its row."""
    idx = index.detach().cpu().long()
    return torch.bincount(idx)[idx]


def depth(deg, H):
    """Longest chain of sequential roundings behind a row of degree `deg` (tensor): the sum inside a chunk, the chain of
    chunk pieces inside a tile, one lane's stride over the tile pieces of the row (32 lanes), the 5-level tree of the
    lanes, and the tail piece."""
    nc = THREADS // min(H, THREADS)
    te = nc * CHUNK
    d = deg.double()
    tiles = torch.ceil(d / te) + 1
    return torch.clamp(d, max=CHUNK) + torch.clamp(torch.ceil(d / CHUNK) + 1, max=nc) + torch.ceil(tiles / 32) + 6


def unit(dtype):
    """Unit roundoff of the accumulator: fp32 for fp32 / bf16 / fp16, fp64 for fp64."""
    return 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24


def forward_tolerance(exp, deg, H, dtype, src, index):
    """Bound on |kernel - fp64| per element.  Every term exp(x - m) has at most 2 ulp of error, every rescale of a
    piece by exp(m_i - M) 2 ulp and every addition of the sequence 1 ulp, relative to the (positive) row sum: at most
    (8 + 3 depth) u relative, the division and the final rounding included.  The rounding of the exp arguments adds
    |x - m| u on the element's numerator and 2 sum_row out |x - m| u on the row sum (rescales included,
    argument_terms).  16-bit outputs: one ulp of the output type on top.  Below the smallest normal of the output type
    only an absolute error of that size is asked (the accumulator's exp underflows there)."""
    e = exp.abs()
    arg, spread = argument_terms(src, index)
    u = unit(dtype)
    tol = ((8 + 3 * depth(deg, H).view(-1, *([1] * (e.dim() - 1)))) * u + arg * u + 2 * spread * u) * e
    if dtype in (torch.bfloat16, torch.float16):
        tol = tol + e * 2.0 ** -(8 if dtype == torch.bfloat16 else 11) * 2
    return tol + torch.finfo(dtype).tiny


def backward_tolerance(exp, out, mag, diff, deg, H, dtype):
    """Bound on |kernel - fp64| of grad_src = out * (g - D), D = sum_row out * g summed in the kernel's order: D carries
    at most (depth + 2) u * sum_row |out * g|; g - D and the product add 2 u of their own; 16-bit outputs one ulp of
    the output type."""
    u = unit(dtype)
    o = out.detach().cpu().double().abs()
    dd = depth(deg, H).view(-1, *([1] * (o.dim() - 1)))
    tol = o * ((dd + 2) * u * mag + 2 * u * diff.abs()) + 2 * u * exp.abs()
    if dtype in (torch.bfloat16, torch.float16):
        tol = tol + exp.abs() * 2.0 ** -(8 if dtype == torch.bfloat16 else 11) * 2
    return tol + torch.finfo(dtype).tiny


def exact_graph(hub=80_001, seed=0):
    """A dst-sorted index with empty rows at the start, in the middle and at the end (rows no edge reaches), rows of
    every length around the chunk (8) and tile (128 .. 2048 edges) sizes, a hub row cut by more than 32 tiles at every H,
    and an odd E (a ragged last chunk).  Returns (index [E] int64, number of rows N > index[-1] + 1)."""
    g = torch.Generator().manual_seed(seed)
    degs = [0, 0, 0]                                              # empty rows at the start
    degs += [1, 2, 7, 8, 9, 15, 16, 17, 1, 1, 127, 128, 129, 255, 256, 257, 1023, 1024, 1025, 2047, 2048, 2049, 4100]
    degs += [0, 0]                                                # empty rows in the middle
    degs += torch.randint(1, 40, (300,), generator=g).tolist()
    degs += [hub]
    degs += torch.randint(1, 600, (40,), generator=g).tolist()
    degs += [0] + [3, 1]
    if sum(degs) % 2 == 0:
        degs[-1] += 1
    deg = torch.tensor(degs)
    index = torch.repeat_interleave(torch.arange(deg.numel()), deg)
    return index.contiguous(), deg.numel() + 5                   # five empty rows at the end


def random_graph(E, N, seed, hub=0):
    """Sorted index of E edges over N rows drawn from a skewed law, optionally with one hub row of `hub` extra edges."""
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(N, generator=g) ** 3
    di = torch.multinomial(w / w.sum(), E, replacement=True, generator=g)
    if hub:
        di = torch.cat([di, torch.full((hub,), N // 2)])
    return di.sort().values.contiguous(), g
