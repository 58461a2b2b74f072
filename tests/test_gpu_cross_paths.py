"""The DCN cross kernels (csrc/cross.cu) at every instantiation dir_cross_fwd / dir_cross_bwd can reach:

  1  `_cross_plan(d, L)` restates the dispatcher; a CPU test enumerates d in [1, 1024] x L in [1, 32] and requires
     the case lists below to reach every forward instantiation and every backward variant;
  2  one profiled run pins the restatement to the library: the kernels each case launches are the ones predicted;
  3  parity against fp64 torch autograd of the layer-by-layer formula, every element held to REL x its own floor, at
     the band edges of every variant, at B = 1 and 37, and at B = 19001 for one pair per variant, with every output
     and the whole workspace poisoned (NaN) before each call;
  4  exact properties: saved and recomputed p_l give bit-identical gradients, two runs are bit-identical, w = 0 gives
     x0 + sum_l b_l, dy = 0 gives zero gradients, B = 0 zeroes dw / db;
  5  negative controls: the same bound rejects a reference that is wrong by one sample, one column term or one layer;
  6  the ABI's alignment rule: misaligned x0 / dy are refused when d % 4 == 0 and computed correctly otherwise.

Floors.  The reference is run a second time on |x0|, |w|, |b| with upstream |dy|.  Every input is then non-negative,
so each output is the sum of the absolute values of the terms the true result sums, over every way of grouping them
-- including the rank-1 order the kernels use (x_l = x0 c_l + beta_l, header of cross.cu).  That is the magnitude
an fp32 evaluation's rounding scales with (SURVEY 7.2), so an element may differ from the fp64 value by REL x floor.
"""
import pytest
import torch

from tests._util import REL

gpu = pytest.mark.gpu

WARPS = 8                  # kCrossWarps
RING_MAX_DEPTH = 4         # kRingMaxDepth
RING_REGS = 184            # floats per lane the ring kernel may keep as batch sums: 4 NPL (LT + 3) <= 184
RING_SMEM = 216 * 1024     # the ring kernel's shared-memory budget
FWD_SMEM = 64 * 1024       # w is staged in shared memory up to this size


# ---------------------------------------------------------------------------------------------------------------
# 1. the dispatch plan

def _cross_shape(d):
    """(VEC, NPL) of cross_shape(): float4 lanes when d % 4 == 0, else one float per lane."""
    if d % 4 == 0:
        n = (d // 4 + 31) // 32
        return 4, (n if n <= 6 else 8)
    n = (d + 31) // 32
    return 1, next(k for k in (1, 2, 4, 8, 16, 32) if n <= k)


def _cross_plan(d, L):
    """The kernels dir_cross_fwd / dir_cross_bwd choose for (d, L) ->
    (forward (VEC, NPL, WSMEM), backward ("ring", NPL, LT, depth) | ("fused", VEC, NPL) | ("twopass", VEC, NPL))."""
    vec, npl = _cross_shape(d)
    fwd = (vec, npl, L * vec * npl * 32 * 4 <= FWD_SMEM)
    if L <= 8 and vec == 4:
        lt = (L + 1) & ~1
        fixed = (L * 4 * npl * 32 + WARPS * 32 + 32 + WARPS) * 4
        depth = RING_MAX_DEPTH
        while depth > 1 and fixed + WARPS * depth * 2 * d * 4 > RING_SMEM:
            depth -= 1
        # Depth 2 is never chosen: d <= 1024 always leaves room for 3 slots (fixed + 8 * 3 * 2 * 1024 * 4 = 203 KiB
        # at d = 1024, L = 8), so the ring runs with 3 or 4 slots.
        if 4 * npl * (lt + 3) <= RING_REGS and depth >= 2:
            return fwd, ("ring", npl, lt, depth)
    if L <= 8:
        return fwd, ("fused", vec, npl)
    return fwd, ("twopass", vec, npl)


def _kernels(d, L):
    """The kernel names the profiler shows for one forward and one backward call (namespace and spaces dropped)."""
    (v, n, wsmem), bwd = _cross_plan(d, L)
    fwd = ["cross_fwd_kernel<%d,%d,%s>" % (v, n, "true" if wsmem else "false")]
    if bwd[0] == "ring":
        first = ["cross_bwd_ring_kernel<%d,%d>" % bwd[1:3]]
    elif bwd[0] == "fused":
        first = ["cross_bwd_fused_kernel<%d,%d>" % bwd[1:]]
    else:
        first = ["cross_bwd_sample_kernel<%d,%d>" % bwd[1:], "cross_bwd_dw_kernel"]
    return fwd, first + ["cross_bwd_finish2_kernel"]


# The band edges of every variant: the smallest and largest d that reaches it, each at its smallest and largest L.
# They include the two-pass dw kernel's 8-layer chunks (L = 9, 16, 17, 32 at d = 999 .. 1024), the forward's
# shared-to-global switch (L = 16 / 17 at NPL 8 and 32, 21 / 22 at NPL 6, 25 / 26 at NPL 5) and odd L for the
# ring's and the fused kernel's padding layer.
_E = (1, 8, 9, 32)                        # one-float widths: fused at L <= 8, two-pass above
_R = tuple(range(1, 10)) + (32,)          # float4 widths below 513: every ring LT at both edges
PAIR_L = {1: _E, 4: _R, 31: _E, 33: _E, 63: _E, 65: _E, 127: _E, 128: _R, 129: _E, 132: _R, 255: _E, 256: _R, 257: _E,
          260: _R, 384: _R, 388: _R, 511: _E, 512: _R, 513: (1, 8, 9, 16, 17, 32),
          516: _R[:9] + (25, 26, 32), 640: _R[:9] + (25, 26, 32),
          644: (1, 2, 3, 4, 5, 8, 9, 21, 22, 32), 768: (1, 2, 3, 4, 5, 8, 9, 21, 22, 32),
          772: (1, 2, 3, 8, 9, 16, 17, 32), 828: (2,), 840: (1,),
          999: (9, 16, 17, 32), 1020: (9, 16, 17, 32), 1023: (1, 8, 9, 16, 17, 32), 1024: (1, 2, 3, 8, 9, 16, 17, 32)}
PAIRS = [(d, L) for d, Ls in PAIR_L.items() for L in Ls]

# One pair per variant, run at B = 19001 (odd, not a multiple of 16): 148 ring CTAs of 8 warps give every warp about
# 16 samples against at most 4 ring slots; 296 fused CTAs walk about four 16-sample tiles each; the forward's 296 x 8
# warps take samples in pairs and wrap four times; the two-pass sample grid (592 x 8 warps) wraps, and its dw grid
# (592 CTAs of 33 samples, not a multiple of kDwUnroll = 8) ends in a partial CTA and 16 CTAs with an empty range
# (any B below 18944 leaves none empty).
BIG_B = 19001
BIG = [(31, 8), (31, 32), (63, 8), (63, 32), (127, 8), (127, 32), (128, 2), (128, 4), (128, 6), (128, 8), (128, 32),
       (255, 8), (255, 32), (256, 2), (256, 4), (256, 6), (256, 8), (256, 32), (384, 2), (384, 4), (384, 6), (384, 8),
       (384, 32), (511, 8), (511, 32), (512, 2), (512, 4), (512, 6), (512, 8), (512, 32), (640, 2), (640, 4), (640, 6),
       (640, 8), (640, 32), (768, 2), (768, 4), (768, 8), (768, 32), (840, 1), (1023, 8), (1023, 32), (1024, 2),
       (1024, 8), (1024, 32)]

PARITY_CASES = [(B, d, L) for d, L in PAIRS for B in (1, 37)] + [(BIG_B, d, L) for d, L in BIG]


def test_cross_plan_covers_every_variant():
    fwd_all, bwd_all = set(), set()
    for d in range(1, 1025):
        for L in range(1, 33):
            f, b = _cross_plan(d, L)
            fwd_all.add(f)
            bwd_all.add(b)
    assert len(fwd_all) == 17 and len(bwd_all) == 45, (len(fwd_all), len(bwd_all))
    assert not any(b[0] == "ring" and b[3] < 3 for b in bwd_all), "ring depth 2 is unreachable"
    for name, pairs in (("PAIRS", PAIRS), ("BIG", BIG)):
        f = {_cross_plan(d, L)[0] for d, L in pairs}
        b = {_cross_plan(d, L)[1] for d, L in pairs}
        assert f == fwd_all, (name, sorted(fwd_all - f))
        assert b == bwd_all, (name, sorted(bwd_all - b, key=str))
    # the edges: for each variant, its smallest and largest d, each at its smallest and largest L, are in PAIRS
    bands = {}
    for d in range(1, 1025):
        for L in range(1, 33):
            for v in _cross_plan(d, L):
                bands.setdefault(v, []).append((d, L))
    edges = set()
    for v, dl in bands.items():
        for d in (min(p[0] for p in dl), max(p[0] for p in dl)):
            Ls = [L for dd, L in dl if dd == d]
            edges.update({(d, min(Ls)), (d, max(Ls))})
    assert edges <= set(PAIRS), sorted(edges - set(PAIRS))
    print("cross plan: %d/%d forward and %d/%d backward variants reached" % (len(fwd_all), 17, len(bwd_all), 45))


# ---------------------------------------------------------------------------------------------------------------
# helpers: data, reference, calls through the C ABI

def _w_scale(d, L):
    """Factor on w that keeps the floors within e^2 of the values they bound.  The floor of c_L grows like
    prod_l (1 + |x0| . |w_l|), and at the reference's init (E|x0| = 0.399, E|w| = 0.0723) each |x0| . |w_l| is about
    0.0288 d: unscaled, d = 1024 and L = 32 would give a floor e^900 times the signed result, and a bound that
    sees nothing.  So w is scaled by 2 / (0.0288 d L) whenever d L > 69 (every case but the narrowest), which keeps
    sum_l |x0| . |w_l| near 2, |p_l| far below 0.5 and c_L, ds_l finite.  The cross terms still move every output by
    far more than REL: at d = 1024, L = 32, c_L - 1 is about 2e-2."""
    return min(1.0, 2.0 / (0.0288 * d * L))


def _data(B, d, L, seed, device="cuda", heavy_tail=False):
    """x0 ~ N(0, 0.5^2), dy ~ N(0, 1), w and b truncated normal(0.1) as CrossNetwork initialises them (w scaled by
    _w_scale).  Drawn on the host so that every machine sees the same numbers.  heavy_tail: the last sample's dy is
    32 times larger and has the signs of its x0.  That sample ends the last partial tile, ring pass and dw range,
    where a dropped sample would be, and it keeps one sample visible against dw's floor: the floor sums
    |dy| . |x0|, about sqrt(d) times an ordinary sample's signed a = dy . x0, so at d ~ 1024 and B = 19001 such a
    sample's share of dw falls below REL x floor; the last sample's a sums without cancellation."""
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn((B, d), generator=g) * 0.5
    dy = torch.randn((B, d), generator=g)
    if heavy_tail:
        dy[-1] = 32.0 * dy[-1].abs() * torch.sign(x0[-1])
    w = torch.nn.init.trunc_normal_(torch.empty(L, d), 0.0, 0.1, -0.2, 0.2, generator=g) * _w_scale(d, L)
    b = torch.nn.init.trunc_normal_(torch.empty(L, d), 0.0, 0.1, -0.2, 0.2, generator=g)
    return tuple(t.float().to(device) for t in (x0, w, b, dy))


def _fp64(x0, w, b, dy, per_sample=False):
    """Autograd of x_{l+1} = x0 * (x_l . w_l) + b_l + x_l in fp64 (DeepCrossNetwork.py:345-346, layer by layer) ->
    dict(xL, s (= x0 . w_l, what dir_cross_fwd saves), dx0, dw, db); with per_sample also the per-layer inputs x_l,
    the gradients ds_l of s_l = x_l . w_l and g_l of x_{l+1}, from which one sample's share of dw_l, db_l follows."""
    x0 = x0.double().requires_grad_(True)
    w = w.double().requires_grad_(True)
    b = b.double().requires_grad_(True)
    xl, xs, ss, outs = x0, [], [], []
    for l in range(w.shape[0]):
        s = xl @ w[l]
        nxt = x0 * s[:, None] + b[l] + xl
        if per_sample:
            s.retain_grad()
            nxt.retain_grad()
            xs.append(xl.detach())
            ss.append(s)
            outs.append(nxt)
        xl = nxt
    xl.backward(dy.double())
    r = dict(xL=xl.detach(), s=x0.detach() @ w.detach().T, dx0=x0.grad, dw=w.grad, db=b.grad)
    if per_sample:
        r.update(x=xs, ds=[s.grad for s in ss], g=[o.grad for o in outs])
    return r


def _reference(x0, w, b, dy, per_sample=False):
    """-> (fp64 reference, floors)."""
    return _fp64(x0, w, b, dy, per_sample), _fp64(x0.abs(), w.abs(), b.abs(), dy.abs())


def _bad(got, ref, floor):
    """Elements of `got` outside REL * floor of the fp64 value (NaN counts as outside)."""
    return int((~((got.double() - ref).abs() <= REL * floor)).sum())


def _worst(got, ref, floor):
    err = (got.double() - ref).abs() / floor.clamp_min(1e-300)
    return float(err.max()) if err.numel() else 0.0


def _lib():
    from dir_b200 import _lib as L
    return L


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _poisoned(shape, dtype=torch.float32):
    """A fresh buffer of 0xFF bytes: NaN as float, so an element no kernel writes fails every bound."""
    t = torch.empty(shape, dtype=dtype, device="cuda")
    t.view(torch.uint8).fill_(0xFF)
    return t


def _fwd(x0, w, b, save_s=True):
    """dir_cross_fwd into poisoned outputs -> (xL, s or None, launches)."""
    L_ = _lib()
    lib = L_.lib()
    B, d = x0.shape
    L = w.shape[0]
    xL = _poisoned((B, d))
    s = _poisoned((B, L)) if save_s else None
    n0 = lib.dir_launch_count()
    L_.check(lib.dir_cross_fwd(L_.ptr(x0), L_.ptr(w), L_.ptr(b), B, d, L, L_.ptr(xL), L_.ptr(s), _stream()),
             "dir_cross_fwd")
    return xL, s, int(lib.dir_launch_count() - n0)


def _bwd(x0, w, b, dy, s):
    """dir_cross_bwd with poisoned outputs and a poisoned workspace -> (dx0, dw, db, launches)."""
    L_ = _lib()
    lib = L_.lib()
    B, d = x0.shape
    L = w.shape[0]
    ws = _poisoned(int(lib.dir_cross_bwd_workspace_bytes(B, d, L)), torch.uint8)
    dx0, dw, db = _poisoned((B, d)), _poisoned((L, d)), _poisoned((L, d))
    n0 = lib.dir_launch_count()
    L_.check(lib.dir_cross_bwd(L_.ptr(x0), L_.ptr(w), L_.ptr(b), L_.ptr(dy), L_.ptr(s), B, d, L, L_.ptr(dx0),
                               L_.ptr(dw), L_.ptr(db), L_.ptr(ws), ws.numel(), _stream()), "dir_cross_bwd")
    return dx0, dw, db, int(lib.dir_launch_count() - n0)


def _check_all(got, ref, flo, what):
    bad = {k: _bad(got[k], ref[k], flo[k]) for k in got}
    assert not any(bad.values()), (what, bad, {k: _worst(got[k], ref[k], flo[k]) for k in got})


# ---------------------------------------------------------------------------------------------------------------
# 5. negative controls: references wrong by one small, well-defined amount

def _controls_dx0(dx0, ref, flo, w):
    """Violations of a reference dx0 in which one sample's last column lacks its w_{L-1} term: dx0 = c_L dy +
    sum_l alpha_l w_l with alpha_l = ds_l c_l and c_l = 1 + sum_{j<l} s_j (header of cross.cu).  The sample is the
    one where that term is largest against the floor."""
    L, d = w.shape
    c = torch.ones_like(ref["ds"][0])
    for l in range(L - 1):
        c = c + ref["x"][l] @ w[l].double()
    term = ref["ds"][L - 1] * c * float(w[L - 1, d - 1])
    bsel = int((term.abs() / flo["dx0"][:, d - 1]).argmax())
    wrong = ref["dx0"].clone()
    wrong[bsel, d - 1] -= term[bsel]
    return _bad(dx0, wrong, flo["dx0"])


def _controls_sample(dw, db, ref, flo):
    """Violations of a reference dw and a reference db that each lack one sample: the one whose own share is largest
    against the floor (a dropped tail or tile sample)."""
    L = len(ref["x"])
    out = []
    for name, got, share in (("dw", dw, lambda l: ref["ds"][l][:, None] * ref["x"][l]),
                             ("db", db, lambda l: ref["g"][l])):
        score = torch.stack([(share(l).abs() / flo[name][l]).amax(1) for l in range(L)]).amax(0)
        bsel = int(score.argmax())
        wrong = ref[name] - torch.stack([share(l)[bsel] for l in range(L)])
        out.append(_bad(got, wrong, flo[name]))
    return out


# ---------------------------------------------------------------------------------------------------------------
# 2. the plan pinned to the library

def _kernel_name(raw):
    """'void dir::cross_fwd_kernel<4, 8, false>(float const*, ...)' -> 'cross_fwd_kernel<4,8,false>'."""
    name = raw.split("(")[0]
    if name.startswith("void "):
        name = name[5:]
    return name.replace("dir::", "").replace(" ", "")


@gpu
def test_cross_plan_matches_launched_kernels(pkg, cuda):
    from torch.profiler import ProfilerActivity, profile
    lib = _lib().lib()
    data = {dl: _data(37, *dl, seed=dl[0] * 64 + dl[1]) for dl in PAIRS}
    counts = []
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for dl in PAIRS:
            x0, w, b, dy = data[dl]
            _, s, nf = _fwd(x0, w, b)
            n0 = lib.dir_launch_count()
            _bwd(x0, w, b, dy, s)
            counts.append((nf, int(lib.dir_launch_count() - n0)))
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "cross_" in e.name),
                key=lambda e: e.time_range.start)
    names = [_kernel_name(e.name) for e in ev]
    # one case = one forward kernel and the backward's launches after it
    starts = [i for i, n in enumerate(names) if n.startswith("cross_fwd_kernel")] + [len(names)]
    got = [names[a:e] for a, e in zip(starts, starts[1:])]
    want = [sum(_kernels(d, L), []) for d, L in PAIRS]
    wrong = [(dl, g, w_) for dl, g, w_ in zip(PAIRS, got, want) if g != w_]
    assert len(got) == len(want) and not wrong, (len(got), len(want), wrong[:5])
    for (d, L), (nf, nb) in zip(PAIRS, counts):
        assert nf == 1 and nb == (3 if _cross_plan(d, L)[1][0] == "twopass" else 2), (d, L, nf, nb)


# ---------------------------------------------------------------------------------------------------------------
# 3-5. parity, exact properties and negative controls at every case

@gpu
@pytest.mark.parametrize("B,d,L", PARITY_CASES)
def test_cross_paths_parity(pkg, cuda, B, d, L):
    x0, w, b, dy = _data(B, d, L, seed=B * 65536 + d * 64 + L, heavy_tail=B == BIG_B)
    xL, s, nf = _fwd(x0, w, b)
    xL2, s2, _ = _fwd(x0, w, b)
    dx0, dw, db, nb = _bwd(x0, w, b, dy, s)
    again = _bwd(x0, w, b, dy, s)
    recomputed = _bwd(x0, w, b, dy, None)
    torch.cuda.synchronize()
    assert nf == 1 and nb == (3 if _cross_plan(d, L)[1][0] == "twopass" else 2)
    assert torch.equal(xL, xL2) and torch.equal(s, s2), "two forward runs must be bit-identical"
    for a, c, r in zip((dx0, dw, db), again[:3], recomputed[:3]):
        assert torch.equal(a, c), "two backward runs must be bit-identical"
        # the forward's p_l and the ring / fused recompute are the same fmaf chain and warp_sum over the same
        # zero-padded w; the two-pass backward ignores s
        assert torch.equal(a, r), "saved and recomputed p_l must give bit-identical gradients"

    ref, flo = _reference(x0, w, b, dy, per_sample=True)
    _check_all(dict(xL=xL, s=s, dx0=dx0, dw=dw, db=db), ref, flo, (B, d, L))
    if B > 1:       # one sample's a = dy . x0 may itself be near zero; of 37 the largest term is chosen
        assert _controls_dx0(dx0, ref, flo, w) > 0, "the bound must see a dropped w_{L-1} term of column d - 1"
    if L == 17:
        wrong = ref["dw"].clone()
        wrong[16] = ref["dw"][15]
        assert _bad(dw, wrong, flo["dw"]) > 0, "the bound must see a lost l0 = 16 chunk"
    if B == BIG_B:
        bad_dw, bad_db = _controls_sample(dw, db, ref, flo)
        assert bad_dw > 0 and bad_db > 0, "the bound must see one dropped sample"


@gpu
@pytest.mark.parametrize("d,L", BIG)
def test_cross_paths_exact(pkg, cuda, d, L):
    """w = 0: x_L = x0 + sum_l b_l exactly (the kernel sums b in layer order and c_L stays 1); dy = 0: every
    gradient is exactly zero."""
    B = 37
    x0, w, b, dy = _data(B, d, L, seed=d * 64 + L + 7)
    zw = torch.zeros_like(w)
    xL, s, _ = _fwd(x0, zw, b)
    beta = torch.zeros(d, device="cuda")
    for l in range(L):
        beta = beta + b[l]
    assert torch.equal(xL, x0 + beta), "KAT-4"
    assert bool((s == 0).all())
    _, s, _ = _fwd(x0, w, b)
    for sv in (s, None):
        dx0, dw, db, _ = _bwd(x0, w, b, torch.zeros_like(dy), sv)
        assert bool((dx0 == 0).all()) and bool((dw == 0).all()) and bool((db == 0).all())


@gpu
@pytest.mark.parametrize("d,L", [(4, 2), (51, 8), (1024, 32)])
def test_cross_paths_empty_batch(pkg, cuda, d, L):
    L_ = _lib()
    lib = L_.lib()
    w, b = _data(1, d, L, seed=3)[1:3]
    dw, db = _poisoned((L, d)), _poisoned((L, d))
    L_.check(lib.dir_cross_bwd(None, L_.ptr(w), L_.ptr(b), None, None, 0, d, L, None, L_.ptr(dw), L_.ptr(db), None,
                               0, _stream()), "dir_cross_bwd")
    torch.cuda.synchronize()
    assert bool((dw == 0).all()) and bool((db == 0).all())


# ---------------------------------------------------------------------------------------------------------------
# 6. alignment

def _offset(t):
    """A copy of t whose data pointer is 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, device=t.device, dtype=t.dtype)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


@gpu
@pytest.mark.parametrize("d,L", [(128, 3), (1024, 17)])
def test_cross_misaligned_refused_when_d_is_a_multiple_of_4(pkg, cuda, d, L):
    lib = _lib().lib()
    x0, w, b, dy = _data(37, d, L, seed=11)
    _, s, _ = _fwd(x0, w, b)
    torch.cuda.synchronize()
    n0 = lib.dir_launch_count()
    with pytest.raises(ValueError, match="alignment"):
        _fwd(_offset(x0), w, b)
    with pytest.raises(ValueError, match="alignment"):
        _bwd(_offset(x0), w, b, dy, s)
    with pytest.raises(ValueError, match="alignment"):
        _bwd(x0, w, b, _offset(dy), s)
    assert lib.dir_launch_count() == n0


@gpu
@pytest.mark.parametrize("d,L", [(51, 2), (429, 9)])
def test_cross_misaligned_computed_when_d_is_not(pkg, cuda, d, L):
    assert d % 4 and _cross_plan(d, L)[1][0] == ("fused" if L <= 8 else "twopass")
    x0, w, b, dy = _data(37, d, L, seed=12)
    xo, dyo = _offset(x0), _offset(dy)
    xL, s, _ = _fwd(xo, w, b)
    dx0, dw, db, _ = _bwd(xo, w, b, dyo, s)
    torch.cuda.synchronize()
    ref, flo = _reference(x0, w, b, dy)
    _check_all(dict(xL=xL, s=s, dx0=dx0, dw=dw, db=db), ref, flo, (d, L))
