"""K1's fused TopK epilogues, bit for bit, on rows built to hit their hard cases.

Reference: ``ops.encode_dense`` on the same packed operands (the fused epilogues run the same MMA
sequence, so its fp32 values are the ones they select from).  From that matrix the reference takes,
per row:

* the k largest values in the order of the order-preserving integer image of the float (-0.0 sorts
  below +0.0; every case asserts that no value tied with the k-th one has the other sign of zero, so
  float comparison, which the epilogues use, gives the same answer);
* ties at the k-th value to the lowest feature index;
* never NaN;
* rows with fewer than k non-NaN values padded with (-inf, -1).

Every call is checked exactly: equal index sets, ``val`` bit-identical to the reference values at the
returned indices, every index in [-1, F), padding slots exactly (-inf, -1).

Rows are built exactly: row r of x combines a few one-hot vectors with power-of-two coefficients, and
the matching columns of W hold small integers (exact in bf16), so pre[r, :] is a designed pattern with
no rounding.  One packed batch carries every row family side by side, in every TMEM lane quarter and
both halves of a CTA pair.  NaN features come from NaN encoder rows, which reach every row of a call,
so they get calls of their own.  Each case asserts its precondition on the ``encode_dense`` matrix
first, so that no case can silently test nothing.

Forms, reached by shape: the scanner / selector kernel (k <= 32, B < 1024 with an explicit nsplit),
the CTA-pair kernel (k <= 32, B >= 1024) and the one-warp ``<128, 2>`` kernel (33 <= k <= 64), each
with nsplit = 1 and with an F-split merged by ``topk_merge_kernel``; the single-CTA and pair kernels
also on identical operands through ``wsae_debug_encode_variant``.

The whole file (43 calls) takes 6.6 s on a B200 at a 1000 W power limit.  At the parent of the
change that added it, 37 of its 40 fused cases failed: the all-+0.0 row (a +0.0 floor), the NaN
group and NaN first tile under the floor, padding indices out of rows with fewer than k valid values,
a dropped +inf at k > 32, and tied -1s lost when larger values came later in the row.
"""

import pytest
import torch

pytestmark = pytest.mark.gpu

NINF_BITS = 0xFF800000 - (1 << 32)   # -inf as a signed int32 bit pattern

# x column of each structured W column (the rest of W, from column 16 on, is Gaussian)
C_HI, C_LO, C_ZERO, C_P7, C_P37, C_P257, C_KTH0, C_FLOOR, C_INF, C_LATE = range(10)
FAMILIES = ("gauss", "rising", "falling", "p7", "p37", "p257", "equal", "kth_zero", "floor32",
            "inf", "nan_row", "late_max")


def _ops():
    from whisper_sae_b200 import ops
    return ops


@pytest.fixture
def encode_variant():
    """Forces the k <= 32 epilogue (2 = single CTA, 3 = CTA pair) and restores the per-batch choice."""
    lib = _ops()._lib.load()
    try:
        yield lib.wsae_debug_encode_variant
    finally:
        lib.wsae_debug_encode_variant(0)


def _nan_features(mode, F, k, ns_eff):
    n_tiles = (F + 255) // 256
    if mode is None:
        return torch.zeros(F, dtype=torch.bool)
    nan = torch.zeros(F, dtype=torch.bool)
    if mode == "group8":          # one aligned group of 8 in the first tile
        nan[8:16] = True
    elif mode == "tile0":         # the whole first tile of the (only) work item
        nan[:256] = True
    elif mode == "split_tile":    # the whole first tile of F-split 1
        t0 = (n_tiles + ns_eff - 1) // ns_eff
        nan[t0 * 256:(t0 + 1) * 256] = True
    elif mode == "sparse":        # every row keeps fewer than k non-NaN values
        nan[:] = True
        keep = k // 2
        if keep:
            nan[(torch.arange(keep) * F) // keep + (F // keep) // 2] = False
    else:
        raise ValueError(mode)
    return nan


def _operands(B, d, F, k, terms, *, nan_mode=None, ns_eff=1, bias=0.0, rot=0, seed=0):
    """Packed operands plus, per family, the rows that carry it."""
    ops = _ops()
    g = torch.Generator().manual_seed(seed)
    f = torch.arange(F)
    nan = _nan_features(nan_mode, F, k, ns_eff)
    w = torch.zeros(F, d)
    w[:, C_HI] = (f // 256).float()                 # 256 * hi + lo = f
    w[:, C_LO] = (f % 256).float()
    w[:, C_P7] = (f % 7).float()                    # ties across tiles, splits and pair halves
    w[:, C_P37] = (f % 37).float()
    w[:, C_P257] = (f % 257).float()
    # k-th largest = +0.0: k // 2 positives, k - k // 2 + 4 zeros, -1 elsewhere, spread over F
    n_pos, n_zero = k // 2, k - k // 2 + 4
    pos = (torch.arange(n_pos + n_zero) * F) // (n_pos + n_zero)
    pos = pos[torch.randperm(len(pos), generator=g)]
    col = torch.full((F,), -1.0)
    col[pos[:n_pos]] = torch.arange(1, n_pos + 1).float()
    col[pos[n_pos:]] = 0.0
    w[:, C_KTH0] = col
    # first tile: group g of 8 has maximum 100 + g at its first column, -1 elsewhere, and a 50 at column
    # 3; -2 after it.  The 32 largest values are 100 .. 131, so at k = 32 the floor (100) is exact; with
    # NaN features 8..15 (group 1) the 32nd largest becomes the 50, below the floor of the other groups.
    col = torch.full((F,), -2.0)
    first = f < 256
    col[first] = -1.0
    col[first & (f % 8 == 0)] = 100.0 + (f[first & (f % 8 == 0)] // 8).float()
    col[3] = 50.0
    w[:, C_FLOOR] = col
    # ties first, larger values last: -1 everywhere but k // 2 distinct positives near the end of the row.
    # The k-th largest is a -1; a select that has already resolved the -1 ties meets the positives later.
    col = torch.full((F,), -1.0)
    col[F - 1 - 3 * torch.arange(k // 2)] = 2.0 + torch.arange(k // 2).float()
    w[:, C_LATE] = col
    # one +inf pre-activation (4 * 2^127 overflows), at a non-NaN feature in the upper half
    valid = (~nan).nonzero().flatten()
    f_inf = int(valid[valid >= F // 2][0]) if bool((valid >= F // 2).any()) else (int(valid[0]) if len(valid) else None)
    if f_inf is not None:
        w[f_inf, C_INF] = 2.0 ** 127
    w[:, 16:] = (torch.randn(F, d - 16, generator=g) / d ** 0.5).bfloat16().float()
    w[nan] = float("nan")

    x = torch.zeros(B, d)
    rows = {fam: [] for fam in FAMILIES}
    for r in range(B):
        fam = FAMILIES[(r + rot) % len(FAMILIES)]
        rows[fam].append(r)
        if fam == "gauss":
            x[r, 16:] = torch.randn(d - 16, generator=g)
        elif fam in ("rising", "inf"):
            x[r, C_HI], x[r, C_LO] = 256.0, 1.0
            if fam == "inf":
                x[r, C_INF] = 4.0
        elif fam == "falling":
            x[r, C_HI], x[r, C_LO] = -256.0, -1.0
        elif fam == "p7":
            x[r, C_P7] = 1.0
        elif fam == "p37":
            x[r, C_P37] = 2.0
        elif fam == "p257":
            x[r, C_P257] = 1.0
        elif fam == "kth_zero":
            x[r, C_KTH0] = 1.0
        elif fam == "floor32":
            x[r, C_FLOOR] = 1.0
        elif fam == "late_max":
            x[r, C_LATE] = 1.0
        elif fam == "nan_row":
            x[r] = float("nan")
        # "equal": x = 0, so every pre-activation is the bias
    b = torch.full((F,), bias)
    a_p = ops.pack_activations(x.cuda(), None, terms)
    w_p = ops.pack_encoder(w.cuda(), b.cuda(), terms)
    return a_p, w_p, rows, nan, f_inf


def _keys(pre):
    """Order-preserving integer image of the floats (int64 in [0, 2^32)); NaN -> -1."""
    bits = pre.view(torch.int32).long()
    key = torch.where(bits < 0, ~bits, bits + (1 << 31))
    return key.masked_fill(torch.isnan(pre), -1)


def _reference(pre, k):
    """Reference indices [B, k] (sorted) and the number of non-NaN values per row."""
    order = torch.sort(_keys(pre), dim=1, descending=True, stable=True).indices[:, :k]
    n_valid = (~torch.isnan(pre)).sum(1)
    want = torch.where(torch.arange(k, device=pre.device) < n_valid[:, None], order, -1)
    return want, n_valid


def _check_exact(idx, val, pre, k, what):
    B, F = pre.shape
    want, n_valid = _reference(pre, k)
    full = n_valid >= k
    # the k-th value's ties share its sign of zero (float order == key order at the k-th position)
    kth = pre.gather(1, want[:, k - 1:].clamp_min(0))
    tied = (pre == kth) & full[:, None]
    assert torch.equal(pre.view(torch.int32)[tied], kth.expand_as(pre).view(torch.int32)[tied]), \
        f"{what}: +0.0 and -0.0 tie at the k-th value (the case is ill-posed)"
    got = idx.long()
    assert bool(((got >= -1) & (got < F)).all()), \
        f"{what}: indices outside [-1, F): {got[(got < -1) | (got >= F)].unique()[:8].tolist()}"
    gs, ws = torch.sort(got, 1).values, torch.sort(want, 1).values
    bad = (gs != ws).any(1)
    assert not bool(bad.any()), \
        f"{what}: {int(bad.sum())} rows differ, first row {int(bad.nonzero()[0])}"
    ok = got >= 0
    ref_val = pre.gather(1, got.clamp_min(0))
    assert torch.equal(val.view(torch.int32)[ok], ref_val.view(torch.int32)[ok]), \
        f"{what}: values are not bit-identical to the encode_dense pre-activations"
    assert bool((val.view(torch.int32)[~ok] == NINF_BITS).all()), f"{what}: padding value is not -inf"


def _first_tile_floor(pre_rows, t0, F):
    """The epilogue's floor on the first tile of an item as the parent code computed it: min over the
    8-column groups of their max, all-NaN groups skipped.  Returns (floor, any all-NaN group)."""
    tile = pre_rows[:, t0 * 256:min(F, t0 * 256 + 256)]
    g = tile.reshape(tile.shape[0], -1, 8)
    all_nan = torch.isnan(g).all(2)
    gmax = torch.where(torch.isnan(g), float("-inf"), g).amax(2).masked_fill(all_nan, float("inf"))
    return gmax.amin(1), bool(all_nan.any())


def _preconditions(pre, rows, k, F, bias, nan_mode, nan, f_inf, ns_eff):
    """What each case is there to exercise must be present in the encode_dense matrix."""
    cpu_nan = nan.to(pre.device)
    want, n_valid = _reference(pre, k)
    r = rows["rising"]
    if r:
        v = pre[r][:, ~cpu_nan]
        assert bool((v[:, 1:] > v[:, :-1]).all()), "rising rows must rise strictly"
    if rows["inf"] and f_inf is not None:
        assert bool((pre[rows["inf"], f_inf] == float("inf")).all()), "the +inf pre-activation overflowed differently"
    if bias == 0.0 and nan_mode is None:
        eq = pre[rows["equal"]]
        if len(rows["equal"]):
            # an all-zero row: every value is +0.0, not -0.0, and so is the first tile's floor unless
            # the tile holds padding columns (F < 256), whose -inf make the floor useless
            assert bool((eq.view(torch.int32) == 0).all()), "the all-zero row is not all +0.0"
            if F >= 256:
                floor, _ = _first_tile_floor(eq, 0, F)
                assert bool((floor.view(torch.int32) == 0).all()), "the first tile's floor is not +0.0"
        kz = rows["kth_zero"]
        if kz:
            kth = pre[kz].gather(1, want[kz, k - 1:])
            assert bool((kth.view(torch.int32) == 0).all()), "the k-th largest of kth_zero rows is not +0.0"
            assert bool((pre[kz] < 0).any(1).all()), "kth_zero rows need negatives"
        lm = rows["late_max"]
        if lm:
            assert bool((pre[lm].gather(1, want[lm, k - 1:]) == -1.0).all()), "late_max rows must tie at -1"
    if nan_mode == "group8":
        fr = rows["floor32"]
        assert k == 32 and fr and F >= 256
        floor, has_nan_group = _first_tile_floor(pre[fr], 0, F)
        kth = pre[fr].gather(1, want[fr, k - 1:]).flatten()
        assert has_nan_group and bool((kth < floor).all()), "the 32nd value must lie below the floor"
    if nan_mode in ("tile0", "split_tile"):
        t0 = 0 if nan_mode == "tile0" else ((F + 255) // 256 + ns_eff - 1) // ns_eff
        assert bool(torch.isnan(pre[:, t0 * 256:t0 * 256 + 256]).all()), "the item's first tile must be all NaN"
        assert bool((n_valid[rows["rising"]] >= k).all())
    if nan_mode == "sparse":
        assert F % 256 != 0 and bool((n_valid < k).all()), "every row must have fewer than k valid values"


# (k, terms, B, F, d, nsplit, nan_mode, bias, rot, variants); variants () = the default choice
CASES = [
    # scanner / selector, single CTA (B < 1024, explicit nsplit)
    (32, 1, 1000, 3072, 384, 1, None, 0.0, 0, ()),
    (32, 1, 1000, 3072, 384, 3, None, 0.0, 0, ()),
    (17, 3, 127, 3000, 64, 1, None, 0.0, 0, ()),
    (4, 6, 127, 3000, 64, 4, None, 0.0, 0, ()),
    (1, 1, 1, 3072, 64, 1, None, 0.0, FAMILIES.index("equal"), ()),
    (1, 1, 1, 200, 64, 1, None, 0.0, FAMILIES.index("kth_zero"), ()),
    (31, 1, 127, 3072, 384, 2, None, 0.25, 0, ()),
    (17, 1, 1000, 40960, 1280, 1, None, 0.0, 0, ()),
    (17, 1, 1000, 40960, 1280, 8, None, 0.0, 0, ()),
    (32, 1, 127, 3072, 64, 1, "group8", 0.0, 0, ()),
    (32, 1, 127, 3072, 64, 3, "group8", 0.0, 0, ()),
    (32, 1, 127, 3072, 64, 1, "tile0", 0.0, 0, ()),
    (17, 3, 127, 3000, 64, 4, "split_tile", 0.0, 0, ()),
    (31, 1, 127, 200, 64, 1, "sparse", 0.0, 0, ()),
    (8, 1, 127, 3000, 64, 12, "sparse", 0.0, 0, ()),
    # CTA pair (B >= 1024)
    (32, 1, 4096, 3072, 384, 1, None, 0.0, 0, ()),
    (32, 1, 4096, 3072, 384, 4, None, 0.0, 0, ()),
    (32, 3, 1030, 3000, 384, 1, None, 0.0, 0, ()),
    (31, 6, 1030, 3072, 64, 3, None, 0.0, 0, ()),
    (4, 1, 4096, 40960, 1280, 1, None, 0.0, 0, ()),
    (17, 1, 1030, 3072, 64, 2, None, 0.25, 0, ()),
    (32, 1, 1030, 3072, 64, 1, "group8", 0.0, 0, ()),
    (32, 3, 1030, 3072, 64, 1, "tile0", 0.0, 0, ()),
    (32, 1, 1030, 3072, 64, 4, "split_tile", 0.0, 0, ()),
    (31, 1, 1030, 200, 64, 1, "sparse", 0.0, 0, ()),
    (17, 6, 1030, 3000, 64, 12, "sparse", 0.0, 0, ()),
    # <128, 2> (33 <= k <= 64)
    (33, 1, 127, 3072, 384, 1, None, 0.0, 0, ()),
    (33, 1, 127, 3072, 384, 3, None, 0.0, 0, ()),
    (48, 3, 1000, 3000, 64, 4, None, 0.0, 0, ()),
    (63, 6, 127, 3000, 64, 1, None, 0.0, 0, ()),
    (64, 1, 4096, 40960, 1280, 1, None, 0.0, 0, ()),
    (64, 1, 1030, 3000, 64, 2, None, 0.25, 0, ()),
    (64, 1, 127, 3000, 64, 1, "sparse", 0.0, 0, ()),
    (48, 3, 127, 200, 64, 1, "sparse", 0.0, 0, ()),
    (33, 1, 127, 3072, 64, 1, "tile0", 0.0, 0, ()),
    # single CTA and pair on identical operands
    (32, 1, 1000, 3072, 384, 1, None, 0.0, 0, (2, 3)),
    (17, 1, 4096, 3072, 384, 2, None, 0.0, 0, (2, 3)),
    (32, 6, 127, 3072, 64, 1, "group8", 0.0, 0, (2, 3)),
    (31, 1, 127, 200, 64, 1, "sparse", 0.0, 0, (2, 3)),
    (4, 3, 1030, 3000, 64, 3, "split_tile", 0.0, 0, (2, 3)),
]


def _case_id(c):
    k, terms, B, F, d, ns, mode, bias, rot, variants = c
    s = f"k{k}-t{terms}-B{B}-F{F}-d{d}-ns{ns}"
    s += f"-{mode}" if mode else ""
    s += f"-bias{bias}" if bias else ""
    s += f"-rot{rot}" if rot else ""
    s += "-variants" + "".join(map(str, variants)) if variants else ""
    return s


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_k1_fused_epilogue_exact(case, encode_variant):
    k, terms, B, F, d, ns, mode, bias, rot, variants = case
    ops = _ops()
    lib = ops._lib.load()
    assert ops.encode_route(B, F, k, ns) == "fused"
    ns_eff = lib.wsae_encode_effective_splits(F, ns)
    assert ns_eff == ns, "the case must run the F-split it names"
    a, w, rows, nan, f_inf = _operands(B, d, F, k, terms, nan_mode=mode, ns_eff=ns_eff, bias=bias, rot=rot,
                                       seed=k * 131 + B + F + d + ns)
    pre = ops.encode_dense(a, w, B, F, d, terms)
    torch.cuda.synchronize()
    _preconditions(pre, rows, k, F, bias, mode, nan, f_inf, ns_eff)
    for v in variants or (0,):
        encode_variant(v)
        idx, val = ops.encode_topk(a, w, B, F, d, terms, k, nsplit=ns)
        torch.cuda.synchronize()
        _check_exact(idx, val, pre, k, f"variant {v}")


@pytest.mark.parametrize("k,F,mode", [(31, 200, "sparse"), (64, 3000, "sparse"), (32, 3072, "group8")])
def test_k1_dense_route_agrees_with_reference(k, F, mode):
    """Cross-check of the reference rule itself: the dense route (radix select on the same keys) returns
    what the reference does on the same adversarial operands."""
    ops = _ops()
    B, d = 127, 64
    assert ops.encode_route(B, F, k) == "dense"
    a, w, rows, nan, f_inf = _operands(B, d, F, k, 1, nan_mode=mode, seed=7)
    pre = ops.encode_dense(a, w, B, F, d, 1)
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k)
    torch.cuda.synchronize()
    _check_exact(idx, val, pre, k, "dense route")
