"""The gather aggregation kernel (``k_aggregate``, dfw_aggregate.cu) bit for bit against the exact CPU oracle, on every one of
its 72 instantiations.

The kernel adds each row's neighbours in CSR order in fp32 with round-to-nearest (``acc += x``, or ``acc = fma(x, s, acc)``
with a per-source scale), then writes ``fma(acc, row_scale, addend)`` or ``acc * row_scale`` with one rounding to the output
type.  ``oracle_csr_aggregate_ex_f32`` performs the same operations in the same order with correctly rounded libm ``fmaf``,
so every output must match to the bit: signed zeros, subnormals and overflow to infinity included.  NaN is compared by
position only (its payload is not part of the contract).

The row width picks the instantiation ``k_aggregate<T, LANES, VPL, HAS_ADD, EXACT, HAS_SRC>``: ``nvec = H * size / 16``
vectors per row go to LANES lanes with VPL vectors each, EXACT when ``nvec == LANES * VPL``.  The three entry forms (sum
or mean, with an addend, per-source scales) give the (HAS_ADD, HAS_SRC) pairs.  Each case asserts from torch.profiler
which instantiation ran.  The graphs put per-group edge counts on the kernel's column-window boundaries, empty rows at
both ends of a group's block and in runs longer than it, a row of over 5 000 edges, ragged last warp steps, and CTAs that
take three or more chunks.  Every raw-ABI output sits inside sentinel-filled guard bands.  No case hands the kernel a
column index outside its source rows: the kernel has no bounds check (range errors are ``CSRGraph.check()``'s job)."""
import re

import numpy as np
import pytest
import torch

from helpers import Arena, launched_kernels, record
from oracle import csr_aggregate_ex

F32, BF16 = torch.float32, torch.bfloat16
NUM_SMS = 148   # dfw_common.cuh kNumSMs
WARPS = 32      # dfw_aggregate.cu kAggThreads / 32: row blocks per chunk
MAX_ROW_BYTES = 2048

# (dtype, H, exact): every (LANES, VPL) shape of dispatch(), each with a row that fills it exactly and ragged rows
TABLE = ([(F32, h, True) for h in (16, 32, 64, 128, 256, 512)]
         + [(F32, h, False) for h in (4, 12, 20, 36, 60, 96, 132, 260, 508)]
         + [(BF16, h, True) for h in (32, 64, 128, 256, 512, 1024)]
         + [(BF16, h, False) for h in (8, 24, 40, 72, 136, 264, 520, 1016)])
FORMS = ("mean", "add", "scaled_add", "src")   # -> (HAS_ADD, HAS_SRC) = (0, 0), (1, 0), (1, 0), (0, 1)


def _tid(dt, h):
    return f"{'f32' if dt == F32 else 'bf16'}_h{h}"


def nvec_of(dt, H):
    return H * (4 if dt == F32 else 2) // 16


def shape_of(nvec):
    """dispatch() in dfw_aggregate.cu: (LANES, VPL) of a row of nvec 16-byte vectors."""
    for limit, lanes, vpl in ((4, 4, 1), (8, 8, 1), (16, 16, 1), (32, 32, 1), (64, 32, 2), (128, 32, 4)):
        if nvec <= limit:
            return lanes, vpl
    raise ValueError(nvec)


def k_u(lanes, vpl):
    """Source rows per batch (the kernel's kU): a column window of LANES holds LANES / kU batches."""
    return min(2 if vpl >= 4 else (4 if vpl == 2 else 8), lanes)


def pick_rows_per_group(N, E, lanes, groups):
    """Python copy of pick_rows_per_group in dfw_aggregate.cu (rows R per lane group)."""
    deg = E / N if N > 0 else 0.0
    hi = int(192.0 / (deg + 1.0))
    hi = max(1, min(hi, min(12, lanes - 1)))
    lo = max(1, (hi * 2 + 2) // 3)
    best, best_eff = hi, -1.0
    for R in range(hi, lo - 1, -1):
        chunk_rows = R * groups * WARPS
        chunks = (N + chunk_rows - 1) // chunk_rows
        waves = (chunks + NUM_SMS - 1) // NUM_SMS
        eff = N / (waves * NUM_SMS * chunk_rows)
        if eff > best_eff + 0.02:
            best_eff, best = eff, R
    return best


def instantiation(dt, H, form):
    lanes, vpl = shape_of(nvec_of(dt, H))
    return ("float" if dt == F32 else "__nv_bfloat16", lanes, vpl, form in ("add", "scaled_add"), nvec_of(dt, H) == lanes * vpl,
            form == "src")


def _kernel_args(names):
    """Template arguments of every k_aggregate launch, normalised to the tuple of instantiation()."""
    out = []
    for n in names:
        m = re.search(r"k_aggregate<([^<>]*)>", n)
        if not m:
            continue
        a = [re.sub(r"^\((int|bool)\)", "", s.strip()) for s in m.group(1).split(",")]  # "(int)16", "(bool)0" or "16", "false"
        b = [{"true": True, "false": False, "1": True, "0": False}[s] for s in a[3:]]
        out.append((a[0], int(a[1]), int(a[2]), *b))
    return out


# ---- graphs -----------------------------------------------------------------------------------------------------------------
def _group_counts(rowptr, R):
    n = rowptr.size - 1
    starts = np.arange(0, n, R)
    return rowptr[np.minimum(starts + R, n)] - rowptr[starts]


def _ragged_last_step(n, R, groups):
    """The last warp step has lane groups past N (they `continue`) next to groups that work."""
    rem = n % (R * groups)
    return groups > 1 and rem > 0 and -(-rem // R) < groups


def _fill_block(rng, deg, r0, nr, c):
    if c == 0:
        return
    live = rng.random(nr) > 0.3
    if not live.any():
        live[rng.integers(nr)] = True
    idx = np.flatnonzero(live)
    deg[r0 + idx] = rng.multinomial(c, np.full(idx.size, 1.0 / idx.size))


def _columns(rng, rowptr, n_src):
    """Random columns in [0, n_src) plus forced self loops, duplicate edges and x / -x neighbour pairs (rows 2m, 2m+1)."""
    n, E = rowptr.size - 1, int(rowptr[-1])
    col = rng.integers(0, n_src, E).astype(np.int32)
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    first = np.zeros(E, bool)
    first[rowptr[:-1][np.diff(rowptr) > 0]] = True
    loops = (rng.random(E) < 0.03) & (rows < n_src)
    col[loops] = rows[loops]
    dup = np.flatnonzero((rng.random(E) < 0.05) & ~first)
    col[dup] = col[dup - 1]
    two = np.flatnonzero((np.diff(rowptr) >= 2) & (rng.random(n) < 0.15))
    m = rng.integers(0, max(n_src // 2, 1), two.size)
    if n_src >= 2:
        col[rowptr[two]], col[rowptr[two] + 1] = 2 * m, 2 * m + 1
    return col


def boundary_graph(lanes, vpl, seed=0):
    """A CSR whose lane groups (blocks of R rows) stream edge counts on every window boundary of the kernel: 0, 1, kU - 1,
    kU, kU + 1, LANES - 1, LANES, LANES + 1, 2 LANES, 2 LANES + 1; plus a block of one row with 5 200 edges, a run of empty
    blocks, and N chosen so that the last warp step is ragged.  Returns (rowptr, col, R)."""
    rng = np.random.default_rng(seed + 1000 * lanes + vpl)
    groups = 32 // lanes
    ku = k_u(lanes, vpl)
    special = sorted({0, 1, ku - 1, ku, ku + 1, lanes - 1, lanes, lanes + 1, 2 * lanes, 2 * lanes + 1})
    hub = 5200
    n = 2000
    while True:
        E = 6 * n + hub
        R = pick_rows_per_group(n, E, lanes, groups)
        if groups == 1 or _ragged_last_step(n, R, groups):
            break
        n += 1
    nblk = -(-n // R)
    counts = np.zeros(nblk, np.int64)
    fixed = np.zeros(nblk, bool)
    for i, c in enumerate(special):
        counts[2 + 2 * i] = c  # every other block, so each special count is one group's whole stream
        fixed[2 + 2 * i] = True
    z = 2 + 2 * len(special)
    fixed[z:z + 3] = True      # three empty blocks in a row: a run of empty rows longer than a group's block
    counts[z + 4] = hub
    fixed[z + 4] = True
    free = np.flatnonzero(~fixed)
    counts[free] = rng.multinomial(E - int(counts.sum()), np.full(free.size, 1.0 / free.size))
    deg = np.zeros(n, np.int64)
    for b in range(nblk):
        r0, nr = b * R, min(R, n - b * R)
        if b == z + 4:
            deg[r0 + nr // 2] = hub
        else:
            _fill_block(rng, deg, r0, nr, int(counts[b]))
    rowptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    assert int(rowptr[-1]) == E
    return rowptr, _columns(rng, rowptr, n), R


def random_graph(n, mean_deg, seed, n_src=None, empty=0.1):
    rng = np.random.default_rng(seed)
    deg = rng.poisson(mean_deg, n) if mean_deg > 0 else np.zeros(n, np.int64)
    deg[rng.random(n) < empty] = 0
    rowptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    return rowptr, _columns(rng, rowptr, n if n_src is None else n_src)


# ---- values -----------------------------------------------------------------------------------------------------------------
def _values(rng, shape, dt, special=True):
    """fp32 values exactly representable in dt: normals, whole rows of subnormals and of values near the fp32 maximum
    (their sums overflow), rows 2m + 1 = -(row 2m) for a tenth of the pairs (x + (-x) = +0), explicit +0 / -0, and, when
    `special`, a few NaN, +Inf and -Inf elements."""
    n = shape[0]
    x = rng.standard_normal(shape).astype(np.float32)
    if x.ndim == 2 and n > 0:
        kind = rng.random(n)
        x[kind < 0.06] *= np.float32(2.0 ** -136)                                          # subnormal
        big = (kind >= 0.06) & (kind < 0.12)
        x[big] = np.sign(x[big]) * rng.uniform(1.2e38, 3.3e38, x[big].shape).astype(np.float32)
        pairs = np.flatnonzero(rng.random(n // 2) < 0.1) * 2
        x[pairs[pairs + 1 < n] + 1] = -x[pairs[pairs + 1 < n]]
        z = rng.random(shape) < 0.02
        x[z] = np.where(rng.random(z.sum()) < 0.5, np.float32(0.0), np.float32(-0.0))
        if special and n >= 8:
            for v in (np.nan, np.nan, np.inf, -np.inf):
                x[rng.integers(n), rng.integers(shape[1])] = v
    return torch.from_numpy(x).to(dt).float().numpy()


def _scales(rng, n, deg=None):
    """Per-row fp32 scales: 1/deg, 0, negative, subnormal, 1 and arbitrary values."""
    s = (rng.standard_normal(n) * 2).astype(np.float32)
    k = rng.integers(0, 6, n)
    if deg is not None:
        s[k == 0] = (1.0 / np.maximum(deg, 1)).astype(np.float32)[k == 0]
    s[k == 1] = 0.0
    s[k == 2] = -np.abs(s[k == 2])
    s[k == 3] *= np.float32(2.0 ** -130)
    s[k == 4] = 1.0
    return s


# ---- launch and compare -----------------------------------------------------------------------------------------------------
def _cabi():
    from deep_fem_uav_wing.gnn import _cabi

    return _cabi


def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_kernel(form, rowptr, col, x, rs, ss, add, n_rows, dt):
    """One raw-ABI launch into a guarded output; returns (out, names of the launched kernels)."""
    cabi = _cabi()
    H = x.shape[1]
    E = int(rowptr[-1])
    d_rp, d_col = _dev(rowptr), (_dev(col) if E else None)
    d_x = _dev(x).to(dt)
    d_rs = _dev(rs) if form in ("mean", "scaled_add") else None
    d_ss = _dev(ss) if form == "src" else None
    d_add = _dev(add).to(dt) if form in ("add", "scaled_add") else None
    ar = Arena()
    out = ar.out((n_rows, H), dt)
    p = lambda t: None if t is None else t.data_ptr()
    stream = torch.cuda.current_stream().cuda_stream
    if form == "src":
        call = lambda: cabi.check(cabi.lib.dfw_sage_aggregate_scaled(d_rp.data_ptr(), p(d_col), d_ss.data_ptr(), d_x.data_ptr(),
                                                                     out.data_ptr(), n_rows, E, H, 0 if dt == F32 else 1, stream))
    else:
        call = lambda: cabi.check(cabi.lib.dfw_sage_aggregate(d_rp.data_ptr(), p(d_col), p(d_rs), d_x.data_ptr(), p(d_add),
                                                              out.data_ptr(), n_rows, E, H, 0 if dt == F32 else 1, stream))
    _, names = launched_kernels(call)
    ar.check(f"{form} {_tid(dt, H)}")
    return out.cpu(), names


def oracle_out(form, rowptr, col, x, rs, ss, add, n_rows, dt):
    ref = csr_aggregate_ex(rowptr, col, x, row_scale=rs if form in ("mean", "scaled_add") else None,
                           src_scale=ss if form == "src" else None, addend=add if form in ("add", "scaled_add") else None,
                           n_rows=n_rows)
    return torch.from_numpy(ref).to(dt)  # torch rounds fp32 -> bf16 to nearest even, as the kernel's store does


def assert_bits(name, got, ref):
    """Bit equality; NaN by position.  Returns (mismatches, NaN rows, non-finite rows)."""
    gn, rn = torch.isnan(got.float()), torch.isnan(ref.float())
    ib = torch.int32 if got.dtype == F32 else torch.int16
    diff = (got.view(ib) != ref.view(ib)) & ~(gn & rn)
    mism = int(diff.sum())
    nonfin = int((~torch.isfinite(ref.float())).any(dim=1).sum()) if ref.numel() else 0
    if mism:
        i = int(diff.flatten().nonzero()[0])
        raise AssertionError(f"{name}: {mism} of {got.numel()} elements differ from the oracle in their bits (first at flat index {i}: "
                             f"got {got.flatten()[i].item()!r} [{hex(int(got.view(ib).flatten()[i]) & 0xffffffff)}], "
                             f"oracle {ref.flatten()[i].item()!r} [{hex(int(ref.view(ib).flatten()[i]) & 0xffffffff)}])")
    return mism, nonfin


def check_case(gate, rowptr, col, dt, H, seed, n_src=None, forms=FORMS, expect_names=True, special=True):
    rng = np.random.default_rng(seed)
    n = rowptr.size - 1
    n_src = n if n_src is None else n_src
    x = _values(rng, (n_src, H), dt, special)
    deg = np.diff(rowptr)
    rs = _scales(rng, n, deg)
    ss = _scales(rng, n_src)
    add = _values(rng, (n, H), dt, special=False)
    seen, mism, nonfin, nans = [], {}, {}, {}
    for form in forms:
        if form == "src" and n_src != n:
            continue  # dfw_sage_aggregate_scaled is square: its source and destination rows are the same N
        got, names = run_kernel(form, rowptr, col, x, rs, ss, add, n, dt)
        ref = oracle_out(form, rowptr, col, x, rs, ss, add, n, dt)
        args = _kernel_args(names)
        if n > 0:
            assert args, f"{gate} {form}: torch.profiler saw no k_aggregate launch in {sorted(set(names))}"
            assert args == [instantiation(dt, H, form)], f"{gate} {form} {_tid(dt, H)}: launched {args}, expected {instantiation(dt, H, form)}"
        else:
            assert not args, f"{gate}: N = 0 launched {args}"
        seen += args
        mism[form], nonfin[form] = assert_bits(f"{gate} {form} {_tid(dt, H)}", got, ref)
        nans[form] = int(torch.isnan(ref.float()).sum())
    record(gate, dtype=str(dt), H=H, N=n, E=int(rowptr[-1]), bit_mismatches=mism, nonfinite_rows=nonfin, nan_elements=nans)
    return seen


@pytest.fixture(scope="module")
def cuda():
    from deep_fem_uav_wing.gnn import ops  # noqa: F401  (loads the library)

    return torch.device("cuda")


# ---- CPU: the table and the graphs are what they claim ----------------------------------------------------------------------
def test_table_covers_the_72_instantiations():
    want = {instantiation(dt, h, f) for dt, h, _ in TABLE for f in FORMS}
    assert len(want) == 72
    for dt, h, exact in TABLE:
        assert (nvec_of(dt, h) == np.prod(shape_of(nvec_of(dt, h)))) == exact
        assert nvec_of(dt, h) * 16 <= MAX_ROW_BYTES and h * (4 if dt == F32 else 2) % 16 == 0


@pytest.mark.parametrize("lanes,vpl", [(4, 1), (8, 1), (16, 1), (32, 1), (32, 2), (32, 4)])
def test_boundary_graphs_hit_every_window_boundary(lanes, vpl):
    rowptr, col, R = boundary_graph(lanes, vpl)
    n, E = rowptr.size - 1, int(rowptr[-1])
    assert R == pick_rows_per_group(n, E, lanes, 32 // lanes)
    ku = k_u(lanes, vpl)
    counts = set(_group_counts(rowptr, R).tolist())
    for c in (0, 1, ku - 1, ku, ku + 1, lanes - 1, lanes, lanes + 1, 2 * lanes, 2 * lanes + 1):
        assert c in counts, (lanes, vpl, R, c)
    deg = np.diff(rowptr)
    blocks = [deg[i:i + R] for i in range(0, n, R)]
    if R > 1:
        assert any(b[0] == 0 and b.sum() > 0 for b in blocks), "empty first row of a working block"
        assert any(b[-1] == 0 and b.sum() > 0 for b in blocks), "empty last row of a working block"
    runs = np.diff(np.flatnonzero(np.diff(np.concatenate([[1], (deg == 0).astype(int), [1]])) != 0))[::2]
    assert runs.max() > R, "a run of empty rows longer than a group's block"
    assert (deg == 1).any() and deg.max() > 5000
    rows = np.repeat(np.arange(n), deg)
    assert (col == rows).any(), "self loops"
    assert (np.diff(col)[np.diff(rows) == 0] == 0).any(), "duplicate edges"
    if lanes < 32:
        assert _ragged_last_step(n, R, 32 // lanes)
    assert col.min() >= 0 and col.max() < n


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt,h,exact", TABLE, ids=[_tid(d, h) for d, h, _ in TABLE])
def test_every_instantiation_is_bit_exact(cuda, dt, h, exact):
    lanes, vpl = shape_of(nvec_of(dt, h))
    rowptr, col, _ = boundary_graph(lanes, vpl)
    seen = check_case("aggregate_exact_boundary", rowptr, col, dt, h, seed=h)
    assert len(set(seen)) == 3 and len(seen) == 4


def _regime_graph(regime, lanes, seed):
    if regime == "deg0":
        return random_graph(777, 0, seed)
    if regime == "deg6":
        return random_graph(1531, 6, seed)
    if regime == "deg14":
        return random_graph(1187, 14, seed)
    if regime == "deg200":  # mean degree > 191: one row per lane group (R = 1)
        return random_graph(211, 200, seed, empty=0.02)
    n = {"n1": 1, "n2": 2, "lanes_minus_1": lanes - 1}[regime]
    return random_graph(n, 6, seed, empty=0.0)


REGIMES = ("deg0", "deg6", "deg14", "deg200", "n1", "n2", "lanes_minus_1")


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("dt,h,exact", TABLE, ids=[_tid(d, h) for d, h, _ in TABLE])
def test_degree_regimes_and_tiny_n_are_bit_exact(cuda, regime, dt, h, exact):
    lanes, _ = shape_of(nvec_of(dt, h))
    rowptr, col = _regime_graph(regime, lanes, seed=h)
    n, E = rowptr.size - 1, int(rowptr[-1])
    if regime == "deg0":
        assert E == 0  # launched with col = NULL
    if regime == "deg200":
        assert pick_rows_per_group(n, E, lanes, 32 // lanes) == 1
    check_case(f"aggregate_exact_{regime}", rowptr, col, dt, h, seed=h + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("dt,h", [(F32, 4), (F32, 20), (F32, 36), (F32, 68)], ids=["lanes4", "lanes8", "lanes16", "lanes32"])
def test_every_cta_takes_three_chunks(cuda, dt, h):
    lanes, vpl = shape_of(nvec_of(dt, h))
    groups = 32 // lanes
    R0 = min(12, lanes - 1)
    n = 3 * NUM_SMS * R0 * groups * WARPS + 12345
    rowptr, col = random_graph(n, 6, seed=lanes)
    R = pick_rows_per_group(n, int(rowptr[-1]), lanes, groups)
    chunks = -(-n // (R * groups * WARPS))
    assert chunks >= 3 * NUM_SMS, (R, chunks)
    check_case("aggregate_exact_three_chunks", rowptr, col, dt, h, seed=lanes, forms=("mean", "scaled_add", "src"))


@pytest.mark.gpu
@pytest.mark.parametrize("dt,h", [(F32, 12), (F32, 128), (BF16, 136), (BF16, 1024)], ids=lambda v: str(v))
def test_rectangular_sources_beyond_the_destination_rows(cuda, dt, h):
    """The partitioned layout (ops.aggregate_rows): columns index [own rows | halo rows], more rows than destinations."""
    n_rows, n_src = 1500, 2300
    rowptr, col = random_graph(n_rows, 8, seed=h, n_src=n_src)
    assert col.max() >= n_rows
    check_case("aggregate_exact_rectangular", rowptr, col, dt, h, seed=h, n_src=n_src, forms=("mean", "add", "scaled_add"))


@pytest.mark.gpu
def test_n0_writes_nothing_and_the_host_refuses_what_the_kernel_cannot_take(cuda):
    cabi = _cabi()
    lib = cabi.lib
    stream = torch.cuda.current_stream().cuda_stream
    rowptr = torch.zeros(1, dtype=torch.int32, device="cuda")
    ar = Arena()
    out = ar.out((0, 64), F32)
    _, names = launched_kernels(lambda: (cabi.check(lib.dfw_sage_aggregate(rowptr.data_ptr(), None, None, out.data_ptr(), None,
                                                                           out.data_ptr(), 0, 0, 64, 0, stream)),
                                         cabi.check(lib.dfw_sage_aggregate_scaled(rowptr.data_ptr(), None, None, out.data_ptr(),
                                                                                  out.data_ptr(), 0, 0, 64, 1, stream))))
    assert not _kernel_args(names)
    ar.check("N = 0")
    # refusals: errors on the host, no launch
    n = 4
    rp = torch.arange(n + 1, dtype=torch.int32, device="cuda")
    cl = torch.arange(n, dtype=torch.int32, device="cuda")
    for dt, H in ((F32, 516), (BF16, 1032)):  # rows of 2064 bytes: wider than the supported 2048
        x = torch.zeros(n, H, dtype=dt, device="cuda")
        o = torch.zeros_like(x)
        with pytest.raises(cabi.DfwError, match="wider than the supported 2048"):
            cabi.check(lib.dfw_sage_aggregate(rp.data_ptr(), cl.data_ptr(), None, x.data_ptr(), None, o.data_ptr(), n, n, H, 0 if dt == F32 else 1, stream))
    for dt, H in ((F32, 6), (BF16, 12)):  # row_bytes % 16 != 0
        x = torch.zeros(n, H, dtype=dt, device="cuda")
        with pytest.raises(cabi.DfwError, match="multiple of 16"):
            cabi.check(lib.dfw_sage_aggregate(rp.data_ptr(), cl.data_ptr(), None, x.data_ptr(), None, x.data_ptr(), n, n, H, 0 if dt == F32 else 1, stream))
    buf = torch.zeros(n * 64 + 4, device="cuda")
    o = torch.zeros(n, 64, device="cuda")
    with pytest.raises(cabi.DfwError, match="16-byte aligned"):  # x 8 bytes past an aligned address
        cabi.check(lib.dfw_sage_aggregate(rp.data_ptr(), cl.data_ptr(), None, buf[2:].data_ptr(), None, o.data_ptr(), n, n, 64, 0, stream))
    with pytest.raises(cabi.DfwError, match="src_scale is NULL"):
        cabi.check(lib.dfw_sage_aggregate_scaled(rp.data_ptr(), cl.data_ptr(), None, o.data_ptr(), o.data_ptr(), n, n, 64, 0, stream))
    assert torch.equal(o, torch.zeros_like(o))
    torch.cuda.synchronize()
