"""GPU parity of the conditioning path one kernel at a time -- the kernels that turn (t, y) into the FiLM table, and the two
fp32 kernels the validation and training paths rest on -- each against fp64 torch of the same operation on the same fp32
inputs:

  vdt_op_linear                  every (rows, K, N) the shipped networks' embedding MLP, FiLM projections and training
                                 backward produce (K = batch in the weight-gradient form, rows = 2 * Cout up to 1536),
                                 ragged and multi-slab edges, NaN sentinels around the output
  vdt_op_timestep_embedding(_ex) the fp64 path to 1 ulp of the oracle's formula; the fp32-t path against the oracle on fp32 t
                                 and against the exact fp32 rounding chain
  vdt_op_class_embed             int ids (0, 1, num_classes, out of range), multitag rows, SiLU at large |v|
  vdt_op_film_rows / multitag    the CFG interleave and the clamp; the hook-built FiLM table against training.py's forward
  vdt_op_attention_f32           the split-precision mode's attention: hi + lo against fp64 softmax attention
  vdt_op_groupnorm_train         GroupNorm -> FiLM -> SiLU -> dropout at the shapes training.py runs

Every test prints its worst measured value on a "PARITY" line; profiles/r10_conditioning_parity.txt holds them.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                               # fp32 unit roundoff
DT = {1: torch.float16, 0: torch.bfloat16}
U16 = {1: 2.0 ** -11, 0: 2.0 ** -8}
FMT = {1: "fp16", 0: "bf16"}

# Bars, each 2-5x the worst value measured over the cases of this file on a B200 at its 1000 W power limit
# (profiles/r10_conditioning_parity.txt); where the measured value is 0 the bar is the contract itself
LIN_C = 6.0           # linear: |out - ref| <= LIN_C * U * (sum_k |W_nk x_rk| + |b_n| + |ref|); measured 2.4 (1536x7x768, SiLU)
TEMB_F64_ULP = 1      # fp64-t embedding: ulps of the fp32 rounding of the oracle's fp64 value; measured 0
TEMB_F32_C = 8.0      # fp32-t embedding vs the oracle on fp32 t: |out - ref| <= TEMB_F32_C * U * (|angle| + 1); measured 3.5
TEMB_CHAIN_ULP = 3    # fp32-t embedding vs fp64 sin / cos of the fp32-chain angle, in ulps of the result; measured 1.43
CLS_C = 4.0           # class embedding: |out - ref| <= CLS_C * U * (|e| + |b| + sum |w y| + |ref|); measured 1.5
FILM_C = 1.0          # FiLM-table composition vs training.py's forward, in U * (sum_k |W_nk a_k| + |b_n|); measured 0
ATT_C = {1: 8.0, 0: 300.0}   # attention hi + lo: |o - ref| <= ATT_C * U * sum_k p_k |v_k| * (1 + max_k S_k) (+ the fp16
                             # pair's 2^-25 floor); measured fp16 3.2, bf16 96 (its lo carries 8 bits)
GN_ABS = 5e-7         # groupnorm_train: |out - ref| <= u16 |ref| + GN_ABS; measured 1.9e-7


@pytest.fixture(scope="module")
def L():
    from v_diffusion_b200 import _lib
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return _lib.lib()


def _p(t):
    return None if t is None else t.data_ptr()


def _check(L, rc):
    assert rc == 0, L.vdt_last_error().decode()


def _report(name, value):
    print(f"PARITY {name} {value:.3e}")


def _ulp32(x):
    """Spacing of fp32 numbers at |x| (x fp64, non-zero normal fp32 magnitudes)."""
    e = torch.floor(torch.log2(x.abs()))
    return torch.exp2(e - 23)


# ----------------------------------------------------------------------------------------------------------------- linear
def _res_couts(hid, mult, nrb):
    """Output channels of every ResidualBlock of unet.py in order (each has a fc of 2 * cout rows)."""
    chs = [hid * m for m in mult]
    lv = len(mult)
    out = []
    for i in range(lv):
        out += [chs[i]] * (nrb + (i != lv - 1))
    out += [chs[-1]] * 2
    for i in range(lv):
        out += [chs[i]] * (nrb + 1 + (i != 0))
    return out


# (hid, E, ch_multipliers, num_res_blocks, num_classes) of the shipped networks
NETS = {"cifar": (256, 1024, (1, 1, 1), 3, 10), "celeba": (192, 768, (1, 2, 3, 4), 3, 40), "mnist": (64, 256, (1, 2, 2), 1, 10)}
BATCHES = (1, 7, 8, 9, 128, 1536)


def _net_shapes():
    shapes = set()
    for hid, E, mult, nrb, ncls in NETS.values():
        couts = _res_couts(hid, mult, nrb)
        film_total = 2 * sum(couts)
        for B in BATCHES:
            # forward (unet.py:287-295, training.py:280-299, 355; plan.cu add_embedding_steps)
            shapes |= {(B, hid, E), (B, E, E), (B, ncls, E), (B, E, film_total)}
            for c in set(couts):
                shapes |= {(B, E, 2 * c),                 # fc
                           (B, 2 * c, E),                 # d emb_act = dfilm W
                           (2 * c, B, E)}                 # d W_fc = dfilm^T emb_act
            # backward of the embedding MLP (training.py:455-464), K = B in the weight-gradient form
            shapes |= {(E, B, ncls), (E, B, E), (E, B, hid)}
        shapes.add((ncls + 1, E, film_total))             # the sampler's per-class FiLM table
    return sorted(shapes)


LIN_NET = _net_shapes()
LIN_EDGE = [(r, k, n) for r in (1, 8, 9, 17) for k in (1, 31, 33, 1536) for n in (5, 13, 1027)]


def _linear_case(L, rows, K, N, silu, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(rows, K, device="cuda", generator=g)
    w = torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)
    b = torch.randn(N, device="cuda", generator=g) * 0.3
    buf = torch.full(((rows + 2) * N,), float("nan"), device="cuda")      # one sentinel row before and after
    out = buf[N:N + rows * N].view(rows, N)
    _check(L, L.vdt_op_linear(_p(x), _p(w), _p(b), out.data_ptr(), rows, K, N, int(silu), None))
    torch.cuda.synchronize()
    assert torch.isnan(buf[:N]).all() and torch.isnan(buf[N + rows * N:]).all(), "linear wrote outside [rows, N]"
    pre = x.double() @ w.double().t() + b.double()
    ref = F.silu(pre) if silu else pre
    scale = x.double().abs() @ w.double().abs().t() + b.double().abs() + ref.abs()
    assert torch.isfinite(out).all(), "linear left part of [rows, N] unwritten"
    return ((out.double() - ref).abs() / (U * scale)).max().item()


@pytest.mark.parametrize("silu", [0, 1])
@pytest.mark.parametrize("shape", LIN_NET, ids=lambda s: "x".join(map(str, s)))
def test_linear_network_shapes(L, shape, silu):
    rows, K, N = shape
    m = _linear_case(L, rows, K, N, silu, seed=rows * 7 + K * 13 + N)
    _report(f"linear {rows}x{K}x{N} silu{silu}", m)
    assert m <= LIN_C, m


@pytest.mark.parametrize("silu", [0, 1])
@pytest.mark.parametrize("shape", LIN_EDGE, ids=lambda s: "x".join(map(str, s)))
def test_linear_edges(L, shape, silu):
    rows, K, N = shape
    m = _linear_case(L, rows, K, N, silu, seed=rows * 7 + K * 13 + N + 1)
    _report(f"linear edge {rows}x{K}x{N} silu{silu}", m)
    assert m <= LIN_C, m


# ----------------------------------------------------------------------------------------------------- timestep embedding
def _temb(L, t64, dim, fp32_t):
    out = torch.full((t64.numel(), dim), float("nan"), device="cuda")
    _check(L, L.vdt_op_timestep_embedding_ex(_p(t64), _p(out), t64.numel(), dim, fp32_t, None))
    torch.cuda.synchronize()
    return out


def _t_values(seed):
    g = torch.Generator().manual_seed(seed)
    grid = torch.cat([torch.arange(1, 101, dtype=torch.float64) / 100, torch.arange(1, 1001, 37, dtype=torch.float64) / 1000])
    return torch.cat([torch.tensor([0.0, 1e-3, 0.5, 1.0], dtype=torch.float64), grid,
                      torch.rand(64, generator=g, dtype=torch.float64)])


@pytest.mark.parametrize("dim", [64, 128, 192, 256, 65])
def test_timestep_embedding_fp64(L, dim):
    from oracle.diffusion_ref import timestep_embedding
    t = _t_values(dim)
    ref = timestep_embedding(t, dim)                       # fp64 on the CPU, rounded to fp32 once
    out = _temb(L, t.cuda(), dim, 0).cpu()
    plain = torch.full_like(out, float("nan")).cuda()
    _check(L, L.vdt_op_timestep_embedding(_p(t.cuda()), _p(plain), t.numel(), dim, None))
    torch.cuda.synchronize()
    assert torch.equal(plain.cpu(), out), "vdt_op_timestep_embedding and the _ex hook with fp32_t = 0 differ"
    if dim % 2:
        assert (out[:, -1] == 0).all()
    zero = ref == 0
    assert (out[zero] == 0).all(), "exact zeros (sin 0, the pad column) must stay exact"
    ulps = ((out.double() - ref.double()).abs()[~zero] / _ulp32(ref.double()[~zero])).max().item()
    _report(f"temb fp64 dim{dim} ulp", ulps)
    assert ulps <= TEMB_F64_ULP, ulps


@pytest.mark.parametrize("dim", [64, 128, 192, 256, 65])
def test_timestep_embedding_fp32_t(L, dim):
    """p_sample_progressive's fp32 step tensor: every op of functions.py:20-25 rounds to fp32.  The angle 1000 t f_k is
    itself an fp32 product, so two correct evaluations (the oracle's CPU exp and the kernel's expf may differ by an ulp
    of f_k) can hold angles an ulp apart: 2^-24 |angle| each, passed through sin / cos with slope <= 1.  The bar is
    therefore proportional to the angle, up to 1000 rad.  A second check pins the kernel to the fp32 rounding chain itself:
    with fr = expf(fl(-k c)) evaluated by torch on the same device, sin and cos of the identical fp32 angle must agree with
    fp64 sin / cos to TEMB_CHAIN_ULP ulps."""
    from oracle.diffusion_ref import timestep_embedding
    t32 = _t_values(dim + 1).float()
    out = _temb(L, t32.double().cuda(), dim, 1)
    ref = timestep_embedding(t32, dim)                     # the oracle evaluated in fp32 (CPU)
    half = dim // 2
    c32 = torch.tensor(math.log(10000.0) / (half - 1), dtype=torch.float32)
    ang_cpu = torch.outer(1000.0 * t32, torch.exp(-torch.arange(half, dtype=torch.float32) * c32)).double()
    err = (out.cpu().double() - ref.double()).abs()
    bound = U * (torch.cat([ang_cpu, ang_cpu], 1).abs() + 1)
    if dim % 2:
        assert (out[:, -1] == 0).all()
        err = err[:, :-1]
    m = (err / bound).max().item()
    _report(f"temb fp32-t dim{dim} vs oracle (U*(|ang|+1))", m)
    assert m <= TEMB_F32_C, m
    # the fp32 chain on the device: ts = fl(1000 t), fr = expf(fl(-k c)), ang = fl(ts fr)
    tc = t32.cuda()
    fr = torch.exp(-torch.arange(half, dtype=torch.float32, device="cuda") * c32.cuda())
    ang = (1000.0 * tc)[:, None] * fr[None, :]
    chain = torch.cat([torch.sin(ang.double()), torch.cos(ang.double())], 1)
    o = out[:, :2 * half].double()
    nz = chain.float().double() != 0
    ulps = ((o - chain).abs()[nz] / _ulp32(chain[nz])).max().item()
    _report(f"temb fp32-t dim{dim} vs fp64 sin/cos of the fp32 angle (ulp)", ulps)
    assert ulps <= TEMB_CHAIN_ULP, ulps


# ------------------------------------------------------------------------------------------------------ class embedding
def _class_embed(L, e, w, b, ncls, y=None, ym=None):
    rows, E = e.shape
    out = torch.full_like(e, float("nan"))
    _check(L, L.vdt_op_class_embed(_p(e), _p(y), _p(ym), _p(w), _p(b), ncls, _p(out), rows, E, None))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("ncls,E", [(10, 1024), (10, 256), (40, 768), (1, 64)])
def test_class_embed_ids(L, ncls, E):
    """OneHot(exclude_zero=True) + Linear (modules.py:190-199): id c in 1..ncls adds b + w[:, c-1], 0 adds b only.  The
    weight sits in front of NaN padding, so an id past ncls that read beyond w[:, ncls-1] would show."""
    g = torch.Generator(device="cuda").manual_seed(ncls + E)
    ids = [0, 1, ncls, 0, ncls // 2 + 1, ncls + 1, ncls + 1000, -1, -(1 << 40), 1 << 40]
    rows = len(ids) + 2
    e = torch.randn(rows, E, device="cuda", generator=g) * 2
    e[-2] = -torch.linspace(80, 1000, E, device="cuda")            # SiLU of large negative inputs: expf(-v) overflows
    e[-1] = torch.linspace(80, 1000, E, device="cuda")
    ids += [ncls, 0]
    e[ids.index(ncls + 1)] = e[ids.index(ncls)]                    # same e, so the clamped id must give the same row
    e[ids.index(-1)] = e[0]
    wbuf = torch.full((E * ncls + 4096,), float("nan"), device="cuda")
    w = wbuf[:E * ncls].view(E, ncls)
    w.copy_(torch.randn(E, ncls, device="cuda", generator=g))
    b = torch.randn(E, device="cuda", generator=g) * 0.5
    y = torch.tensor(ids, dtype=torch.int64, device="cuda")
    out = _class_embed(L, e, w, b, ncls, y=y)
    cls = y.clamp(max=ncls)
    onehot = torch.zeros(rows, ncls, dtype=torch.float64, device="cuda")
    sel = cls > 0
    onehot[sel, cls[sel] - 1] = 1
    add = onehot @ w.double().t()
    v = e.double() + b.double() + add
    ref = F.silu(v)
    assert torch.isfinite(out).all()
    m = ((out.double() - ref).abs() / (U * (e.double().abs() + b.double().abs() + add.abs() + ref.abs()))).max().item()
    _report(f"class_embed ids ncls{ncls} E{E}", m)
    assert m <= CLS_C, m
    assert torch.equal(out[ids.index(ncls + 1)], out[ids.index(ncls)]), "ids above num_classes clamp to num_classes"
    assert torch.equal(out[ids.index(-1)], out[0]), "negative ids add the bias only"


@pytest.mark.parametrize("ncls,E", [(40, 768), (40, 256), (7, 64)])
def test_class_embed_multitag(L, ncls, E):
    """unet.py:290-294: y / sqrt(count_nonzero(y).clamp(min=1)) through the Linear; nonzeros are counted, the sum is
    value-weighted."""
    g = torch.Generator(device="cuda").manual_seed(ncls * 3 + E)
    ym = torch.zeros(8, ncls, device="cuda")
    ym[1, ncls // 2] = 1                                           # one tag
    ym[2] = 1                                                      # every tag
    ym[3, :3] = torch.tensor([0.5, 2.0, -1.0], device="cuda")      # non-binary values
    ym[4] = (torch.rand(ncls, device="cuda", generator=g) < 0.12).float()
    ym[5] = torch.randn(ncls, device="cuda", generator=g)
    ym[6, -1] = 3.0
    # row 0 and row 7: all zero (the clamp(min=1) path)
    e = torch.randn(8, E, device="cuda", generator=g)
    e[7] = -torch.linspace(80, 1000, E, device="cuda")
    w = torch.randn(E, ncls, device="cuda", generator=g) / math.sqrt(ncls)
    b = torch.randn(E, device="cuda", generator=g) * 0.5
    out = _class_embed(L, e, w, b, ncls, ym=ym)
    yd = ym.double()
    nnz = (yd != 0).sum(1, keepdim=True).clamp(min=1)
    add = (yd / nnz.sqrt()) @ w.double().t()
    ref = F.silu(e.double() + b.double() + add)
    sc = e.double().abs() + b.double().abs() + (yd.abs() / nnz.sqrt()) @ w.double().abs().t() + ref.abs()
    assert torch.isfinite(out).all()
    m = ((out.double() - ref).abs() / (U * sc)).max().item()
    _report(f"class_embed multitag ncls{ncls} E{E}", m)
    assert m <= CLS_C, m


# -------------------------------------------------------------------------------------------------------------- FiLM rows
@pytest.mark.parametrize("rep", [1, 2])
def test_film_rows(L, rep):
    ncls = 10
    labels = [0, 1, 5, ncls, ncls + 1, -1, 1 << 40, -(1 << 40), 3]
    lab = torch.tensor(labels, dtype=torch.int64, device="cuda")
    rows = len(labels) * rep
    buf = torch.full((rows + 8,), -7, dtype=torch.int32, device="cuda")
    _check(L, L.vdt_op_film_rows(_p(lab), rows, rep, ncls, _p(buf), None))
    torch.cuda.synchronize()
    want = []
    for i in range(rows):
        v = 0 if (rep == 2 and i % 2) else labels[i // rep]
        want.append(min(max(v, 0), ncls))
    assert buf[:rows].tolist() == want
    assert (buf[rows:] == -7).all(), "film_rows wrote past rows"
    _check(L, L.vdt_op_film_rows(None, rows, rep, ncls, _p(buf), None))      # no labels: every row reads table row 0
    torch.cuda.synchronize()
    assert (buf[:rows] == 0).all() and (buf[rows:] == -7).all()


@pytest.mark.parametrize("rep", [1, 2])
def test_multitag_rows(L, rep):
    ncls, imgs = 40, 5
    g = torch.Generator(device="cuda").manual_seed(rep)
    lab = torch.randn(imgs, ncls, device="cuda", generator=g)
    rows = imgs * rep
    buf = torch.full((rows + 2, ncls), float("nan"), device="cuda")
    _check(L, L.vdt_op_multitag_rows(_p(lab), rows, rep, ncls, _p(buf), None))
    torch.cuda.synchronize()
    want = lab.repeat_interleave(rep, 0)
    if rep == 2:
        want[1::2] = 0
    assert torch.equal(buf[:rows], want)
    assert torch.isnan(buf[rows:]).all()


def test_film_table_matches_training_forward(L):
    """The sampler's conditioning, composed from the hooks as the plan runs it (plan.cu add_embedding_steps): a FiLM table
    over the class ids 0..ncls at one t, indexed per UNet row by film_rows with the CFG interleave -- against the per-row
    FiLM vectors training.py's forward builds for the same (t, y) at B = 128 UNet rows (64 images, odd rows y = 0)."""
    from tests.cases import _cfg
    from v_diffusion_b200 import UNet
    from v_diffusion_b200.training import UNetTrainGraph
    cfg = _cfg(num_classes=10)
    torch.manual_seed(5)
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
               cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"], num_heads=cfg["num_heads"],
               num_classes=cfg["num_classes"]).cuda()
    with torch.no_grad():                                   # non-trivial biases (the reference initialises some to zero)
        for n, p in net.named_parameters():
            if n.endswith(".bias"):
                p.normal_(0, 0.1)
    ncls, hid, E = cfg["num_classes"], cfg["hid_channels"], cfg["embedding_dim"]
    imgs, rep = 64, 2
    B = imgs * rep
    g = torch.Generator(device="cuda").manual_seed(9)
    labels = torch.randint(0, ncls + 1, (imgs,), device="cuda", generator=g)
    t = 0.37
    y_rows = labels.repeat_interleave(2)
    y_rows[1::2] = 0
    graph = UNetTrainGraph(net)
    with torch.no_grad():
        graph.forward(torch.randn(B, cfg["in_channels"], 16, 16, device="cuda"), torch.full((B,), t, dtype=torch.float64),
                      y_rows, drop_rate=0.0)
    P = {k: v.detach() for k, v in net.named_parameters()}
    fc = sorted(k[:-len(".fc.weight")] for k in P if k.endswith(".fc.weight"))
    emb_act = graph._emb["emb_act"]
    film_train = torch.cat([graph.ops.linear(emb_act, P[n + ".fc.weight"], P[n + ".fc.bias"]) for n in fc], 1)

    def lin(x, w, b, silu):
        out = torch.empty(x.shape[0], w.shape[0], device="cuda")
        _check(L, L.vdt_op_linear(_p(x), _p(w.contiguous()), _p(b), _p(out), x.shape[0], x.shape[1], w.shape[0], silu, None))
        return out

    er = ncls + 1
    temb = _temb(L, torch.full((er,), t, dtype=torch.float64, device="cuda"), hid, 0)
    e1 = lin(temb, P["time_embed.0.weight"], P["time_embed.0.bias"], 1)
    e2 = lin(e1, P["time_embed.2.weight"], P["time_embed.2.bias"], 0)
    act = _class_embed(L, e2, P["class_embed.1.weight"], P["class_embed.1.bias"], ncls,
                       y=torch.arange(er, dtype=torch.int64, device="cuda"))
    w_all = torch.cat([P[n + ".fc.weight"] for n in fc], 0).contiguous()
    b_all = torch.cat([P[n + ".fc.bias"] for n in fc], 0).contiguous()
    table = lin(act, w_all, b_all, 0)
    film_row = torch.empty(B, dtype=torch.int32, device="cuda")
    _check(L, L.vdt_op_film_rows(_p(labels), B, rep, ncls, _p(film_row), None))
    torch.cuda.synchronize()
    assert torch.equal(film_row.long(), y_rows)
    film_hook = table[film_row.long()]
    scale = emb_act.double().abs() @ w_all.double().abs().t() + b_all.double().abs()
    m = ((film_hook.double() - film_train.double()).abs() / (U * scale)).max().item()
    same = torch.equal(film_hook, film_train)
    _report(f"film table vs training forward (bit-identical: {same})", m)
    assert m <= FILM_C, m


# --------------------------------------------------------------------------------------------------------- fp32 attention
ATT_CASES = [(d, heads, n) for d in (64, 128, 192, 256) for heads in (1, 2, 3) for n in (16, 49, 196, 1024)]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("case", ATT_CASES, ids=lambda c: "d{}_h{}_n{}".format(*c))
def test_attention_f32(L, case, f16):
    d, heads, n = case
    B = 2
    hid = heads * d
    g = torch.Generator(device="cuda").manual_seed(d + 7 * heads + n)
    qkv = torch.randn(B * n, 3 * hid, device="cuda", generator=g)
    qkv[:3, :hid] *= 25.0                                   # peaky rows: softmax close to one-hot
    qkv[n:n + 2, :hid] = 0.0                                # flat rows: uniform softmax
    hi = torch.empty(B * n, hid, dtype=DT[f16], device="cuda")
    lo = torch.empty_like(hi)
    _check(L, L.vdt_op_attention_f32(_p(qkv), _p(hi), _p(lo), B, n, heads, d, f16, None))
    torch.cuda.synchronize()
    q, k, v = qkv.double().view(B, n, 3, heads, d).unbind(2)           # [B, n, heads, d]
    s = torch.einsum("bihd,bjhd->bhij", q, k) / math.sqrt(d)
    p = torch.softmax(s, dim=-1)
    ref = torch.einsum("bhij,bjhd->bihd", p, v).reshape(B * n, hid)
    pv = torch.einsum("bhij,bjhd->bihd", p, v.abs()).reshape(B * n, hid)
    S = (torch.einsum("bihd,bjhd->bhij", q.abs(), k.abs()) / math.sqrt(d)).amax(-1)      # [B, heads, n]
    S = S.permute(0, 2, 1).reshape(B * n, heads, 1).expand(B * n, heads, d).reshape(B * n, hid)
    o = hi.double() + lo.double()
    # below fp16's normal range (2^-14) hi is subnormal and lo = round16(o - hi) underflows, so an fp16 pair holds o only to
    # half the subnormal spacing: 2^-25 absolute (peaky rows whose winning value is ~1e-5 reach it); bf16 has fp32's range
    floor = 2.0 ** -25 if f16 else 0.0
    m = (((o - ref).abs() - floor).clamp_min(0) / (U * pv * (1 + S))).max().item()
    # hi is a nearest 16-bit value of hi + lo (a tie may round either way)
    r = o.float().to(DT[f16])
    off = (r != hi) & ((o - hi.double()).abs() != (o - r.double()).abs())
    _report(f"attention_f32 {FMT[f16]} d{d} h{heads} n{n}", m)
    assert int(off.sum()) == 0, f"{int(off.sum())} hi values are not a 16-bit rounding of hi + lo"
    assert m <= ATT_C[f16], m


# ------------------------------------------------------------------------------------------------------ groupnorm_train
# (B, H, C): norm2 of the ResidualBlocks training.py runs -- CIFAR 256 at 32 / 16 / 8, CelebA 192 / 384 / 576 / 768 at
# 64 / 32 / 16 / 8, MNIST 64 / 128 at 28 / 14 / 7
GN_CASES = [(2, 32, 256), (2, 16, 256), (3, 8, 256), (2, 64, 192), (2, 32, 384), (2, 16, 576), (2, 8, 768),
            (2, 28, 64), (3, 14, 128), (2, 7, 128)]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("case", GN_CASES, ids=lambda c: "B{}_{}x{}_c{}".format(c[0], c[1], c[1], c[2]))
def test_groupnorm_train(L, case, p, f16):
    B, H, Cc = case
    g = torch.Generator(device="cuda").manual_seed(B + H + Cc)
    x = torch.randn(B, H, H, Cc, device="cuda", generator=g) * 1.3 + 0.4
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.2
    film = torch.randn(B, 2 * Cc, device="cuda", generator=g) * 0.3
    seed, layer = 987654321, 5
    out = torch.empty(B, H, H, Cc, dtype=DT[f16], device="cuda")
    _check(L, L.vdt_op_groupnorm_train(_p(x), Cc, B, H, H, _p(gamma), _p(beta), _p(film), 2 * Cc, 0, 1, _p(out), f16,
                                       C.c_float(p), seed, layer, None))
    torch.cuda.synchronize()
    y = F.group_norm(x.double().permute(0, 3, 1, 2), 32, gamma.double(), beta.double(), 1e-6).permute(0, 2, 3, 1)
    fd = film.double()
    y = F.silu(y * (1 + fd[:, Cc:].view(B, 1, 1, Cc)) + fd[:, :Cc].view(B, 1, 1, Cc))   # unet.py:145: shift | scale
    if p > 0:
        keep = out != 0                                     # the kernel's own mask
        frac = keep.double().mean().item()
        n = keep.numel()
        assert abs(frac - (1 - p)) < 6 * math.sqrt(p * (1 - p) / n), frac
        y = y * keep.double() / (1 - p)
    err = (out.double() - y).abs() - U16[f16] * y.abs()
    m = err.max().item()
    _report(f"groupnorm_train {FMT[f16]} p{p} B{B} {H}x{H} c{Cc} (excess over u16|ref|)", m)
    assert m <= GN_ABS, m
    if p == 0:
        plain = torch.empty_like(out)
        _check(L, L.vdt_op_groupnorm(_p(x), Cc, None, 0, B, H, H, _p(gamma), _p(beta), _p(film), 2 * Cc, 0, 1, 0, _p(plain),
                                     None, None, f16, None, None, 4, 0, None))
        torch.cuda.synchronize()
        assert torch.equal(plain, out), "drop_p = 0 must be bit-identical to vdt_op_groupnorm with the same FiLM"
