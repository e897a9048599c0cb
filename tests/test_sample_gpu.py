"""Op-level parity of the decode frame's sampler and bookkeeping, each driven alone through its production launcher
(fsb_op_sample / fsb_op_frame_end, include/fishb200.h):

  sample_kernel     (csrc/lm_kernels.cu) head logits from the partials, top-k / top-p / temperature, the RAS re-draw,
                    the token mapping, <|im_end|> flags, per-slot control and the Philox stream
  frame_end_kernel  (csrc/lm_kernels.cu) records the frame, advances n_out / positions / slot states and the step counter

The end-to-end tests reach the sampler with the tiny model (97 slow candidates, 96 codes) or greedily at S2-Pro size.
Here it runs at S2-Pro's head sizes (4097 slow candidates = 4096 semantic tokens + <|im_end|>, 4096 codes) and up to
kSampleMaxN = 8192, where it loops over several 1024-thread strides and the 4096-wide partial-sum pass.

Logits are compared bit for bit (rbf of the slot-ordered fp32 sum). Stochastic decisions are compared with the
reference algorithm itself: the kernel's logits, in token-id order, go through oracle.lm_oracle.logits_to_probs
verbatim and then argmax(probs / -log(U)) in bf16 (inference.py:43-93), with the uniforms U the kernel is fed through
its noise hook. Slot 0 alone takes those uniforms, so each decision is one launch; a row of a 32-row partial set is
chosen by offsetting the workspace pointer, and each launch writes its own token through its own output pointer.

Two rules decide where kernel and reference may part:
  * the reference's torch.sort orders equal logits arbitrarily (CPU sort put two tied values in opposite orders at two
    vector lengths), so where equal logits straddle the top-k / top-p cut, the survivors are those of the kernel's
    stated order (larger logit first, ties by candidate row) or the reference's;
  * a decision may differ where the reference's own decision is a near-tie (top-2 scores within 2 bf16 ulps, or a
    cumulative probability within 2 ulps of top_p): the kernel sums its softmax in another order. Such decisions are
    counted and bounded per configuration; every other decision is identical.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import lm_oracle as O

pytestmark = pytest.mark.gpu

ROWS = 32      # batch rows of a partial set (kStepRows)
SEL_CAP = 256  # ranks the sampler materialises (kSelCap); a larger top_k behaves like 256 (scheduler.py:100)
MAX_N = 8192   # kSampleMaxN
BF = torch.bfloat16
S2 = dict(sem_begin=151678, im_end=151645, cb=4096)   # S2-Pro token ids (configs.py)
TINY = dict(sem_begin=1000, im_end=999, cb=96)        # the tiny test model (oracle.lm_oracle.tiny_config)
NEAR_TIE_SHARE = 0.02


def _st():
    return torch.cuda.current_stream().cuda_stream


def _lib():
    from fish_speech_b200 import _lib

    return _lib, _lib.lib()


def cdiv(a, b):
    return (a + b - 1) // b


def rbf(x):
    """fp32 -> nearest bf16 (ties to even) -> fp32."""
    return x.float().to(BF).float()


def bf(x):
    return float(torch.tensor(x).to(BF).float())


def bits(t):
    return t.view(torch.int32)


def slot_sums(ws, nparts, n_out):
    """[32, n_out] fp32 value of a partial set: slots q < nparts[tile] added in slot order, as the kernels do."""
    tiles = ws.shape[1]
    acc = torch.zeros(tiles, ROWS, 128)
    npt = torch.as_tensor(np.asarray(nparts)).view(tiles, 1, 1)
    for q in range(int(npt.max())):
        acc = torch.where(npt > q, acc + ws[q], acc)
    return acc.permute(1, 0, 2).reshape(ROWS, tiles * 128)[:, :n_out]


class Parts:
    """A partial set on the device: ws [max_parts, tiles, 32, 128] fp32, nparts [tiles]."""

    def __init__(self, ws, nparts, n):
        self.n, self.tiles, self.max_parts = n, ws.shape[1], int(nparts.max())
        self.ws_host = ws
        self.ws = ws.cuda()
        self.nparts = torch.as_tensor(nparts, dtype=torch.int32).cuda()

    def row_ptr(self, r):
        """Workspace pointer under which row r of the set is row 0 (one-row launches)."""
        return self.ws.data_ptr() + 4 * 128 * r


def random_parts(n, rows, max_parts, seed):
    """Random partials, a different count per tile (one tile at max_parts); dead slots and rows past `rows` are NaN.
    Returns (Parts, expected logits [rows, n])."""
    g = torch.Generator().manual_seed(seed)
    tiles = cdiv(n, 128)
    nparts = torch.randint(1, max_parts + 1, (tiles,), generator=g).to(torch.int32)
    nparts[torch.randint(0, tiles, (1,), generator=g)] = max_parts
    ws = torch.randn(max_parts, tiles, ROWS, 128, generator=g) * 1.5
    q = torch.arange(max_parts).view(-1, 1, 1, 1)
    ws = torch.where(q >= nparts.view(1, -1, 1, 1), float("nan"), ws)
    ws[:, :, rows:] = float("nan")
    want = rbf(slot_sums(ws, nparts.numpy(), n))[:rows]
    return Parts(ws, nparts.numpy(), n), want


def exact_parts(logits):
    """One-slot partial set holding bf16 logits [rows <= 32, n] exactly; everything else NaN."""
    rows, n = logits.shape
    tiles = cdiv(n, 128)
    flat = torch.full((ROWS, tiles * 128), float("nan"))
    flat[:rows, :n] = logits
    ws = flat.view(ROWS, tiles, 128).permute(1, 0, 2).contiguous().unsqueeze(0)
    return Parts(ws, np.ones(tiles, dtype=np.int32), n)


def head(n, slow):
    ids = TINY if n == 97 else S2
    return dict(slow=int(slow), n_sem=n - 1 if slow else 0, sem_begin=ids["sem_begin"], im_end_id=ids["im_end"],
                codebook_size=ids["cb"] if slow else n)


def token_of(e, h):
    """Token id of candidate row e (slow head) or the code (fast head)."""
    if not h["slow"]:
        return e
    return h["sem_begin"] + e if e < h["n_sem"] else h["im_end_id"]


def token_order(n, h):
    """Candidate rows in token-id order (<|im_end|> precedes the semantic tokens in both vocabularies)."""
    if not h["slow"]:
        return np.arange(n)
    assert h["im_end_id"] < h["sem_begin"]
    return np.concatenate([[n - 1], np.arange(n - 1)])


def ptr(t):
    return t.data_ptr() if t is not None else None


def sample_args(parts, rows, h, *, temperature=1.0, top_p=1.0, top_k=1, num_cb=10, cb_index=0, cur_tok=None,
                logits_out=None, finished=None, row_slot=None, use_ras=0, ras_window=None, ras_update=0, seed=0,
                rng_offset=None, draw_id=0, noise=None, noise_draws=0, noise_ld=0, ctl=None):
    _l, _ = _lib()
    a = _l.SampleArgs()
    a.ws, a.nparts, a.tiles, a.max_parts = parts.ws.data_ptr(), parts.nparts.data_ptr(), parts.tiles, parts.max_parts
    a.n, a.rows = parts.n, rows
    a.temperature, a.top_p, a.top_k = temperature, top_p, top_k
    a.slow, a.n_sem, a.sem_begin, a.im_end_id, a.codebook_size = (h["slow"], h["n_sem"], h["sem_begin"], h["im_end_id"],
                                                                  h["codebook_size"])
    a.use_ras, a.ras_window, a.ras_update = use_ras, ptr(ras_window), ras_update
    a.seed, a.rng_offset, a.draw_id = seed, ptr(rng_offset), draw_id
    a.cur_tok, a.cb_index, a.num_cb = ptr(cur_tok), cb_index, num_cb
    a.logits_out, a.finished, a.row_slot = ptr(logits_out), ptr(finished), ptr(row_slot)
    a.noise_u, a.noise_draws, a.noise_ld = ptr(noise), noise_draws, noise_ld
    if ctl is not None:
        for k in ("state", "limit", "temperature", "top_p", "top_k", "seed", "n_out"):
            setattr(a.ctl, k, ctl[k].data_ptr())
    return a


def run(a):
    _l, L = _lib()
    _l.check(L.fsb_op_sample(C.byref(a), _st()))


def slot_ctl(slots, *, state=1, limit=1000, temperature=1.0, top_p=1.0, top_k=1, seed=0, n_out=0):
    def col(v, dt):
        return torch.as_tensor(np.broadcast_to(np.asarray(v), (slots,)).copy()).to(dt).cuda()

    return dict(state=col(state, torch.int32), limit=col(limit, torch.int32),
                temperature=col(temperature, torch.float32), top_p=col(top_p, torch.float32),
                top_k=col(top_k, torch.int32), seed=col(np.asarray(seed, dtype=np.uint64).view(np.int64), torch.int64),
                n_out=col(n_out, torch.int32))


# ------------------------------------------------------------------------------------------------
# the reference decision
# ------------------------------------------------------------------------------------------------
def _cut(sorted_logits, top_p, top_k):
    """Survivor count of logits_to_probs' mask on a sorted vector (its remove mask is monotone)."""
    cum = torch.cumsum(F.softmax(sorted_logits, dim=-1), dim=-1)
    ranks = torch.arange(sorted_logits.shape[-1])
    remove = (cum > top_p) | (ranks >= top_k)
    remove[0] = False
    return int(remove.float().argmax()) if bool(remove.any()) else sorted_logits.numel(), cum


def _probs_in_order(logits, temperature, top_p, top_k, order):
    """logits_to_probs with the sort's order of equal logits fixed to `order`."""
    idx = torch.as_tensor(order)
    sorted_logits = logits[idx]
    cum = torch.cumsum(F.softmax(sorted_logits, dim=-1), dim=-1)
    ranks = torch.arange(sorted_logits.shape[-1])
    remove = (cum > top_p) | (ranks >= top_k)
    remove[0] = False
    remove = remove.scatter(dim=-1, index=idx, src=remove)
    logits = torch.where(remove, float("-Inf"), logits)
    logits = logits / torch.clip(temperature, min=1e-5)
    return F.softmax(logits, dim=-1)


def reference_decision(lt, rows_of_tok, temperature, top_p, top_k, u):
    """lt: bf16 logits in token-id order; rows_of_tok: the kernel's candidate row of each; u: bf16 uniforms.
    Returns (choices, near): the reference's decision, plus the one with the kernel's tie order at the cut when equal
    logits straddle it; near = the reference's decision is a near-tie."""
    T, P = torch.tensor(temperature, dtype=BF), torch.tensor(top_p, dtype=BF)
    k = min(top_k, SEL_CAP)  # the documented divergence for top_k > 256 (scheduler.py:100)
    q = -torch.log(u)
    probs = O.logits_to_probs(lt, T, P, k)
    score = probs / q
    choices = {int(torch.argmax(score))}
    sorted_logits = torch.sort(lt, descending=True).values
    m, cum = _cut(sorted_logits, P, k)
    if m < lt.numel() and sorted_logits[m - 1] == sorted_logits[m]:
        order = np.lexsort((rows_of_tok, -lt.float().numpy()))
        choices.add(int(torch.argmax(_probs_in_order(lt, T, P, k, order) / q)))
    fin = score[torch.isfinite(score)].float()
    top2 = torch.topk(fin, 2).values if fin.numel() >= 2 else torch.tensor([1.0, 0.0])
    near = float(top2[0] - top2[1]) <= 2 * 2 ** -7 * float(top2[0].abs())
    near |= float((cum[: k + 1].float() - float(P)).abs().min()) <= 2 * 2 ** -7 * float(P)
    return choices, near


# ------------------------------------------------------------------------------------------------
# logits
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_parts", [1, 20])
@pytest.mark.parametrize("n", [1, 96, 97, 4096, 4097, 8192])
def test_logits_and_greedy_choice(n, max_parts):
    """logits_out == rbf(slot-ordered sum) bit for bit, NaN of dead slots / rows never read, rows past the batch never
    written; top_k = 1 picks the largest logit, the smallest candidate row on a tie."""
    rows = 29
    parts, want = random_parts(n, rows, max_parts, seed=n * 31 + max_parts)
    h = head(n, n % 2 == 1)
    lo = torch.full((ROWS, n), -7.0, device="cuda")
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    run(sample_args(parts, rows, h, top_k=1, cur_tok=ct, logits_out=lo, cb_index=2))
    lo, ct = lo.cpu(), ct.cpu()
    assert torch.equal(bits(lo[:rows]), bits(want)), f"logits differ at {(bits(lo[:rows]) != bits(want)).nonzero()[:4]}"
    assert (lo[rows:] == -7.0).all()
    best = want.max(dim=1, keepdim=True).values
    first = torch.where(want == best, torch.arange(n), n).min(dim=1).values
    if h["slow"]:
        assert ct[:rows, 0].tolist() == [token_of(int(e), h) for e in first]
    else:
        assert ct[:rows, 3].tolist() == first.tolist()
    assert (ct[rows:] == -5).all()


def test_launcher_rejects_bad_n_and_top_k():
    """n > kSampleMaxN and top_k < 1 without slot control are refused before anything is launched."""
    _l, L = _lib()
    ct = torch.zeros(ROWS, 11, dtype=torch.int32, device="cuda")
    for n, k in ((MAX_N + 1, 5), (4096, 0)):
        parts = exact_parts(torch.zeros(1, n))
        a = sample_args(parts, 1, head(n, False), top_k=k, cur_tok=ct)
        before = _l.launch_count()
        assert L.fsb_op_sample(C.byref(a), _st()) != 0
        assert _l.launch_count() == before, (n, k)


# ------------------------------------------------------------------------------------------------
# greedy
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4097, 8192])
def test_greedy_argmax_and_tie_rule(n):
    """top_k = 1: the largest logit at every thread-stride and 4096-pass edge; on an exact tie the smallest candidate
    row wins, across thread strides and across the 4096 boundary. Greedy breaks ties by ROW; the stochastic path
    breaks them by token id (the argmax `key`, where <|im_end|> -- the last row -- has the smallest id). The reference
    orders ties arbitrarily (torch.sort), so it must pick one of the tied candidates; the kernel must pick the first."""
    plants = [[0], [1023], [1024], [4095], [4096], [n - 1], [5, 1029], [1023, 1024], [4095, 4096], [100, n - 1],
              [4096, n - 1], [2047, 3071, 4096], [0, n - 1]]
    g = torch.Generator().manual_seed(n)
    lg = rbf(torch.randn(len(plants), n, generator=g))
    for r, p in enumerate(plants):
        lg[r, p] = 9.0
    h = head(n, n == 4097)
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    run(sample_args(exact_parts(lg), len(plants), h, top_k=1, cur_tok=ct))
    got = ct.cpu()[:, 0 if h["slow"] else 1]
    order = token_order(n, h)
    for r, p in enumerate(plants):
        assert int(got[r]) == token_of(min(p), h), (r, p, int(got[r]))
        if h["slow"]:
            probs = O.logits_to_probs(lg[r, order].to(BF), torch.tensor(1.0, dtype=BF), torch.tensor(1.0, dtype=BF), 1)
            ref_row = int(order[int(torch.argmax(probs))])
            assert ref_row in p, (r, p, ref_row)


# ------------------------------------------------------------------------------------------------
# stochastic decisions against the reference
# ------------------------------------------------------------------------------------------------
TEMPS = [bf(t) for t in (1e-6, 0.1, 0.7, 1.0, 1.9)]  # the host passes bf16-rounded values (scheduler.py)
TOP_PS = [bf(0.05), 0.5, 0.8984375, 0.90234375, 1.0]
TOP_KS = [2, 30, 256, 257, 4097]
SHAPES = ["gauss", "flat", "few", "dominant", "im_end_max", "offset"]


def shaped_logits(shape, rows, n, g):
    if shape == "gauss":
        x = torch.randn(rows, n, generator=g) * 2
    elif shape == "flat":  # top-p needs more than 256 ranks
        x = torch.randn(rows, n, generator=g) * 0.05
    elif shape == "few":  # heavy bf16 ties
        x = torch.tensor([-1.0, 0.0, 0.5, 1.25])[torch.randint(0, 4, (rows, n), generator=g)]
    elif shape == "dominant":  # one survivor
        x = torch.randn(rows, n, generator=g)
        x[torch.arange(rows), torch.randint(0, n, (rows,), generator=g)] = 20.0
    elif shape == "im_end_max":  # the last row (<|im_end|> of the slow head) is the maximum
        x = torch.randn(rows, n, generator=g) * 2
        x[:, -1] = x.max(dim=1).values + torch.rand(rows, generator=g) * 2
    else:  # offsets around -30 and +80
        x = torch.randn(rows, n, generator=g) * 2 + torch.where(torch.arange(rows) % 2 == 0, -30.0, 80.0).view(-1, 1)
    return rbf(x)


def uniforms(shape, g):
    """bf16 uniforms in (0, 1) as torch.rand draws them (multiples of 2^-8), U = 0 excluded (the documented quirk)."""
    return torch.randint(1, 256, shape, generator=g).float() / 256


class OneRowLauncher:
    """Launches of one partial-set row each, as slot 0, with uniforms noise[f] (f = the launch's frame counter) and
    outputs written through per-launch pointers."""

    def __init__(self, parts, h, launches, noise_draws, num_cb=10):
        self.parts, self.h = parts, h
        self.stride = num_cb + 1
        self.ct = torch.full((launches, self.stride), -5, dtype=torch.int32, device="cuda")
        self.offs = torch.arange(launches, dtype=torch.int64, device="cuda")
        self.noise = torch.full((launches, noise_draws, parts.n), 0.5, device="cuda")
        self.noise_draws = noise_draws
        self.a = sample_args(parts, 1, h, num_cb=num_cb, noise=self.noise, noise_draws=noise_draws,
                             noise_ld=parts.n)

    def launch(self, i, row, **kw):
        a = self.a
        a.ws = self.parts.row_ptr(row)
        a.rng_offset = self.offs.data_ptr() + 8 * i
        a.cur_tok = self.ct.data_ptr() + 4 * self.stride * i
        for k, v in kw.items():
            setattr(a, k, v)
        run(a)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("n", [97, 4096, 4097])
def test_stochastic_matches_reference(n, shape):
    """Every (temperature, top_p) pair with each top_k once per temperature and once per top_p (a Latin square over
    the five values of each), 32 rows per setting: 800 decisions, the reference's near-ties bounded at 2 %.
    n = 4096 is the fast head (slow = 0, codes), 97 and 4097 the slow head. top_k 257 and 4097 are compared with the
    reference at 256: the sampler materialises at most 256 ranks (the documented divergence, scheduler.py:100)."""
    slow = n != 4096
    h = head(n, slow)
    g = torch.Generator().manual_seed(1000 * n + SHAPES.index(shape))
    lg = shaped_logits(shape, ROWS, n, g)
    parts = exact_parts(lg)
    settings = [(T, p, TOP_KS[(i + j) % 5]) for i, T in enumerate(TEMPS) for j, p in enumerate(TOP_PS)]
    L1 = OneRowLauncher(parts, h, len(settings) * ROWS, 1)
    u_rows = uniforms((len(settings) * ROWS, n), g)
    L1.noise.copy_(u_rows.view(-1, 1, n))
    lo = torch.full((ROWS, n), -7.0, device="cuda")
    i = 0
    for T, p, k in settings:
        for r in range(ROWS):
            extra = dict(logits_out=lo.data_ptr() + 4 * n * r) if i < ROWS else dict(logits_out=None)
            L1.launch(i, r, temperature=T, top_p=p, top_k=k, **extra)
            i += 1
    assert torch.equal(bits(lo.cpu()), bits(lg)), "kernel logits differ from the planted values"
    col = 0 if slow else 1
    got = L1.ct.cpu()[:, col]
    order = token_order(n, h)
    rows_of_tok = order
    near, tied = 0, 0
    i = 0
    for T, p, k in settings:
        for r in range(ROWS):
            lt = lg[r, order].to(BF)
            ut = u_rows[i, order].to(BF)
            choices, is_near = reference_decision(lt, rows_of_tok, T, p, k, ut)
            want = {token_of(int(order[c]), h) for c in choices}
            if int(got[i]) not in want:
                assert is_near, (f"T={T} top_p={p} top_k={k} row {r}: kernel {int(got[i])}, reference {sorted(want)} "
                                 "and the reference's decision is not a near-tie")
                near += 1
            tied += len(want) > 1
            i += 1
    print(f"n={n} {shape}: {i} decisions, {near} near-tie differences, {tied} with a tie at the cut")
    assert near <= NEAR_TIE_SHARE * i, f"{near} of {i} decisions differ at near-ties"


def plateau_logits(n, rows, g):
    """Rows whose largest logit (8.0) holds a softmax probability of 0.5003 (bf16 0.5) over a flat bulk whose
    probabilities are each below half a bf16 ulp of 0.5: the sorted cumulative sum stays exactly 0.5 for 16 ranks."""
    out = []
    for _ in range(rows):
        z = torch.randn(n, generator=g) * 0.02
        top = int(torch.randint(0, n, (1,), generator=g))
        lo, hi = -3.0, 3.0
        for _ in range(40):  # bisect the bulk's level
            x = rbf(z + (lo + hi) / 2)
            x[top] = 8.0
            if float(torch.softmax(x.double(), 0)[top]) > 0.5003:
                lo = (lo + hi) / 2
            else:
                hi = (lo + hi) / 2
        out.append(x)
    return torch.stack(out)


@pytest.mark.parametrize("n", [4096, 4097])
def test_top_p_keeps_ranks_whose_cumulative_sum_equals_top_p(n):
    """top_p = 0.5 with a cumulative sum that sits exactly at 0.5 for 16 ranks: the reference removes a rank only when
    cum > top_p, so all 16 survive (and the rank walk must not stop at the first cum == top_p). At T = 1.9 the bulk
    ranks win about a sixth of the draws."""
    h = head(n, n == 4097)
    g = torch.Generator().manual_seed(n + 3)
    lg = plateau_logits(n, ROWS, g)
    order = token_order(n, h)
    for r in range(ROWS):
        m, cum = _cut(torch.sort(lg[r, order].to(BF), descending=True).values, torch.tensor(0.5, dtype=BF), SEL_CAP)
        assert m >= 12 and float(cum[0]) == 0.5, (r, m)
    settings = [(bf(1.9), k) for k in (30, 256, 30, 256)]
    L1 = OneRowLauncher(exact_parts(lg), h, len(settings) * ROWS, 1)
    u = uniforms((len(settings) * ROWS, n), g)
    L1.noise.copy_(u.view(-1, 1, n))
    i = 0
    for T, k in settings:
        for r in range(ROWS):
            L1.launch(i, r, temperature=T, top_p=0.5, top_k=k)
            i += 1
    got = L1.ct.cpu()[:, 0 if h["slow"] else 1]
    near, bulk, i = 0, 0, 0
    for T, k in settings:
        for r in range(ROWS):
            # every decision here sits on a top-p near-tie (cum == top_p): differences are only counted
            choices, _ = reference_decision(lg[r, order].to(BF), order, T, 0.5, k, u[i, order].to(BF))
            near += int(got[i]) not in {token_of(int(order[c]), h) for c in choices}
            bulk += int(got[i]) != token_of(int(lg[r].argmax()), h)
            i += 1
    print(f"n={n}: {i} decisions, {bulk} drawn from the plateau ranks, {near} differ from the reference")
    assert near <= NEAR_TIE_SHARE * i, f"{near} of {i} decisions differ from the reference"
    assert bulk >= 0.05 * i


def test_low_temperature_clamp_matches_reference():
    """Temperatures below 1e-5 are clamped as the reference clamps its bf16 temperature tensor: torch.clip(T, min=1e-5)
    yields bf16(1e-5) = 1.0013580322265625e-05. The scaled logits are ~3e5 and round to bf16 steps of 2048, so the
    divisor decides which of two adjacent logits collapse into a tie (and share the probability) and which do not.
    The rows hold such adjacent pairs on top of a low floor; every decision must be the reference's."""
    n = 4097
    h = head(n, True)
    d_ref = torch.tensor(1e-5, dtype=BF).float()
    v = torch.arange(0x4000, 0x4100, dtype=torch.int32).to(torch.int16).view(BF).float()  # [2, 8)
    tie = rbf(v / d_ref)
    tie = tie[1:] == tie[:-1]
    tie_k = rbf(v / torch.tensor(1e-5))
    tie_k = tie_k[1:] == tie_k[:-1]
    pairs = (tie != tie_k).nonzero().view(-1)[:ROWS]
    assert pairs.numel() == ROWS
    g = torch.Generator().manual_seed(5)
    lg = rbf(torch.randn(ROWS, n, generator=g) - 20)
    a_pos = torch.randint(0, n, (ROWS,), generator=g)
    b_pos = (a_pos + 1 + torch.randint(0, n - 1, (ROWS,), generator=g)) % n
    lg[torch.arange(ROWS), a_pos] = v[pairs + 1]
    lg[torch.arange(ROWS), b_pos] = v[pairs]
    frames = 8
    L1 = OneRowLauncher(exact_parts(lg), h, frames * ROWS, 1)
    u = uniforms((frames * ROWS, n), g)
    L1.noise.copy_(u.view(-1, 1, n))
    T = bf(1e-6)
    for i in range(frames * ROWS):
        L1.launch(i, i % ROWS, temperature=T, top_p=1.0, top_k=30)
    got = L1.ct.cpu()[:, 0]
    order = token_order(n, h)
    bad = []
    for i in range(frames * ROWS):
        r = i % ROWS
        choices, _ = reference_decision(lg[r, order].to(BF), order, T, 1.0, 30, u[i, order].to(BF))
        want = {token_of(int(order[c]), h) for c in choices}
        if int(got[i]) not in want:
            bad.append((r, int(got[i]), sorted(want)))
    assert not bad, f"{len(bad)} of {frames * ROWS} decisions differ from the reference, e.g. {bad[:4]}"


@pytest.mark.parametrize("slow", [1, 0])
def test_stochastic_tie_breaks_on_token_id(slow):
    """Equal scores (equal logits, equal uniforms): the reference's torch.argmax returns the smallest token id. For
    the slow head that is <|im_end|> (id 151645, below the semantic ids) although it is the LAST candidate row."""
    n = 4097 if slow else 4096
    h = head(n, slow)
    g = torch.Generator().manual_seed(9 + slow)
    lg = rbf(torch.randn(ROWS, n, generator=g) - 10)
    partner = torch.randint(0, n - 101, (ROWS,), generator=g)
    top = torch.full((ROWS,), n - 1) if slow else n - 1 - torch.randint(0, 100, (ROWS,), generator=g)
    lg[torch.arange(ROWS), top] = 4.0
    lg[torch.arange(ROWS), partner] = 4.0
    L1 = OneRowLauncher(exact_parts(lg), h, ROWS, 1)
    L1.noise.fill_(0.5)
    for r in range(ROWS):
        L1.launch(r, r, temperature=0.7, top_p=1.0, top_k=30)
    got = L1.ct.cpu()[:, 0 if slow else 1]
    order = token_order(n, h)
    u = torch.full((n,), 0.5, dtype=BF)
    for r in range(ROWS):
        choices, _ = reference_decision(lg[r, order].to(BF), order, 0.7, 1.0, 30, u)
        assert len(choices) == 1
        want = token_of(int(order[choices.pop()]), h)
        assert int(got[r]) == want == min(token_of(int(partner[r]), h), token_of(int(top[r]), h)), r


@pytest.mark.parametrize("shape", ["gauss", "im_end_max"])
@pytest.mark.parametrize("top_p", [0.5, 0.9609375])
def test_ras_matches_reference(top_p, shape):
    """Repetition-aware sampling (inference.py:114-144): the main token is replaced by the high-temperature draw (draw
    1: T = 1, top_p = 0.9, the same top_k) only when it is in the slot's 10-token window AND semantic; <|im_end|> in
    the window is never replaced. top_p below 0.9 makes the sampler rank up to p_lim = 0.9 for draw 1 while draw 0
    keeps fewer survivors; above 0.9 both cuts are top_p-bound. ras_update shifts the window by one."""
    n = 4097
    h = head(n, True)
    g = torch.Generator().manual_seed(77 + int(top_p * 100) + len(shape))
    lg = shaped_logits(shape, ROWS, n, g)
    settings = [(bf(T), k) for T in (0.3, 0.7) for k in (30, 256)]
    launches = len(settings) * ROWS * 2
    L1 = OneRowLauncher(exact_parts(lg), h, launches, 2)
    u = uniforms((launches, 2, n), g)
    L1.noise.copy_(u)
    order = token_order(n, h)
    sem = lambda t: h["sem_begin"] <= t < h["sem_begin"] + h["n_sem"]  # noqa: E731
    win = torch.zeros(launches, 10, dtype=torch.int32)
    plan = []
    i = 0
    for T, k in settings:
        for r in range(ROWS):
            for rep in range(2):
                lt = lg[r, order].to(BF)
                mc, mnear = reference_decision(lt, order, T, top_p, k, u[i, 0, order].to(BF))
                hc, hnear = reference_decision(lt, order, 1.0, 0.8984375, k, u[i, 1, order].to(BF))
                mains = {token_of(int(order[c]), h) for c in mc}
                highs = {token_of(int(order[c]), h) for c in hc}
                w = h["sem_begin"] + torch.randint(0, h["n_sem"], (10,), generator=g)
                if rep == 0:  # the main token in the window
                    w[int(torch.randint(0, 10, (1,), generator=g))] = min(mains)
                if r % 4 == 0:
                    w[int(torch.randint(0, 10, (1,), generator=g))] = h["im_end_id"]
                win[i] = w
                plan.append((T, k, r, mains, highs, mnear, hnear))
                i += 1
    wd = win.cuda()
    for i, (T, k, r, *_rest) in enumerate(plan):
        L1.launch(i, r, temperature=T, top_p=top_p, top_k=k, use_ras=1, ras_update=1,
                  ras_window=wd.data_ptr() + 40 * i)
    got, wd = L1.ct.cpu(), wd.cpu()
    near, substituted, kept_im_end = 0, 0, 0
    for i, (T, k, r, mains, highs, mnear, hnear) in enumerate(plan):
        want = set()
        for m in mains:
            hit = bool((win[i] == m).any()) and sem(m)
            want |= highs if hit else {m}
        tok = int(got[i, 0])
        if tok not in want:
            assert mnear or hnear, f"T={T} top_k={k} row {r}: kernel {tok}, reference {sorted(want)}"
            near += 1
        substituted += tok in highs and tok not in mains
        kept_im_end += tok == h["im_end_id"] and bool((win[i] == tok).any())
        assert int(got[i, 1]) == min(max(tok - h["sem_begin"], 0), h["codebook_size"] - 1)
        assert wd[i].tolist() == win[i, 1:].tolist() + [tok], "window not shifted by one"
    print(f"RAS top_p={top_p} {shape}: {len(plan)} decisions, {substituted} substituted, {kept_im_end} <|im_end|> "
          f"kept in the window, {near} near-tie differences")
    assert near <= NEAR_TIE_SHARE * len(plan)
    assert substituted >= 10
    if shape == "im_end_max":
        assert kept_im_end >= 5


# ------------------------------------------------------------------------------------------------
# token mapping, flags, slots
# ------------------------------------------------------------------------------------------------
def planted(n, maxima, seed=3):
    lg = rbf(torch.randn(len(maxima), n, generator=torch.Generator().manual_seed(seed)))
    for r, e in enumerate(maxima):
        lg[r, e] = 9.0
    return lg


def test_token_mapping_and_flags():
    """Slow head: cur_tok[slot][0..1] = (token, clamped code), <|im_end|> gives code 0 and sets `finished`; with slot
    control <|im_end|> moves the state to 3 only from the second frame on (n_out >= 1). Fast head: column cb_index + 1
    only."""
    n = 4097
    h = head(n, True)
    maxima = [0, 4095, 4096, 17, 4096, 4096, 2048, 4096]
    lg = planted(n, maxima)
    rows = len(maxima)
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    fin = torch.full((ROWS,), 7, dtype=torch.int32, device="cuda")
    n_out = [0, 0, 0, 0, 1, 5, 1, 0]
    ctl = slot_ctl(ROWS, top_k=1, n_out=n_out + [0] * (ROWS - rows))
    run(sample_args(exact_parts(lg), rows, h, cur_tok=ct, finished=fin, ctl=ctl))
    ct, fin, state = ct.cpu(), fin.cpu(), ctl["state"].cpu()
    for r, e in enumerate(maxima):
        tok = token_of(e, h)
        code = 0 if e == 4096 else e
        assert ct[r, :2].tolist() == [tok, code], r
        assert (ct[r, 2:] == -5).all()
        assert int(fin[r]) == (1 if e == 4096 else 7), r
        assert int(state[r]) == (3 if e == 4096 and n_out[r] >= 1 else 1), r
    assert (ct[rows:] == -5).all() and (fin[rows:] == 7).all() and (state[rows:] == 1).all()
    # fast head: one column
    hf = head(4096, False)
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    run(sample_args(exact_parts(planted(4096, [5, 4095, 1024])), 3, hf, top_k=1, cur_tok=ct, cb_index=6,
                    finished=fin))
    ct = ct.cpu()
    assert ct[:3, 7].tolist() == [5, 4095, 1024]
    ct[:3, 7] = -5
    assert (ct == -5).all()


def test_row_slot_mapping():
    """row_slot = a permutation into sparse slots: every output of row r lands in slot row_slot[r], nothing else is
    written."""
    n = 4097
    h = head(n, True)
    row_slot = [17, 3, 30, 0, 9, 22, 5, 12]
    maxima = [4096, 12, 4095, 700, 0, 3000, 4096, 1]
    rows = len(row_slot)
    lg = planted(n, maxima)
    rs = torch.tensor(row_slot, dtype=torch.int32, device="cuda")
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    fin = torch.full((ROWS,), 7, dtype=torch.int32, device="cuda")
    lo = torch.full((ROWS, n), -7.0, device="cuda")
    win0 = torch.arange(ROWS * 10, dtype=torch.int32).view(ROWS, 10) + 151678
    win = win0.cuda()
    run(sample_args(exact_parts(lg), rows, h, top_k=1, cur_tok=ct, finished=fin, logits_out=lo, row_slot=rs,
                    use_ras=1, ras_window=win, ras_update=1))
    ct, fin, lo, win = ct.cpu(), fin.cpu(), lo.cpu(), win.cpu()
    for s in range(ROWS):
        if s in row_slot:
            r = row_slot.index(s)
            tok = token_of(maxima[r], h)
            assert ct[s, :2].tolist() == [tok, 0 if maxima[r] == 4096 else maxima[r]]
            assert int(fin[s]) == (1 if maxima[r] == 4096 else 7)
            assert torch.equal(bits(lo[s]), bits(lg[r]))
            assert win[s].tolist() == win0[s, 1:].tolist() + [tok]
        else:
            assert (ct[s] == -5).all() and int(fin[s]) == 7 and (lo[s] == -7.0).all() and torch.equal(win[s], win0[s])


def test_idle_and_frozen_slots_untouched():
    """Slot control: state 0 (idle) and 2 (finished) slots keep cur_tok, ras_window, finished, logits_out and state;
    states 1 and 3 sample (and <|im_end|> takes 1 to 3)."""
    n = 4097
    h = head(n, True)
    states = [1, 0, 2, 3] * 8
    lg = planted(n, [4096] * ROWS)
    ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
    fin = torch.full((ROWS,), 7, dtype=torch.int32, device="cuda")
    lo = torch.full((ROWS, n), -7.0, device="cuda")
    win0 = torch.arange(ROWS * 10, dtype=torch.int32).view(ROWS, 10) + 151678
    win = win0.cuda()
    ctl = slot_ctl(ROWS, state=states, top_k=1, n_out=2)
    run(sample_args(exact_parts(lg), ROWS, h, cur_tok=ct, finished=fin, logits_out=lo, use_ras=1, ras_window=win,
                    ras_update=1, ctl=ctl))
    ct, fin, lo, win, state = ct.cpu(), fin.cpu(), lo.cpu(), win.cpu(), ctl["state"].cpu()
    for s, st in enumerate(states):
        if st in (0, 2):
            assert (ct[s] == -5).all() and int(fin[s]) == 7 and (lo[s] == -7.0).all(), s
            assert torch.equal(win[s], win0[s]) and int(state[s]) == st, s
        else:
            assert ct[s, :2].tolist() == [h["im_end_id"], 0] and int(fin[s]) == 1 and int(state[s]) == 3, s
            assert torch.equal(bits(lo[s]), bits(lg[s])) and win[s, 9] == h["im_end_id"], s


def test_mixed_batch_equals_each_slot_alone():
    """Per-slot temperature / top_p / top_k / seed / n_out: every slot of a full batch draws what it draws alone (the
    stream depends on the request's seed and frame index, not on the slot or its neighbours)."""
    n = 4097
    h = head(n, True)
    g = torch.Generator().manual_seed(11)
    lg = rbf(torch.randn(ROWS, n, generator=g))
    parts = exact_parts(lg)
    temps = [TEMPS[i % 5] for i in range(ROWS)]
    tps = [TOP_PS[(i // 5) % 5] for i in range(ROWS)]
    tks = [[1, 2, 30, 256, 4097][(i * 3) % 5] for i in range(ROWS)]
    seeds = [int(x) for x in torch.randint(0, 2 ** 62, (ROWS,), generator=g)]
    for frame in range(3):
        n_out = [frame * 7 + i % 3 for i in range(ROWS)]
        ctl = slot_ctl(ROWS, temperature=temps, top_p=tps, top_k=tks, seed=seeds, n_out=n_out)
        ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
        run(sample_args(parts, ROWS, h, cur_tok=ct, ctl=ctl))
        batch = ct.cpu()[:, 0]
        alone = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
        for s in range(ROWS):
            rs = torch.tensor([s], dtype=torch.int32, device="cuda")
            a = sample_args(parts, 1, h, cur_tok=alone, row_slot=rs, ctl=ctl)
            a.ws = parts.row_ptr(s)
            run(a)
        assert torch.equal(batch, alone.cpu()[:, 0]), frame


# ------------------------------------------------------------------------------------------------
# the Philox stream
# ------------------------------------------------------------------------------------------------
def draw_many(parts, h, frames, *, draw_id=0, **kw):
    """32 rows (slots 0..31, no slot control) at rng_offset 0..frames-1: tokens [frames, 32]."""
    stride = 11
    ct = torch.full((frames, ROWS, stride), -5, dtype=torch.int32, device="cuda")
    offs = torch.arange(frames, dtype=torch.int64, device="cuda")
    a = sample_args(parts, ROWS, h, draw_id=draw_id, **kw)
    for f in range(frames):
        a.rng_offset = offs.data_ptr() + 8 * f
        a.cur_tok = ct.data_ptr() + 4 * stride * ROWS * f
        run(a)
    return ct.cpu()[:, :, 0 if h["slow"] else 1]


@pytest.mark.parametrize("n,top_k,top_p", [(4097, 30, 0.80078125), (4096, 30, 0.80078125), (4097, 256, 1.0)])
def test_philox_frequencies(n, top_k, top_p):
    """>= 10 000 draws (32 slots x 313 frame counters) of one logit row against the float64 softmax(logits / T) over
    the reference's survivors: chi-square below its 99.9th percentile (bins with expected count < 5 merged), and no
    draw ever outside the survivors."""
    from scipy.stats import chi2

    T = 0.8984375
    h = head(n, n == 4097)
    g = torch.Generator().manual_seed(n + top_k)
    row = rbf(torch.randn(n, generator=g) * 2)
    parts = exact_parts(row.expand(ROWS, n))
    frames = 313
    toks = draw_many(parts, h, frames, temperature=T, top_p=top_p, top_k=top_k).view(-1)
    order = token_order(n, h)
    lt = row[order].to(BF)
    # survivors in the kernel's order of equal logits (the cut falls inside a run of equal bf16 logits here)
    probs = _probs_in_order(lt, torch.tensor(T, dtype=BF), torch.tensor(top_p, dtype=BF), min(top_k, SEL_CAP),
                            np.lexsort((order, -lt.float().numpy())))
    sorted_logits = torch.sort(lt, descending=True).values
    m, cum = _cut(sorted_logits, torch.tensor(top_p, dtype=BF), min(top_k, SEL_CAP))
    assert float((cum[: m + 1].float() - top_p).abs().min()) > 2 * 2 ** -7 * top_p, "top-p cut is a near-tie"
    support = (probs > 0).nonzero().view(-1)
    assert support.numel() == m
    cand = torch.as_tensor(order)[support]
    # target: float64 softmax of the scaled logits as the reference forms them (bf16 logit / bf16 temperature)
    p64 = torch.softmax((lt[support] / torch.tensor(T, dtype=BF)).double(), 0)
    tok_ids = torch.tensor([token_of(int(e), h) for e in cand])
    counts = torch.tensor([(toks == t).sum() for t in tok_ids]).double()
    assert int(counts.sum()) == toks.numel(), "draws outside the support"
    exp = p64 * toks.numel()
    o = torch.argsort(exp)
    bins_e, bins_o, ae, ao = [], [], 0.0, 0.0
    for j in o.tolist():
        ae += float(exp[j]); ao += float(counts[j])
        if ae >= 5:
            bins_e.append(ae); bins_o.append(ao); ae, ao = 0.0, 0.0
    if ae > 0:
        bins_e[-1] += ae; bins_o[-1] += ao
    e_, o_ = np.array(bins_e), np.array(bins_o)
    stat = float(((o_ - e_) ** 2 / e_).sum())
    df = len(e_) - 1
    assert df >= 5
    assert stat < chi2.ppf(0.999, df), f"chi2 {stat:.1f} over {df} dof (99.9%: {chi2.ppf(0.999, df):.1f})"


def test_philox_streams_are_distinct():
    """Without slot control every (draw, slot) has its own stream; the RAS re-draw (draw 1) is not the main draw's
    (draw 0) stream. With slot control the stream is the request's: the same (seed, n_out) gives the same token in
    slot 3 and slot 17, another n_out another stream."""
    n = 4097
    h = head(n, True)
    g = torch.Generator().manual_seed(21)
    row = rbf(torch.randn(n, generator=g) * 0.05)
    row[-1] = -1.0  # <|im_end|> out of the top 10
    parts = exact_parts(row.expand(ROWS, n))
    frames = 20
    kw = dict(temperature=1.0, top_p=1.0, top_k=256)
    d0 = draw_many(parts, h, frames, draw_id=0, **kw)
    d2 = draw_many(parts, h, frames, draw_id=1, **kw)
    assert float((d0 == d2).float().mean()) < 0.05, "draw_id 0 and 1 share a stream"
    assert float((d0[:, 0] == d0[:, 1]).float().mean()) < 0.2 and float((d0[:, :-1] == d0[:, 1:]).float().mean()) < 0.05
    # draw 1 of a frame (the RAS re-draw, T = 1, top_p 0.9) against draw 0 with the same parameters: the window holds
    # every survivor of the top 10, so the main token is always replaced by the re-draw
    order = np.argsort(-row.numpy(), kind="stable")[:10]
    top10 = torch.tensor([token_of(int(e), h) for e in order], dtype=torch.int32)
    win = top10.repeat(frames * ROWS, 1).cuda()
    stride = 11
    ct = torch.full((frames, ROWS, stride), -5, dtype=torch.int32, device="cuda")
    offs = torch.arange(frames, dtype=torch.int64, device="cuda")
    a = sample_args(parts, ROWS, h, temperature=1.0, top_p=0.8984375, top_k=10, use_ras=1)
    for f in range(frames):
        a.rng_offset = offs.data_ptr() + 8 * f
        a.cur_tok = ct.data_ptr() + 4 * stride * ROWS * f
        a.ras_window = win.data_ptr() + 4 * 10 * ROWS * f
        run(a)
    d1 = ct.cpu()[:, :, 0]
    plain = draw_many(parts, h, frames, temperature=1.0, top_p=0.8984375, top_k=10)
    assert set(d1.view(-1).tolist()) <= set(top10.tolist())
    assert float((d1 == plain).float().mean()) < 0.3, "the re-draw repeats the main draw's stream"
    # slot control: the request's stream
    rs = torch.tensor([3, 17], dtype=torch.int32, device="cuda")
    a_tok, b_tok = [], []
    for f in range(40):
        ctl = slot_ctl(ROWS, top_k=256, seed=0x1234567890ABCDEF, n_out=f)
        ct = torch.full((ROWS, 11), -5, dtype=torch.int32, device="cuda")
        run(sample_args(parts, 2, h, cur_tok=ct, row_slot=rs, ctl=ctl))
        a_tok.append(int(ct[3, 0]))
        b_tok.append(int(ct[17, 0]))
    assert a_tok == b_tok, "slot 3 and slot 17 of one (seed, n_out) differ"
    assert sum(x == y for x, y in zip(a_tok[:-1], a_tok[1:])) < 4, "n_out does not change the stream"


# ------------------------------------------------------------------------------------------------
# frame_end
# ------------------------------------------------------------------------------------------------
def frame_end(cur_tok, out_tokens, n_out, pos, step, rows, ncols, T_cap, row_slot=None, set_pos_rows=None,
              row_pos_src=None, ctl=None):
    _l, L = _lib()
    c = None
    if ctl is not None:
        c = _l.SlotCtlArgs()
        c.state, c.limit = ctl["state"].data_ptr(), ctl["limit"].data_ptr()
    _l.check(L.fsb_op_frame_end(cur_tok.data_ptr(), out_tokens.data_ptr(), n_out.data_ptr(), pos.data_ptr(),
                                ptr(row_slot), ptr(set_pos_rows), ptr(row_pos_src), step.data_ptr(), rows, ncols, T_cap,
                                C.byref(c) if c is not None else None, _st()))


def _frame_state(slots, ncols, T_cap, n_out):
    cur = torch.arange(slots * ncols, dtype=torch.int32).view(slots, ncols) + 1000
    out = torch.full((slots, ncols, T_cap), -1, dtype=torch.int32)
    return cur, out, torch.tensor(n_out, dtype=torch.int32), torch.arange(slots, dtype=torch.int32) * 10


def test_frame_end_records_and_advances():
    """out_tokens[slot][c][n_out] = cur_tok[slot][c] and n_out + 1 (nothing written once n_out >= T_cap); pos + 1, or
    row_pos_src[set_pos_rows[row]] + 1 in the prefill form; the step counter + 1 per launch."""
    slots, ncols, T_cap = ROWS, 11, 6
    n_out0 = [i % 8 for i in range(slots)]
    cur, out, n_out, pos = _frame_state(slots, ncols, T_cap, n_out0)
    row_slot = [5, 0, 31, 17, 8, 6, 7, 22, 13, 2]
    rows = len(row_slot)
    d = [t.cuda() for t in (cur, out, n_out, pos)]
    step = torch.tensor([41], dtype=torch.int64, device="cuda")
    rs = torch.tensor(row_slot, dtype=torch.int32, device="cuda")
    frame_end(*d, step, rows, ncols, T_cap, row_slot=rs)
    o, no, p = d[1].cpu(), d[2].cpu(), d[3].cpu()
    for s in range(slots):
        if s in row_slot:
            f = n_out0[s]
            want = out[s].clone()
            if f < T_cap:
                want[:, f] = cur[s]
            assert torch.equal(o[s], want), s
            assert int(no[s]) == f + 1 and int(p[s]) == int(pos[s]) + 1, s
        else:
            assert (o[s] == -1).all() and int(no[s]) == n_out0[s] and int(p[s]) == int(pos[s]), s
    assert int(step.cpu()) == 42
    # prefill form
    src = torch.tensor([100, 200, 300, 400], dtype=torch.int32, device="cuda")
    spr = torch.tensor([3, 0, 2], dtype=torch.int32, device="cuda")
    rs = torch.tensor([4, 9, 1], dtype=torch.int32, device="cuda")
    frame_end(*d, step, 3, ncols, T_cap, row_slot=rs, set_pos_rows=spr, row_pos_src=src)
    p = d[3].cpu()
    assert [int(p[4]), int(p[9]), int(p[1])] == [401, 101, 301]
    assert int(step.cpu()) == 43


def test_frame_end_slot_control():
    """State 3 -> 2 and `limit` reached -> 2, both with the position frozen (also in the prefill form); idle (0) and
    finished (2) slots untouched."""
    slots, ncols, T_cap = ROWS, 11, 8
    states0 = [1, 3, 0, 2] * 8
    n_out0 = [2] * slots
    limit = [3 if s % 8 == 4 else 100 for s in range(slots)]  # f + 1 == limit for slots 4, 12, 20, 28
    cur, out, n_out, pos = _frame_state(slots, ncols, T_cap, n_out0)
    d = [t.cuda() for t in (cur, out, n_out, pos)]
    ctl = slot_ctl(slots, state=states0, limit=limit)
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    frame_end(*d, step, slots, ncols, T_cap, ctl=ctl)
    o, no, p, st = d[1].cpu(), d[2].cpu(), d[3].cpu(), ctl["state"].cpu()
    for s in range(slots):
        if states0[s] in (0, 2):
            assert (o[s] == -1).all() and int(no[s]) == 2 and int(p[s]) == int(pos[s]) and int(st[s]) == states0[s], s
            continue
        assert torch.equal(o[s, :, 2], cur[s]) and int(no[s]) == 3, s
        frozen = states0[s] == 3 or limit[s] == 3
        assert int(st[s]) == (2 if frozen else 1), s
        assert int(p[s]) == int(pos[s]) + (0 if frozen else 1), s
    assert int(step.cpu()) == 1
    # prefill form: a frozen slot takes the source position without the + 1
    ctl = slot_ctl(slots, state=[3, 1] + [0] * (slots - 2), limit=100)
    src = torch.tensor([50, 60], dtype=torch.int32, device="cuda")
    spr = torch.tensor([0, 1], dtype=torch.int32, device="cuda")
    frame_end(*d, step, 2, ncols, T_cap, set_pos_rows=spr, row_pos_src=src, ctl=ctl)
    p = d[3].cpu()
    assert [int(p[0]), int(p[1])] == [50, 61]
    assert ctl["state"].cpu()[:2].tolist() == [2, 1]
    assert int(step.cpu()) == 2
