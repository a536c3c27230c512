"""ub_gemm_bf16 against the fp64 reference of tests/gemm_ref.py, element by element, through the C ABI (GemmEpilogue directly, so
that every refusal comes from the library):
  - every tile configuration (128-wide, 256-wide x 1 CTA, CTA pair, cluster of four) x every instantiated epilogue, at the shape
    edges of each (ragged M / N / K, a pair or cluster whose last CTAs hold no valid rows), in child processes that pin the tile
    width with UB_GEMM_BN (read once per process) and confirm from the profiler which kernel ran;
  - the full product of the epilogue options on one small ragged shape: each combination is refused or correct;
  - the grouped GEMMs of the decoders on every configuration;
  - results that must not depend on the grid (ub_set_sm_limit, max_ctas, repeated launches);
  - the shipped shapes at full size.
Outputs are views into larger sentinel-filled buffers (extra rows after M, ld > N): every sentinel must survive."""
import ctypes as C
import itertools
import math
import os
import re
import subprocess
import sys

import pytest
import torch

from tests import gemm_ref as R

pytestmark = pytest.mark.gpu

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
SENTINEL = {BF16: 0x7FA5, F16: 0x7E5A, F32: 0x7FA5A5A5}          # NaNs no kernel produces
GUARD = 8                                                         # guard rows before and after, guard columns after every output


# ---------------------------------------------------------------------------------------------------------------- buffers
def _bits(t):
    return t.view(torch.int32 if t.dtype == F32 else torch.int16)


def _guarded(rows, cols, dtype):
    """(buffer, view): view = rows x cols inside a sentinel-filled buffer with GUARD rows around it and ld = cols + GUARD."""
    buf = torch.empty(rows + 2 * GUARD, cols + GUARD, dtype=dtype, device=DEV)
    _bits(buf).fill_(SENTINEL[dtype])
    return buf, buf[GUARD:GUARD + rows, :cols]


def _guards_intact(buf, rows, cols):
    keep = torch.ones(buf.shape, dtype=torch.bool, device=DEV)
    keep[GUARD:GUARD + rows, :cols] = False
    return bool((_bits(buf)[keep] == SENTINEL[buf.dtype]).all())


def _strided(rows, cols, dtype, gen, scale=1.0, shift=0.0):
    """rows x cols values in a buffer with a wider row pitch (the operand's ld > its width)."""
    ld = (cols + 7) // 8 * 8 + 8
    buf = torch.randn(rows, ld, device=DEV, generator=gen) * scale + shift
    return buf.to(dtype)[:, :cols]


def _ptr(t):
    return t.data_ptr() if t is not None else None


# ---------------------------------------------------------------------------------------------------------------- one call
DEFAULTS = dict(a_mn=False, b_mn=False, ab=BF16, out=BF16, bias=False, act=R.ACT_NONE, aux_out=False, residual=None, alias=False,
                rps=0, accumulate=False, split_k=1, ln=False, stats=False, colsum=False, group=None, dot_seq_len=0, tile_ctas=0,
                max_ctas=0)


class Call:
    """Inputs and guarded outputs of one ub_gemm_bf16 call (case: DEFAULTS overridden), built from a seed."""

    def __init__(self, M, N, K, seed=0, cache=None, **kw):
        c = dict(DEFAULTS, **kw)
        self.c, self.M, self.N, self.K = c, M, N, K
        g = torch.Generator(device=DEV).manual_seed(seed * 1000003 + M * 7919 + N * 131 + K)
        grp = c["group"]
        G = M // grp["rows"] if grp else 1
        a_k_ext, a_m_ext = K + (G - 1) * (grp or {}).get("a_k", 0), (grp or {}).get("a_m", 0) or M
        b_k_ext, b_n_ext = K + (G - 1) * (grp or {}).get("b_k", 0), N + (G - 1) * (grp or {}).get("b_n", 0)
        cache = {} if cache is None else cache          # inputs shared by calls of one shape (the option-space sweep)

        def mk(key, fn):
            if key not in cache:
                cache[key] = fn()
            return cache[key]
        ab = c["ab"]
        ash = (2.0, 0.3) if c["ln"] else (1.0, 0.0)
        ashape = (a_k_ext, a_m_ext) if c["a_mn"] else (a_m_ext, a_k_ext)
        bshape = (b_k_ext, b_n_ext) if c["b_mn"] else (b_n_ext, b_k_ext)
        self.A = mk(("A", ashape, ab, ash), lambda: _strided(*ashape, ab, g, *ash))
        self.B = mk(("B", bshape, ab), lambda: _strided(*bshape, ab, g, 1.0 / math.sqrt(K)))
        nb = N + (G - 1) * (grp or {}).get("bias", 0)
        self.bias = mk(("bias", nb), lambda: torch.randn(nb, device=DEV, generator=g)) if c["bias"] else None
        act = c["act"]
        self.aux_in = mk(("aux", M, N), lambda: _strided(M, N, BF16, g)) if act in (R.ACT_DGELU, R.ACT_DOT_AUX) else None
        self.aux_buf, self.aux_out = _guarded(M, N, BF16) if c["aux_out"] else (None, None)
        self.ld_aux = (self.aux_in if self.aux_in is not None else self.aux_out).stride(0) if (self.aux_in is not None or c["aux_out"]) else 0
        self.cbuf, self.C = _guarded(M, N, c["out"])
        self.c_in = None
        if c["accumulate"] or c["alias"]:
            self.C.copy_(torch.randn(M, N, device=DEV, generator=g))
            self.c_in = self.C.clone()
        self.residual = None
        if c["alias"]:
            self.residual = self.C
        elif c["residual"] == "f32":
            self.residual = mk(("res32", M, N), lambda: _strided(M, N, F32, g))
        elif c["residual"] == "f16":
            self.residual = mk(("res16", M, N), lambda: _strided(M, N, F16, g))
        self.row_scale = None
        if c["rps"]:
            choice = torch.tensor([0.0, 1.0 / 0.9, 0.5, 1.7], device=DEV)
            self.row_scale = mk(("rs", M, c["rps"]), lambda: choice[torch.randint(0, 4, (-(-M // c["rps"]),), device=DEV, generator=g)])
        self.ln = None
        if c["ln"]:
            def fold():
                a = self.A.double()
                stats = torch.stack([a.sum(1), (a * a).sum(1)], 1).float().contiguous()
                return (stats, self.B.double().sum(1).float().contiguous(), float(torch.tensor(1.0 / K, dtype=F32)), 1e-5)
            self.ln = mk(("ln", ashape, bshape, ab), fold)
        self.stats_buf = self.stats = self.stats_in = None
        if c["stats"]:
            self.stats_buf = torch.full((2 * M + 2 * GUARD,), float("nan"), device=DEV)
            self.stats = self.stats_buf[GUARD:GUARD + 2 * M].view(M, 2)
            self.stats.copy_(torch.randn(M, 2, device=DEV, generator=g))
            self.stats_in = self.stats.clone()
        self.colsum_buf = self.colsum = self.colsum_in = None
        if c["colsum"]:
            self.colsum_buf = torch.full((N + 2 * GUARD,), float("nan"), device=DEV)
            self.colsum = self.colsum_buf[GUARD:GUARD + N]
            self.colsum.copy_(torch.randn(N, device=DEV, generator=g))
            self.colsum_in = self.colsum.clone()
        self.dot_buf = self.dot = None
        if act == R.ACT_DOT_AUX:
            n = M * (N // 64)
            self.dot_buf = torch.full((n + 2 * GUARD,), float("nan"), device=DEV)
            self.dot = self.dot_buf[GUARD:GUARD + n]

    def epilogue(self):
        from unite_b200 import _cabi
        c = self.c
        ep = _cabi.GemmEpilogue()
        ep.bias = _ptr(self.bias)
        ep.residual = _ptr(self.residual)
        ep.ldr = self.residual.stride(0) if self.residual is not None else 0
        ep.residual_f16 = int(self.residual is not None and self.residual.dtype == F16)
        ep.row_scale, ep.rows_per_scale = _ptr(self.row_scale), c["rps"]
        ep.aux_in, ep.aux_out, ep.ld_aux = _ptr(self.aux_in), _ptr(self.aux_out), self.ld_aux
        ep.act, ep.out_fp32, ep.accumulate = c["act"], int(c["out"] == F32), int(c["accumulate"])
        ep.tile_ctas, ep.max_ctas, ep.ab_f16 = c["tile_ctas"], c["max_ctas"], int(c["ab"] == F16)
        if self.ln is not None:
            ep.ln_stats, ep.ln_c, ep.ln_inv_d, ep.ln_eps = _ptr(self.ln[0]), _ptr(self.ln[1]), self.ln[2], self.ln[3]
        ep.stats_out, ep.colsum_out = _ptr(self.stats), _ptr(self.colsum)
        ep.dot_out, ep.dot_seq_len = _ptr(self.dot), c["dot_seq_len"]
        grp = c["group"] or {}
        ep.group_rows = grp.get("rows", 0)
        ep.group_a_k, ep.group_a_m, ep.group_b_k = grp.get("a_k", 0), grp.get("a_m", 0), grp.get("b_k", 0)
        ep.group_b_n, ep.group_bias = grp.get("b_n", 0), grp.get("bias", 0)
        return ep

    def launch(self):
        """0 when enqueued, else the library's message."""
        from unite_b200 import _cabi
        lib, c = _cabi.lib, self.c
        ep = self.epilogue()
        rc = lib.ub_gemm_bf16(self.A.data_ptr(), self.A.stride(0), int(c["a_mn"]), self.B.data_ptr(), self.B.stride(0), int(c["b_mn"]),
                              self.C.data_ptr(), self.C.stride(0), self.M, self.N, self.K, C.byref(ep), c["split_k"],
                              torch.cuda.current_stream().cuda_stream)
        return 0 if rc == 0 else lib.ub_last_error().decode()

    def check(self):
        """Failures (strings) of the outputs against the reference; [] when every element is inside its bound."""
        torch.cuda.synchronize()
        c, M, N = self.c, self.M, self.N
        bad = []

        def within(name, got, ref, bound):
            err = (got.double() - ref).abs()
            ok = err <= bound
            if not bool(ok.all()):
                idx = (~ok).nonzero()[0].tolist()
                r = R.ratio(err, bound)
                bad.append(f"{name}: {int((~ok).sum())} of {ok.numel()} elements outside their bound, worst "
                           f"{float(r.nan_to_num(float('inf')).max()):.3g} x bound, first at {idx}: got {float(got[tuple(idx)])} "
                           f"want {float(ref[tuple(idx)]):.6g} +- {float(bound[tuple(idx)]):.3g}")

        if not _guards_intact(self.cbuf, M, N):
            bad.append("C: a sentinel outside the output was overwritten")
        if self.aux_buf is not None and not _guards_intact(self.aux_buf, M, N):
            bad.append("aux_out: a sentinel outside the output was overwritten")
        for name, buf in (("stats_out", self.stats_buf), ("colsum_out", self.colsum_buf), ("dot_out", self.dot_buf)):
            if buf is not None and not bool(torch.isnan(buf[:GUARD]).all() and torch.isnan(buf[-GUARD:]).all()):
                bad.append(f"{name}: a sentinel outside the output was overwritten")
        ref = R.gemm(self.A, self.B, M, N, self.K, c["a_mn"], c["b_mn"], bias=self.bias, act=c["act"], aux_in=self.aux_in,
                     row_scale=self.row_scale, rows_per_scale=max(1, c["rps"]),
                     residual=self.c_in if c["alias"] else self.residual, c_in=self.c_in if c["accumulate"] else None,
                     out_dtype=c["out"], split_k=c["split_k"], ln=self.ln, colsum_in=self.colsum_in, group=c["group"])
        within("C", self.C, ref["c"], ref["c_bound"])
        if self.aux_out is not None:
            within("aux_out", self.aux_out, ref["aux"], ref["aux_bound"])
        if self.colsum is not None:
            within("colsum_out", self.colsum, ref["colsum"], ref["colsum_bound"])
        if self.stats is not None:
            sref, sb = R.row_stats(self.C, self.stats_in)
            within("stats_out", self.stats, sref, sb)
        if self.dot is not None:
            dref, db = R.head_dot(self.C, self.aux_in, c["dot_seq_len"])
            within("dot_out", self.dot.view(dref.shape), dref, db)
        return bad

    def outputs(self):
        return [t.clone() for t in (self.C, self.aux_out, self.colsum, self.stats, self.dot) if t is not None]


def run_one(M, N, K, **kw):
    call = Call(M, N, K, **kw)
    msg = call.launch()
    assert msg == 0, f"refused: {msg}"
    bad = call.check()
    assert not bad, f"M={M} N={N} K={K} {kw}:\n  " + "\n  ".join(bad)
    return call


# ---------------------------------------------------------------------------------------------------------------- configurations
M_EDGES = [1, 127, 129, 257, 260, 513, 640, 1000]
N_EDGES = [8, 120, 136, 264, 320, 392]
K_EDGES = [8, 56, 72, 200]                  # K-major operands
T_EDGES = [1, 7, 65]                        # token counts: K of MN-major operands

# (name, case options, N restriction): the epilogues launch_gemm instantiates per operand-major form
EPILOGUES = [
    ("NT bf16", dict(), None),
    ("NT bf16 bias+GELU", dict(bias=True, act=R.ACT_GELU), None),
    ("NT fp32", dict(out=F32), None),
    ("NT fp32 residual+DropPath", dict(out=F32, bias=True, residual="f32", rps=7), None),
    ("NT fp32 residual aliasing C", dict(out=F32, bias=True, alias=True), None),
    ("NT DGELU", dict(act=R.ACT_DGELU, rps=5), None),
    ("NT DOT_AUX", dict(act=R.ACT_DOT_AUX, bias=True), 64),
    ("NT fp16 residual+stats", dict(out=F16, bias=True, residual="f16", stats=True), None),
    ("NT fp16 operands, fp16 residual+stats", dict(ab=F16, out=F16, bias=True, residual="f16", stats=True), None),
    ("NT bf16 bias+GELU+pre-activation copy", dict(bias=True, act=R.ACT_GELU, aux_out=True, rps=3), None),
    ("NT fp16 operands, LN fold+QuickGELU", dict(ab=F16, ln=True, bias=True, act=R.ACT_QUICKGELU), None),
    ("NT fp16 operands, LN fold", dict(ab=F16, ln=True, bias=True), None),
    ("NT bf16 operands, LN fold+QuickGELU", dict(ln=True, bias=True, act=R.ACT_QUICKGELU), None),
    ("NN bf16", dict(b_mn=True), None),
    ("NN DGELU+colsum", dict(b_mn=True, act=R.ACT_DGELU, colsum=True), None),
    ("TN fp32", dict(a_mn=True, b_mn=True, out=F32), None),
    ("TN fp32 accumulate", dict(a_mn=True, b_mn=True, out=F32, accumulate=True), None),
    ("TN fp32 accumulate split-K 3", dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=3), None),
    ("TN fp32 accumulate, more splits than k-blocks", dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=9), None),
]


def _config(bn, ctas, M, N, group_rows, cap4):
    """(BN, NCTA) the host must pick in a process with UB_GEMM_BN=bn for tile_ctas=ctas."""
    if bn == 128 or N <= 128:
        return 128, 1
    ncta = {1: 1, 2: 2 if M > 128 else 1, 4: 4 if (M >= 512 and cap4 > 0) else (2 if M > 128 else 1)}[ctas]
    if ncta == 4 and group_rows % 512:
        ncta = 2
    return 256, ncta


def table(bn, ctas):
    """[(name, M, N, K, options)] of one configuration: every epilogue at the M edges the configuration can take, cycling N and K."""
    if bn == 128:
        ms, ns = M_EDGES, N_EDGES
    else:
        ms = [m for m in M_EDGES if (ctas == 1 or m > 128) and (ctas != 4 or m >= 512)]
        ns = [n for n in N_EDGES if n > 128]
    cases = []
    for e, (name, opt, nmul) in enumerate(EPILOGUES):
        for i, M in enumerate(ms):
            N = ns[(i + e) % len(ns)]
            if nmul:
                N = max(64 * (N // 64), 64 if bn == 128 else 192)
            kl = T_EDGES + K_EDGES[-1:] if opt.get("b_mn") else K_EDGES
            if opt.get("b_mn") and not opt.get("a_mn"):
                kl = T_EDGES + K_EDGES
            K = kl[(i + 2 * e) % len(kl)]
            o = dict(opt, tile_ctas=ctas if bn == 256 else 0)
            if opt.get("act") == R.ACT_DOT_AUX:
                o["dot_seq_len"] = M // 2 if M % 2 == 0 else M
            cases.append((name, M, N, K, o))
    # the strided / aliasing edges once more on a shape every configuration takes, and the decoders' grouped calls
    for gr in (256, 512, 768, 1024, 1280):
        n_out, d = (264, 320) if bn == 256 else (120, 136)
        cases.append((f"grouped fwd rows={gr}", 2 * gr, n_out, 128,
                      dict(bias=True, out=F32, group=dict(rows=gr, b_n=n_out, bias=n_out + 8), tile_ctas=ctas if bn == 256 else 0)))
        cases.append((f"grouped dgrad rows={gr}", 2 * gr, d, 128,
                      dict(b_mn=True, group=dict(rows=gr, b_k=128), tile_ctas=ctas if bn == 256 else 0)))
        cases.append((f"grouped wgrad rows={gr}", 2 * gr, d, 192,
                      dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=2, group=dict(rows=gr, a_k=192, a_m=gr, b_k=192),
                           tile_ctas=ctas if bn == 256 else 0)))
    return cases


_KNAME = [re.compile(r"gemm_kernel<(\d+), \d+, (?:true|false), (?:true|false), \d, (?:true|false), (\d)>"),
          re.compile(r"gemm_kernelILi(\d+)ELi\d+ELb[01]ELb[01]ELi\dELb[01]ELi(\d)E")]


def _kernel_config(fn):
    """(BN, NCTA) of the gemm_kernel instantiations fn launches, from the profiler's kernel names."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for ev in prof.events():
        for rx in _KNAME:
            m = rx.search(ev.name)
            if m:
                found.add((int(m.group(1)), int(m.group(2))))
    return found


def child_main(bn):
    """Runs the case table of every configuration of this process's tile width; prints one line per failure, exits 1 on any."""
    from unite_b200 import _cabi
    cap4 = _cabi.lib.ub_gemm_cluster4_capacity()
    assert cap4 > 0, "the device holds no cluster of four GEMM CTAs"
    fails, n = [], 0
    for ctas in ((0,) if bn == 128 else (1, 2, 4)):
        seen = set()
        for name, M, N, K, o in table(bn, ctas):
            want = _config(bn, ctas, M, N, (o.get("group") or {}).get("rows", 0), cap4)
            call = Call(M, N, K, seed=n, **o)
            n += 1
            tag = f"[BN={bn} tile_ctas={ctas}] {name} M={M} N={N} K={K}"
            msg = []
            if want not in seen:
                got = _kernel_config(lambda: msg.append(call.launch()))
                seen.add(want)
                if msg[0] == 0 and got != {want}:
                    fails.append(f"{tag}: ran {sorted(got)}, expected BN, NCTA = {want}")
            else:
                msg.append(call.launch())
            if msg[0] != 0:
                fails.append(f"{tag}: refused: {msg[0]}")
                continue
            for b in call.check():
                fails.append(f"{tag}: {b}")
        print(f"BN={bn} tile_ctas={ctas}: configurations seen {sorted(seen)}", flush=True)
    print(f"{n} cases, {len(fails)} failures", flush=True)
    for f in fails:
        print("FAIL " + f, flush=True)
    sys.exit(1 if fails else 0)


@pytest.mark.parametrize("bn", [128, 256])
def test_every_configuration_and_epilogue(bn):
    env = dict(os.environ, UB_GEMM_BN=str(bn))
    env.pop("UB_GEMM_NCTA", None)
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from tests import test_gemm_edges_gpu as T; T.child_main({bn})"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    print(r.stdout[-6000:])
    assert r.returncode == 0, (r.stdout[-6000:], r.stderr[-3000:])


# ---------------------------------------------------------------------------------------------------------------- option space
FORMS = {"NT": (False, False), "NN": (False, True), "TN": (True, True)}


@pytest.mark.parametrize("form", list(FORMS))
def test_every_epilogue_option_combination_is_refused_or_correct(form):
    a_mn, b_mn = FORMS[form]
    flags = itertools.product([False, True], [None, "f32", "f16"], [0, 3], range(5), [False, True], [False, True], [1, 3],
                              [False, True], [False, True], [False, True], [False, True], [BF16, F32], [BF16, F16])
    accepted, refused, fails, cache = 0, 0, [], {}
    for (bias, res, rps, act, aux_out, acc, split, ln, stats, colsum, grouped, out, ab) in flags:
        if grouped:
            M, N, K = 512, 192, 192
            group = {"NT": dict(rows=256, b_n=N, bias=N), "NN": dict(rows=256, b_k=K),
                     "TN": dict(rows=256, a_k=K, a_m=256, b_k=K)}[form]
        else:
            M, N, K, group = 260, 192, 200, None
        if res == "f16" and out != F32:
            out = F16                        # a 2-byte C is fp16 exactly when the residual is
        o = dict(a_mn=a_mn, b_mn=b_mn, ab=ab, out=out, bias=bias, act=act, aux_out=aux_out, residual=res, rps=rps, accumulate=acc,
                 split_k=split, ln=ln, stats=stats, colsum=colsum, group=group, dot_seq_len=130)
        call = Call(M, N, K, cache=cache, **o)
        msg = call.launch()
        if msg != 0:
            refused += 1
            continue
        accepted += 1
        for b in call.check():
            fails.append(f"{o}: {b}")
    print(f"\n{form}: {accepted} combinations accepted and checked, {refused} refused")
    assert not fails, f"{len(fails)} accepted combinations are wrong, e.g.\n" + "\n".join(fails[:8])


def test_refusals():
    # max_ctas < 0 has no meaning
    call = Call(256, 256, 128, max_ctas=-1)
    assert call.launch() != 0
    # split_k > 1 with a bias or an activation, unless the clamp to the k-blocks leaves one split
    assert Call(256, 256, 128, a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=2, bias=True).launch() != 0
    assert Call(256, 256, 128, out=F32, accumulate=True, split_k=2, act=R.ACT_GELU).launch() != 0
    run_one(256, 256, 64, out=F32, accumulate=True, split_k=4, bias=True, act=R.ACT_GELU)
    # DGELU with a bias
    assert Call(256, 256, 128, act=R.ACT_DGELU, bias=True).launch() != 0
    assert Call(260, 256, 128, b_mn=True, act=R.ACT_DGELU, bias=True, colsum=True).launch() != 0


# ---------------------------------------------------------------------------------------------------------------- grid independence
@pytest.fixture
def sm_limit():
    """Sets the library's persistent-grid size (0 = the whole device) and restores it."""
    from unite_b200 import _cabi
    lib = _cabi.lib
    full = lib.ub_set_sm_limit(0)

    def set_limit(n):
        got = lib.ub_set_sm_limit(n)
        assert got == (n if n else full), f"ub_set_sm_limit({n}) gave {got}"
    try:
        yield set_limit
    finally:
        lib.ub_set_sm_limit(0)


GRID_CASES = [
    ("NT GELU + pre-activation copy", 1000, 392, 200, dict(bias=True, act=R.ACT_GELU, aux_out=True), True),
    ("NT pair fp32 residual", 1000, 392, 200, dict(bias=True, out=F32, residual="f32", tile_ctas=2), True),
    ("NN 128-wide", 1000, 120, 72, dict(b_mn=True), True),
    ("TN accumulate", 392, 264, 1000, dict(a_mn=True, b_mn=True, out=F32, accumulate=True), True),
    ("TN accumulate split-K 3", 392, 264, 1000, dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=3), False),
    ("NN DGELU colsum", 1000, 264, 72, dict(b_mn=True, act=R.ACT_DGELU, colsum=True), False),
    ("NT fp16 residual stats", 1000, 264, 200, dict(out=F16, bias=True, residual="f16", stats=True), False),
]


@pytest.mark.parametrize("name,M,N,K,o,plain", GRID_CASES, ids=[c[0] for c in GRID_CASES])
def test_results_do_not_depend_on_the_grid(sm_limit, name, M, N, K, o, plain):
    """Plain stores: bit-identical over grids and launches.  Atomically reduced outputs (split-K, colsum_out, stats_out): each
    within its bound of the reference."""
    first = None
    for limit, max_ctas in [(0, 0), (146, 0), (74, 0), (16, 0), (2, 0), (0, 1), (0, 3), (0, 64)]:
        sm_limit(limit)
        for rep in range(2):
            call = run_one(M, N, K, seed=1, max_ctas=max_ctas, **o)
            if plain:
                outs = call.outputs()
                if first is None:
                    first = outs
                for x, y in zip(outs, first):
                    assert torch.equal(_bits(x), _bits(y)), f"{name}: differs at sm_limit={limit} max_ctas={max_ctas} (launch {rep})"


def test_multi_problem_weight_gradient_does_not_depend_on_the_grid(sm_limit):
    from unite_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(5)
    K, widths = 1000, [(200, 328), (512, 64), (8, 1032)]
    data = [((torch.randn(K, M, device=DEV, generator=g) * 0.5).bfloat16(), (torch.randn(K, N, device=DEV, generator=g) * 0.5).bfloat16(),
             torch.randn(M, N, device=DEV, generator=g)) for M, N in widths]
    first = None
    for limit in (0, 146, 74, 16, 2):
        sm_limit(limit)
        for rep in range(2):
            probs = [(dy, x, gw.clone()) for dy, x, gw in data]
            ops.gemm_wgrad_multi(probs, split_k=1)
            torch.cuda.synchronize()
            outs = [p[2] for p in probs]
            if first is None:
                first = outs
                for (dy, x, gw0), got in zip(data, outs):
                    r = R.gemm(dy, x, dy.shape[1], x.shape[1], K, True, True, c_in=gw0, out_dtype=F32)
                    assert bool(((got.double() - r["c"]).abs() <= r["c_bound"]).all())
            for a, b in zip(outs, first):
                assert torch.equal(_bits(a), _bits(b)), f"ub_gemm_wgrad_multi differs at sm_limit={limit} (launch {rep})"


# ---------------------------------------------------------------------------------------------------------------- shipped shapes
SHIPPED = [
    # (name, M, N, K, options): profiles/gemm_shapes_r02_final.json with the epilogue of each call site, and the teacher's fp16 stream
    ("teacher conv1", 50176, 768, 768, dict(out=F32)),
    ("teacher in_proj, LN fold", 50432, 2304, 768, dict(ab=F16, ln=True, bias=True)),
    ("teacher out_proj, fp16 residual + stats", 50432, 768, 768, dict(out=F16, bias=True, residual="f16", stats=True)),
    ("teacher c_fc, LN fold + QuickGELU", 50432, 3072, 768, dict(ab=F16, ln=True, bias=True, act=R.ACT_QUICKGELU)),
    ("teacher c_proj, fp16 residual + stats", 50432, 768, 3072, dict(out=F16, bias=True, residual="f16", stats=True)),
    ("student qkv", 10240, 2304, 768, dict(bias=True)),
    ("student proj, residual + DropPath", 10240, 768, 768, dict(out=F32, bias=True, residual="f32", rps=320)),
    ("student fc1, GELU + pre-activation", 10240, 3072, 768, dict(bias=True, act=R.ACT_GELU, aux_out=True)),
    ("student fc2, residual + DropPath", 10240, 768, 3072, dict(out=F32, bias=True, residual="f32", rps=320)),
    ("student bf16 out", 10240, 768, 3072, dict(bias=True)),
    ("student bf16 out, K 768", 10240, 768, 768, dict()),
    ("fc2 dgrad, DGELU + colsum", 10240, 3072, 768, dict(b_mn=True, act=R.ACT_DGELU, colsum=True)),
    ("fc1 dgrad", 10240, 768, 3072, dict(b_mn=True)),
    ("qkv dgrad", 10240, 768, 2304, dict(b_mn=True)),
    ("proj dgrad, DOT_AUX", 10240, 768, 768, dict(b_mn=True, act=R.ACT_DOT_AUX, dot_seq_len=320)),
    ("decoder heads, grouped", 61440, 512, 768, dict(out=F32, bias=True, group=dict(rows=10240, b_n=512, bias=512))),
    ("decoder dgrad, grouped", 61440, 768, 512, dict(b_mn=True, group=dict(rows=10240, b_k=512))),
    ("decoder wgrad, grouped", 3072, 768, 10240, dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=2,
                                                       group=dict(rows=512, a_k=10240, a_m=512, b_k=10240))),
    ("wgrad 3072 x 768", 3072, 768, 10240, dict(a_mn=True, b_mn=True, out=F32, accumulate=True)),
    ("wgrad 768 x 768", 768, 768, 10240, dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=2)),
    # the shapes the earlier relative-norm check ran
    ("square", 128, 128, 64, dict()),
    ("wide", 128, 256, 256, dict()),
    ("fp32", 256, 512, 768, dict(out=F32)),
    ("ragged fp32", 200, 264, 200, dict(out=F32)),
    ("fp32 bias + residual", 1000, 768, 768, dict(out=F32, bias=True, residual="f32")),
    ("bias", 2048, 2304, 768, dict(bias=True)),
    ("bias + QuickGELU", 2048, 3072, 768, dict(bias=True, act=R.ACT_QUICKGELU)),
    ("bias + GELU", 2048, 3072, 768, dict(bias=True, act=R.ACT_GELU)),
    ("dgrad", 256, 256, 128, dict(b_mn=True)),
    ("dgrad 2048", 2048, 768, 3072, dict(b_mn=True)),
    ("wgrad store", 256, 256, 256, dict(a_mn=True, b_mn=True, out=F32)),
    ("wgrad split-K 4", 768, 768, 4096, dict(a_mn=True, b_mn=True, out=F32, accumulate=True, split_k=4)),
]


@pytest.mark.parametrize("name,M,N,K,o", SHIPPED, ids=[s[0] for s in SHIPPED])
def test_shipped_shapes(name, M, N, K, o):
    run_one(M, N, K, seed=3, **o)


def test_shipped_multi_problem_weight_gradient():
    """The four weight gradients of a ViT-B block in one ub_gemm_wgrad_multi launch over 10240 tokens."""
    from unite_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(9)
    K = 10240
    probs, refs = [], []
    for M, N in ((2304, 768), (768, 768), (3072, 768), (768, 3072)):
        dy = (torch.randn(K, M, device=DEV, generator=g) * 0.5).bfloat16()
        x = (torch.randn(K, N, device=DEV, generator=g) * 0.5).bfloat16()
        gw = torch.randn(M, N, device=DEV, generator=g)
        refs.append(R.gemm(dy, x, M, N, K, True, True, c_in=gw.clone(), out_dtype=F32, split_k=2))
        probs.append((dy, x, gw))
    ops.gemm_wgrad_multi(probs, split_k=2)
    torch.cuda.synchronize()
    for (_, _, gw), r in zip(probs, refs):
        assert bool(((gw.double() - r["c"]).abs() <= r["c_bound"]).all())
