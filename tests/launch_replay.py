"""Launch replay: every kernel launch of a real forward (or train step) checked against a high-precision
reference of its contract, on the launch's own inputs.

A Recorder wraps the launchers of diffusion_pruning_b200.kernels (the engine and train.py call them as
`K.<fn>`). For each launch it snapshots the storage of every tensor argument (tensors that share a storage,
such as an in-place residual or the q / k / v column blocks of one buffer, map to one copy), runs the real
kernel, synchronizes, then runs the reference of tests/cpu_kernel_sim.py on the snapshot in float64 (or
float32 without TF32) and compares:

- every element the reference writes, against its unrounded value, with a tolerance scaled to the launch's
  output (TOL_RULES, bounded per feature group by BOUNDS);
- every other byte of every argument storage: it must be bit-identical to the pre-launch snapshot (columns
  past n_store, neighbouring column blocks, rows of inactive buckets, pruned heads, ...).

Per-sample GroupNorm column-statistic planes are compared as sums over the blocks of each sample: the block
order of conv boxes is not part of the contract. Launchers without a reference run unchecked and are counted.
Each grouped-GEMM launch is also tagged with the features it exercises (scheme, boxes, placeholder tiles,
epilogues, ...) so a test can assert that the launches it claims to check were issued."""
from __future__ import annotations

import ast
import collections
import contextlib
import inspect
import json
import math
import os

import numpy as np
import torch

import cpu_kernel_sim as S
from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200._lib import (A_CONV3X3, A_CONV3X3_S2, A_LINEAR, EPI_GEGLU, EPI_RES_F32, OUT_BF16,
                                         OUT_F32_NCHW)

# launchers with a reference in cpu_kernel_sim (same name, same signature)
CHECKED = ("grouped_gemm", "groupnorm_stats", "groupnorm_stats_from_partials", "groupnorm_apply", "layernorm",
           "ln_rowstats", "depth_lerp", "copy_rows", "copy_rows_cvt", "depth_lerp_f32", "upsample2x_cvt",
           "upsample2x", "im2col_input", "timestep_embedding", "cast_f32_bf16", "silu_bf16", "attention",
           "attention_bwd", "wgrad")
_NOT_LAUNCHERS = {"gemm_max_pairs", "check_abort", "poll_abort", "build_schedule", "upload", "conv_box"}
MIN_2SM_K = 1280   # taps * a_k from which aptp_grouped_gemm_fwd takes the 2-SM scheme (library default)


def launchers():
    """Public top-level functions of kernels.py (read from its source: the module may be monkey-patched)."""
    tree = ast.parse(open(K.__file__).read())
    return [n.name for n in tree.body if isinstance(n, ast.FunctionDef) and not n.name.startswith("_")
            and n.name not in _NOT_LAUNCHERS]


# ------------------------------------------------------------------------------------------------
# tolerances: ratio = max |got - ref| / tol(ref); a launch passes when ratio <= BOUNDS[group]
# ------------------------------------------------------------------------------------------------
def _tol(ref: torch.Tensor, dtype, k: int, floor: float = 0.0) -> torch.Tensor:
    rms = ref.pow(2).mean().sqrt()
    if dtype == torch.bfloat16:   # one bf16 rounding of the result plus accumulation noise of the launch's scale
        return 2.0 ** -8 * ref.abs() + 1e-3 * rms + floor
    return 1e-5 * ref.abs() + 1e-6 * math.sqrt(max(k, 1)) * rms + floor   # fp32: relative + length-scaled absolute


TOL_RULES = ("bf16: 2^-8 |ref| + 1e-3 rms(ref);  fp32: 1e-5 |ref| + 1e-6 sqrt(K) rms(ref);  attention + 2^-8 rms(V), "
             "attention_bwd + 2^-5 rms(grad);  zero padding exact")
# 2..4 x the worst ratio of each group over all cases of tests/test_launch_replay_gpu.py on a B200 (1000 W), groups
# not seen there keep 2.5. Every bf16 bound stays <= 2.5, so a written bf16 value is held to 1 % of |ref| + 0.25 %
# of the region's rms, tighter than the 1e-2 relative / 2e-2 absolute of tests/kernel_checks.py; 2.5 is also what
# lets a 4-ulp error be caught (tests/test_launch_replay_cpu.py).
BOUNDS = collections.defaultdict(lambda: 2.5, {
    "gemm 1sm plain f32": 0.5,                  # worst 0.124
    "gemm 2sm plain f32": 2.0,                  # worst 0.542
    "gemm colstat": 4.0,                        # worst 1.770
    "gemm rowstat": 2.0,                        # worst 0.617
    "groupnorm_stats f32": 0.075,               # worst 0.019
    "groupnorm_stats_from_partials f32": 0.15,  # worst 0.039
    "ln_rowstats f32": 0.075,                   # worst 0.019
    "depth_lerp_f32 f32": 0.25,                 # worst 0.065
    "copy_rows_cvt f32": 0.01,                  # exact copies (worst 0)
    "attention bf16": 2.5,                      # worst 0.793 (with the 2^-8 rms(V) floor)
    "attention lse f32": 0.05,                  # worst 0.016
    "attention_bwd grad bf16": 2.5,             # worst 6.7 under a 2^-8 rms floor, i.e. ~3 % of rms: floor now 2^-5
    "attention_bwd delta f32": 0.15,            # worst 0.044
    "wgrad f32": 0.4,                           # worst 0.123
    "wgrad bias f32": 0.12,                     # worst 0.035
})


def group_of(name: str, dtype, meta: dict, tags=()) -> str:
    if name == "grouped_gemm":
        scheme = "2sm" if "2sm" in tags else "1sm"
        if "blocks" in meta:
            return "gemm colstat"
        if meta.get("part") == "rowstat":
            return "gemm rowstat"
        kind = "geglu" if "geglu" in tags else ("lnfold" if "lnfold" in tags else "plain")
        return f"gemm {scheme} {kind} {'bf16' if dtype == torch.bfloat16 else 'f32'}"
    part = f" {meta['part']}" if "part" in meta else ""
    return f"{name}{part} {'bf16' if dtype == torch.bfloat16 else 'f32'}"


# ------------------------------------------------------------------------------------------------
# grouped-GEMM feature tags
# ------------------------------------------------------------------------------------------------
def _tile_width(sched, tiles_of_seg, geglu):
    w32 = int(tiles_of_seg[0, 3] >> 8) & 0xFF
    width = w32 * 32 if w32 else sched.bn
    return (width // 2 if geglu else width), bool(w32)


def gemm_tags(kw: dict, sched) -> set:
    mode = kw.get("mode", A_LINEAR)
    taps = 1 if mode == A_LINEAR else 9
    geglu = bool(kw.get("flags", 0) & EPI_GEGLU)
    two = sched.a_stat == 0 and taps * kw["a_k"] >= MIN_2SM_K
    tags = {"2sm" if two else "1sm", {A_LINEAR: "linear", A_CONV3X3: "conv", A_CONV3X3_S2: "conv_s2"}[mode]}
    if mode != A_LINEAR:
        tags.add("box%dx%dx%d" % tuple(sched.box))
        if two and mode == A_CONV3X3 and tuple(sched.box) == (8, 16, 1) and os.environ.get("APTP_CONV_HALO", "1") != "0":
            tags.add("halo")
    segs = sched.segs.cpu().numpy()[:sched.n_segs]
    tiles = sched.tiles.cpu().numpy()
    live = tiles[(tiles[:, 3] & K.TILE_SKIP) == 0]
    act = np.unique(live[:, 0])
    if len(act) > 1:
        tags.add("multiseg")
    if len(act) < sched.n_segs:
        tags.add("inactive_seg")
    if (live[:, 3] & K.TILE_PLACEHOLDER).any():
        tags.add("placeholder")
    if (len(live) // 2) % 2:
        tags.add("odd_pairs")
    for si in act:
        rb, re, nv, ns = (int(v) for v in segs[si][:4])
        if mode == A_LINEAR and rb % 128:
            tags.add("unaligned_start")
        width, balanced = _tile_width(sched, live[live[:, 0] == si], geglu)
        nt = len(np.unique(live[live[:, 0] == si][:, 2]))
        if balanced:
            tags.add("balanced")
        if nt * width > max(nv, ns):
            tags.add("ragged")
        if int(segs[si][8]) > 0:
            tags.add("col_off")
    for key, tag in (("ln_rowstats", "lnfold"), ("rowstat_out", "rowstat"), ("colstat", "colstat"), ("a2", "a2"),
                     ("gate", "gate"), ("residual", "residual"), ("rowvec", "rowvec"), ("border_tab", "border")):
        if kw.get(key) is not None:
            tags.add(tag)
    if geglu:
        tags.add("geglu")
    if kw.get("flags", 0) & EPI_RES_F32:
        tags.add("res_f32")
    if kw.get("out_mode", OUT_BF16) == OUT_F32_NCHW:
        tags.add("nchw")
    if sched.a_stat > 0:
        tags.add("a_stat")
    if sched.n_tiles // 2 > K.gemm_max_pairs():
        tags.add("multi_tile_pairs")
    return tags


def _tile_at(sched, kw, si, row, col):
    """(row base, column base) of the tile of segment `si` that covers output (row, col), or None."""
    mode = kw.get("mode", A_LINEAR)
    geglu = bool(kw.get("flags", 0) & EPI_GEGLU)
    tiles = sched.tiles.cpu().numpy()
    mine = tiles[((tiles[:, 3] & K.TILE_SKIP) == 0) & (tiles[:, 0] == si)]
    if len(mine) == 0:
        return None
    oco = int(sched.segs.cpu().numpy()[si][8])
    width, _ = _tile_width(sched, mine, geglu)
    stride = 2 if mode == A_CONV3X3_S2 else 1
    Ho, Wo = kw.get("H", 1) // stride, kw.get("W", 1) // stride
    bw, bh, bb = sched.box
    base = None
    for m in np.unique(mine[:, 1]):
        if mode == A_LINEAR:
            hit = m <= row < m + 128
        else:
            img0, rem = divmod(int(m), Ho * Wo)
            oy0, ox0 = divmod(rem, Wo)
            img, rem = divmod(int(row), Ho * Wo)
            oy, ox = divmod(rem, Wo)
            hit = img0 <= img < img0 + bb and oy0 <= oy < oy0 + bh and ox0 <= ox < ox0 + bw
        if hit:
            base = int(m)
            break
    n0 = ((col - oco) // width) * width + oco if col >= oco else None
    return base, n0


# ------------------------------------------------------------------------------------------------
# snapshots
# ------------------------------------------------------------------------------------------------
def _tensors(obj):
    if torch.is_tensor(obj):
        yield obj
    elif isinstance(obj, (tuple, list)):
        for o in obj:
            yield from _tensors(o)


def _as(storage, t_like_dtype, offset, size, stride, device):
    return torch.empty(0, dtype=t_like_dtype, device=device).set_(storage, offset, size, stride)


class _Snapshot:
    """One copy per distinct storage among the tensor arguments; args remapped onto the copies."""

    def __init__(self, bound: dict):
        self.stores = {}   # data_ptr -> [original storage, copy, first (argument name, tensor)]
        self.args = {k: self._map(k, v) for k, v in bound.items()}

    def _map(self, name, v):
        if torch.is_tensor(v):
            if v.untyped_storage().nbytes() == 0:
                return v
            st = v.untyped_storage()
            ent = self.stores.get(st.data_ptr())
            if ent is None:
                ent = self.stores[st.data_ptr()] = [st, st.clone(), (name, v)]
            return _as(ent[1], v.dtype, v.storage_offset(), v.size(), v.stride(), v.device)
        if isinstance(v, tuple):
            return tuple(self._map(name, o) for o in v)
        if isinstance(v, list):
            return [self._map(name, o) for o in v]
        return v

    def copy_of(self, t: torch.Tensor):
        """The snapshot entry whose copy `t` lives in."""
        for ent in self.stores.values():
            if ent[1].data_ptr() == t.untyped_storage().data_ptr():
                return ent
        return None

    def original(self, t: torch.Tensor):
        return self.stores.get(t.untyped_storage().data_ptr())


class ReplayFailure(AssertionError):
    pass


class Recorder:
    """Wraps the kernel launchers; see the module docstring. `fault(rec, name, args, snap)` (tests only) runs after
    the device launch and may alter device tensors, so that the harness' own detection can be checked."""

    def __init__(self, cdt=torch.float64, label=lambda: "", fault=None, bounds=None):
        self.cdt = cdt
        self.label = label
        self.fault = fault
        self.bounds = bounds if bounds is not None else BOUNDS
        self.lines = []          # per launch: dict(i, fn, label, tags, ratio, group ratios)
        self.failures = []
        self.counts = collections.Counter()
        self.unchecked = collections.Counter()
        self.worst = {}          # group -> (ratio, launch index)
        self.tally = collections.Counter()
        self.phase = "fwd"       # set to "bwd" by a caller around a backward pass: GEMM launches then carry a "bwd" tag
        self._orig = {}

    # ---- installation -------------------------------------------------------------------------------------
    def install(self, setattr_fn):
        for name in launchers():
            dev = getattr(K, name)
            self._orig[name] = dev
            ref = getattr(S, name) if name in CHECKED else None
            setattr_fn(K, name, self._wrap(name, dev, ref))
        return self

    def _wrap(self, name, dev, ref):
        sig = inspect.signature(dev)

        def launch(*args, **kwargs):
            return self._launch(name, dev, ref, sig, args, kwargs)
        launch.__name__ = name
        return launch

    # ---- one launch -------------------------------------------------------------------------------------
    def _sync(self, device):
        if device.type == "cuda":
            torch.cuda.synchronize(device)
        K.check_abort()

    def _launch(self, name, dev, ref, sig, args, kwargs):
        self.counts[name] += 1
        if ref is None:
            self.unchecked[name] += 1
            return dev(*args, **kwargs)
        bound = sig.bind(*args, **kwargs)
        bound.apply_defaults()
        bargs = dict(bound.arguments)
        ts = [t for v in bargs.values() for t in _tensors(v)]
        device = ts[0].device if ts else torch.device("cpu")
        if name == "grouped_gemm" and bargs["sched"].n_tiles == 0:
            return dev(*args, **kwargs)
        self._sync(device)
        snap = _Snapshot(bargs)
        dev(*args, **kwargs)
        self._sync(device)
        i = len(self.lines)
        if self.fault is not None:
            self.fault(self, name, bargs, snap)
        tags = ()
        if name == "grouped_gemm":
            kw = {k: v for k, v in bargs.items() if k not in ("a", "w", "out", "sched")}
            tags = gemm_tags(kw, bargs["sched"]) | ({"bwd"} if self.phase == "bwd" else set())
            self.tally[" ".join(sorted(tags))] += 1
        elif name == "wgrad":
            conv = bargs["conv"]
            tags = {"wgrad", "linear" if conv is None else ("conv" if bargs["stride"] == 1 else "conv_s2")}
            if max(bargs["n_out"], bargs["k_in"]) >= 1280:
                tags.add("width1280")
            self.tally[" ".join(sorted(tags))] += 1
        label = self.label()
        ctx = torch.backends.cudnn.flags(enabled=False) if device.type == "cuda" else contextlib.nullcontext()
        tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            with ctx, S.reference_mode(self.cdt) as writes:
                ref(**snap.args)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = tf32
        line = dict(i=i, fn=name, label=label, tags=sorted(tags), ratio=0.0)
        self._compare(name, bargs, snap, writes, tags, line)
        self.lines.append(line)

    # ---- comparison ------------------------------------------------------------------------------------------
    def _where(self, name, bargs, meta, idx):
        """Human-readable position of element `idx` (multi-index into a written region)."""
        if name == "grouped_gemm" and "row0" in meta and len(idx) >= 2:
            if "blocks" in meta:
                return f"segment {meta['seg']}, partial-sum block row {meta['row0'] // 32 + idx[0]}, column {meta['col0'] + idx[1]}"
            row = meta["row0"] + idx[0]
            col = meta["col0"] + idx[1] * (32 if meta.get("part") == "rowstat" else 1)
            kw = {k: v for k, v in bargs.items() if k not in ("a", "w", "out", "sched")}
            tile = _tile_at(bargs["sched"], kw, meta["seg"], row, col)
            return f"segment {meta['seg']}, tile (row base {tile[0] if tile else '?'}, column base " \
                   f"{tile[1] if tile else '?'}), first bad (row {row}, col {col})"
        return f"element {tuple(int(v) for v in idx)} of the region"

    def _fail(self, msg):
        self.failures.append(msg)

    def _compare(self, name, bargs, snap, writes, tags, line):
        head = f"launch {line['i']} {name} [{line['label']}]"
        for dst, val, meta in writes:
            ent = snap.copy_of(dst)
            if ent is None:
                self._fail(f"{head}: the reference wrote outside the arguments")
                continue
            got = _as(ent[0], dst.dtype, dst.storage_offset(), dst.size(), dst.stride(), dst.device)
            if dst.numel():
                g, r = got.to(val.dtype), val
                k = int(meta.get("k", 1))
                if "stored" in meta:   # statistics of the output values as stored (already the device's, see below)
                    src, pw = meta["stored"]
                    x = src.to(val.dtype).reshape(-1, 32, src.shape[1])
                    r = (x if pw == 1 else x * x).sum(1)
                if "blocks" in meta:   # per-sample sums over the partial-sum blocks
                    nb = meta["blocks"]
                    g = g.reshape(-1, nb, g.shape[-1]).sum(1)
                    r = r.reshape(-1, nb, r.shape[-1]).sum(1)
                    k = k * nb
                err = (g - r).abs()
                if meta.get("exact"):   # e.g. zero padding: any difference fails
                    rat = torch.where(g == r, torch.zeros_like(err), torch.full_like(err, float("inf")))
                else:
                    tol = _tol(r, dst.dtype, k, meta.get("floor", 0.0)).clamp_min(torch.finfo(torch.float32).tiny)
                    rat = torch.where(torch.isfinite(g), err / tol, torch.full_like(err, float("inf")))
                worst = float(rat.max())
                grp = group_of(name, dst.dtype, meta, tags)
                line["ratio"] = max(line["ratio"], worst)
                line.setdefault("groups", {})
                line["groups"][grp] = max(line["groups"].get(grp, 0.0), worst)
                if worst > self.worst.get(grp, (-1.0, -1))[0]:
                    self.worst[grp] = (worst, line["i"])
                if not worst <= self.bounds[grp]:
                    bad = (rat > self.bounds[grp]) | ~torch.isfinite(rat)
                    first = torch.nonzero(bad)[0].tolist()
                    self._fail(f"{head}: {grp}: error ratio {worst:.3g} > bound {self.bounds[grp]:.3g} at "
                               f"{self._where(name, bargs, meta, first)}: got {float(g[tuple(first)]):.6g}, "
                               f"ref {float(r[tuple(first)]):.6g}")
            dst.copy_(got)   # the written region now holds the device's values: the rest must match byte for byte
        for ptr, (orig, copy, (arg, t)) in snap.stores.items():
            a = torch.empty(0, dtype=torch.uint8, device=t.device).set_(orig)
            b = torch.empty(0, dtype=torch.uint8, device=t.device).set_(copy)
            if torch.equal(a, b):
                continue
            byte = int(torch.nonzero(a != b)[0])
            el = byte // t.element_size() - t.storage_offset()
            pos, extra = f"element {el} past the start of `{arg}`", ""
            if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) > 0:
                row, col = divmod(el, t.stride(0))
                pos = f"`{arg}` (row {row}, col {col})"
                if name == "grouped_gemm":
                    segs = bargs["sched"].segs.cpu().numpy()[:bargs["sched"].n_segs]
                    si = [j for j in range(len(segs)) if segs[j][0] <= row < segs[j][1]]
                    extra = f" (segment {si[0] if si else 'none'}"
                    if si:
                        kw = {k: v for k, v in bargs.items() if k not in ("a", "w", "out", "sched")}
                        tile = _tile_at(bargs["sched"], kw, si[0], row, col)
                        if tile is not None:
                            extra += f", tile row base {tile[0]}"
                    extra += ")"
            self._fail(f"{head}: wrote outside its contract: {pos} changed{extra}")
            line["ratio"] = float("inf")

    # ---- reporting ------------------------------------------------------------------------------------------
    def has(self, *tags) -> bool:
        want = set(tags)
        return any(want <= set(k.split()) for k in self.tally)

    def report(self) -> str:
        out = [f"{sum(self.counts.values())} launches, {sum(self.counts.values()) - sum(self.unchecked.values())} "
               f"checked; unchecked: {dict(self.unchecked) or 'none'}"]
        out.append("grouped-GEMM launches by feature set:")
        for k, v in sorted(self.tally.items(), key=lambda kv: (-kv[1], kv[0])):
            out.append(f"  {v:4d}  {k}")
        out.append(f"worst error ratio per group ({TOL_RULES}):")
        for g, (r, i) in sorted(self.worst.items()):
            out.append(f"  {g:40s} {r:8.3f}  (bound {self.bounds[g]:.2f}, launch {i} [{self.lines[i]['label']}])")
        return "\n".join(out)

    def dump(self, case: str):
        """Append this case's summary to $APTP_REPLAY_LOG (JSON lines), if set."""
        path = os.environ.get("APTP_REPLAY_LOG")
        if not path:
            return
        row = {"case": case, "launches": dict(self.counts), "unchecked": dict(self.unchecked),
               "tally": dict(self.tally), "worst": {g: [round(r, 4), i] for g, (r, i) in self.worst.items()},
               "failures": self.failures[:20]}
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "a") as f:
            f.write(json.dumps(row) + "\n")

    def assert_clean(self):
        if self.failures:
            more = f"\n... and {len(self.failures) - 20} more" if len(self.failures) > 20 else ""
            raise ReplayFailure(f"{len(self.failures)} launch mismatches:\n" + "\n".join(self.failures[:20]) + more)


# ------------------------------------------------------------------------------------------------
# forward cases
# ------------------------------------------------------------------------------------------------
def replay_forward(model, arch, B, H, ctx_dim, device, setattr_fn, cdt=torch.float64, fault=None, seed=1):
    """Drive _Engine.run (no CUDA graph) for one forward of `model` with gates `arch`, under a Recorder."""
    from diffusion_pruning_b200.synthetic import split_arch
    from diffusion_pruning_b200.unet import _Engine
    g = torch.Generator().manual_seed(seed)
    sample = torch.randn(B, 4, H, H, generator=g)
    ctx = torch.randn(B, 77, ctx_dim, generator=g)
    t = torch.tensor([981, 661, 341, 21] * ((B + 3) // 4))[:B]
    st = model.get_structure()
    model.set_structure(split_arch(arch.clone().to(device), st))
    eng = _Engine(model, torch.device(device))
    rec = Recorder(cdt=cdt, label=lambda: eng._label, fault=fault).install(setattr_fn)
    with torch.no_grad():
        eng.run(sample.to(device), t.to(device), ctx.to(device))
    return rec, eng
