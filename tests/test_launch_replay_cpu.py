"""The launch-replay harness (tests/launch_replay.py) checked on CPU: the tiny U-Net runs on the torch emulation of
the kernels (tests/cpu_kernel_sim.py) standing in for the device, wrapped by the recorder. A clean run must pass;
wrong numbers injected into the "device" outputs must each be caught and located."""
import numpy as np
import pytest
import torch

import cpu_kernel_sim
import launch_replay as LR
from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200._lib import EPI_GEGLU, OUT_BF16
from diffusion_pruning_b200.synthetic import synthetic_codes
from diffusion_pruning_b200.unet import UNet2DConditionModelGated
from oracle.unet_oracle import GatedUNetOracle, UNetConfig, seeded_init

TINY = dict(block_out_channels=(64, 128, 256, 256), attention_head_dim=(1, 2, 4, 4), cross_attention_dim=128)


def _model():
    oracle = GatedUNetOracle(UNetConfig.tiny()).eval()
    seeded_init(oracle, 0, 0.1)
    model = UNet2DConditionModelGated(**TINY).eval()
    model.load_state_dict(oracle.state_dict())
    return model


def _run(monkeypatch, fault=None, H=16):
    cpu_kernel_sim.install(monkeypatch)
    model = _model()
    codes = synthetic_codes(model.get_structure(), 8)
    return LR.replay_forward(model, codes[[0, 3, 3, 7, 5]], 5, H, 128, "cpu", monkeypatch.setattr, fault=fault)[0]


def test_replay_clean_on_emulation(monkeypatch):
    rec = _run(monkeypatch)
    print(rec.report())
    rec.assert_clean()
    assert rec.counts["grouped_gemm"] > 50 and rec.counts["attention"] > 0 and rec.counts["groupnorm_apply"] > 0
    assert rec.has("multiseg", "placeholder") and rec.has("col_off") and rec.has("geglu", "lnfold")
    assert rec.has("conv_s2") and rec.has("colstat") and rec.has("rowstat")


class _Faults:
    """Injects one fault per kind into the first grouped-GEMM launch (bf16 output) that allows it, one launch each.
    Records (launch index, label, text the report must contain)."""

    KINDS = ("ulp", "past_n_store", "neighbour_block", "stale_tile", "placeholder_partner")

    def __init__(self):
        self.done = {}

    def __call__(self, rec, name, args, snap):
        if name != "grouped_gemm" or args["out_mode"] != OUT_BF16 or args["flags"] & EPI_GEGLU:
            return
        sched, out, ld = args["sched"], args["out"], args["out_ld"]
        segs = sched.segs.cpu().numpy()[:sched.n_segs]
        tiles = sched.tiles.cpu().numpy()
        tiles = tiles[(tiles[:, 3] & K.TILE_SKIP) == 0]
        act = [int(s) for s in np.unique(tiles[:, 0])]
        rows = int(segs[:, 1].max())
        O = torch.as_strided(out, (rows, ld), (ld, 1), out.storage_offset())
        i, label = len(rec.lines), rec.label()

        def written(r, c):  # is (r, c) inside the contract of an active segment of this launch?
            return any(segs[s][0] <= r < segs[s][1] and segs[s][8] <= c < segs[s][8] + max(segs[s][2], segs[s][3])
                       for s in act)

        for kind in self.KINDS:
            if kind in self.done:
                continue
            for s in act:
                rb, re, nv, ns, oco = int(segs[s][0]), int(segs[s][1]), int(segs[s][2]), int(segs[s][3]), int(segs[s][8])
                nst = max(nv, ns)
                if kind == "ulp":
                    j = int(O[rb, oco:oco + nv].float().abs().argmax())
                    O.view(torch.int16)[rb, oco + j] += 4
                    want = f"first bad (row {rb}, col {oco + j})"
                elif kind == "past_n_store":
                    c = oco + nst
                    if c >= ld or written(rb, c):
                        continue
                    O[rb, c] += 1.0
                    want = f"(row {rb}, col {c}) changed"
                elif kind == "neighbour_block":
                    c = oco - 1
                    if oco == 0 or written(rb, c):
                        continue
                    O[rb, c] += 1.0
                    want = f"(row {rb}, col {c}) changed"
                elif kind == "stale_tile":
                    mine = tiles[tiles[:, 0] == s]
                    if args["mode"] != 0 or len(np.unique(mine[:, 1])) < 2:
                        continue
                    m, n0 = int(mine[-2, 1]), int(mine[-2, 2])
                    width = LR._tile_width(sched, mine, False)[0]
                    r1, c0, c1 = min(m + 128, re), oco + n0, oco + min(n0 + width, nst)
                    pre = LR._as(snap.original(out)[1], out.dtype, out.storage_offset(), (rows, ld), (ld, 1),
                                 out.device)
                    if torch.equal(pre[m:r1, c0:c1], O[m:r1, c0:c1]):
                        continue
                    O[m:r1, c0:c1] = pre[m:r1, c0:c1]
                    want = f"tile (row base {m}, column base {c0})"
                else:  # the row of the placeholder's partner tile rewritten with another row's values
                    mine = tiles[tiles[:, 0] == s].reshape(-1, 2, 4)
                    ph = mine[(mine[:, 1, 3] & K.TILE_PLACEHOLDER) != 0]
                    if len(ph) == 0 or args["mode"] != 0:
                        continue
                    m = int(ph[0, 0, 1])
                    src = m + 1 if m + 1 < re else m - 1
                    if src < rb or torch.equal(O[m, oco:oco + nv], O[src, oco:oco + nv]):
                        continue
                    O[m, oco:oco + nv] = O[src, oco:oco + nv]
                    want = f"tile (row base {m}, column base {oco})"
                self.done[kind] = (i, label, want)
                return  # one fault per launch


def test_replay_catches_injected_faults(monkeypatch):
    faults = _Faults()
    rec = _run(monkeypatch, fault=faults, H=8)
    assert set(faults.done) == set(_Faults.KINDS), f"no launch allowed faults {set(_Faults.KINDS) - set(faults.done)}"
    for kind, (i, label, want) in faults.done.items():
        hits = [f for f in rec.failures if f.startswith(f"launch {i} grouped_gemm [{label}]")]
        assert hits, f"{kind}: launch {i} [{label}] not reported; failures: {rec.failures}"
        assert any(want in f for f in hits), f"{kind}: expected '{want}' in {hits}"
    assert {int(f.split()[1]) for f in rec.failures} == {i for i, _, _ in faults.done.values()}, rec.failures
    with pytest.raises(LR.ReplayFailure):
        rec.assert_clean()
