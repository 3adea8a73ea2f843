"""K5 (csrc/bcd.cu, onmf_update_dict[_ws]) in every launch variant, against the FP64 oracle.

The launcher picks among the one-CTA kernel, the cluster kernel (1-16 CTAs, 1-32 lanes per row, W shares in registers
or not, three signalling forms) and the cooperative grid from (dtype, d, k), the device limits and the ONMF_BCD_*
switches.  onmf_update_dict_plan reports that choice without a GPU, so the CPU part pins which shape takes which variant
and checks the invariants every plan must meet; the GPU part runs each pinned shape on four input families and compares
with oracle.onmf_oracle.update_dict on the same (dtype-rounded) inputs.

Bars: fp64 1e-12 per atom; fp32 per atom max(16 x the error of a numpy fp32 emulation of the sweep, 1e-6), and 1e-5 in
any case.  test_mutants_are_far_above_the_fp32_bar shows that these inputs and bars tell a broken sweep from rounding."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import _bcd_worker as BW
from onmf_ontf_ndl_b200 import _lib
from oracle import onmf_oracle as O

F32, F64 = "float32", "float64"
SMEM_OPTIN = 232448               # B200 opt-in shared memory per block (the library assumes it without a device)

# one row per variant and edge: (dtype, d, k) -> (kind, CTAs, lanes per row, registers).  The GPU tests take their shapes
# from here; a retuned dispatch fails this table instead of silently testing other variants.
PINNED = {
    (F32, 100, 25): ("small", 1, 1, 0),        # cfg1
    (F32, 300, 49): ("small", 1, 1, 0),        # cfg2
    (F32, 441, 25): ("small", 1, 1, 0),        # cfg3
    (F32, 400, 100): ("small", 1, 1, 0),       # cfg4
    (F32, 77, 3): ("small", 1, 1, 0),          # k < 4
    (F32, 5, 1): ("small", 1, 1, 0),
    (F32, 16, 256): ("cluster", 1, 32, 0),     # 4x4 patches, 256 atoms: was the misaligned register form
    (F32, 12, 300): ("cluster", 1, 32, 0),     # (was misaligned)
    (F32, 9, 400): ("cluster", 1, 32, 0),      # (was misaligned)
    (F32, 1, 256): ("cluster", 1, 32, 0),      # (was misaligned) and k > 4 x threads: the prefetch tail of the column of A
    (F32, 13, 301): ("cluster", 1, 32, 0),     # odd k
    (F32, 17, 256): ("cluster", 1, 16, 1),
    (F32, 20, 512): ("cluster", 1, 16, 1),     # registers, k = 32 tpr
    (F32, 17, 257): ("cluster", 1, 16, 0),
    (F32, 40, 256): ("cluster", 1, 8, 1),      # registers, k = 32 tpr
    (F32, 40, 255): ("cluster", 1, 8, 0),
    (F32, 201, 256): ("cluster", 2, 4, 0),     # d % CTAs != 0
    (F32, 321, 128): ("cluster", 4, 4, 1),     # registers, k = 32 tpr, d % CTAs != 0
    (F32, 1024, 256): ("cluster", 8, 4, 0),    # cfg5
    (F32, 900, 128): ("cluster", 8, 4, 1),     # registers, d % CTAs != 0
    (F32, 520, 100): ("cluster", 8, 4, 1),     # registers, k % (4 tpr) != 0
    (F32, 1000, 130): ("cluster", 8, 4, 0),
    (F32, 2048, 128): ("cluster", 8, 2, 0),
    (F32, 2047, 130): ("cluster", 8, 2, 0),
    (F32, 2700, 25): ("cluster", 8, 1, 0),
    (F32, 1025, 3): ("cluster", 8, 1, 0),      # k < 4
    (F32, 2045, 256): ("cluster", 16, 4, 0),
    (F32, 12001, 97): ("grid", 147, 32, 0),
    (F32, 512, 1600): ("grid", 128, 32, 0),    # past the cluster's lane-count edge (had no kernel before)
    (F64, 100, 25): ("small", 1, 1, 0),        # cfg1
    (F64, 300, 49): ("small", 1, 1, 0),        # cfg2
    (F64, 441, 25): ("small", 1, 1, 0),        # cfg3
    (F64, 77, 3): ("small", 1, 1, 0),
    (F64, 5, 1): ("small", 1, 1, 0),
    (F64, 400, 100): ("cluster", 4, 4, 0),     # cfg4
    (F64, 1024, 256): ("cluster", 16, 8, 0),   # cfg5
    (F64, 16, 256): ("cluster", 1, 32, 0),
    (F64, 1, 256): ("cluster", 1, 32, 0),      # prefetch tail
    (F64, 13, 301): ("cluster", 1, 32, 0),
    (F64, 17, 257): ("cluster", 1, 16, 0),
    (F64, 40, 255): ("cluster", 1, 8, 0),
    (F64, 201, 256): ("cluster", 2, 4, 0),
    (F64, 900, 128): ("cluster", 8, 4, 0),
    (F64, 1000, 130): ("cluster", 8, 4, 0),
    (F64, 2700, 25): ("cluster", 8, 1, 0),
    (F64, 1025, 3): ("cluster", 8, 1, 0),
    (F64, 2048, 128): ("cluster", 16, 4, 0),
    (F64, 2047, 130): ("cluster", 16, 4, 0),
    (F64, 8193, 64): ("grid", 147, 32, 0),
    (F64, 512, 1600): ("grid", 128, 32, 0),
}
CFG = [(100, 25), (300, 49), (441, 25), (400, 100), (1024, 256)]
REGW_ROWS = [key for key, v in PINNED.items() if v[3]]


def plan(dt, d, k):
    return _lib.update_dict_plan(getattr(torch, dt), d, k)


def row_id(key):
    return "%s-%dx%d" % key


# ------------------------------------------------------------------------------------------------------------------ CPU
def _grid():
    ds = sorted(set(range(1, 65)) | set(range(65, 4097, 37)) | {2 ** e + o for e in range(6, 13) for o in (-1, 0, 1)})
    ks = sorted(set(range(1, 65)) | set(range(65, 513, 3)) | {128, 255, 256, 257, 384, 511, 512})
    return ds, ks


@pytest.mark.parametrize("dt", [F32, F64])
def test_plan_invariants(dt):
    """every shape up to k = 512 gets a plan, and every plan is launchable and aligned"""
    ds, ks = _grid()
    tdt = getattr(torch, dt)
    bad = []
    for d in ds:
        for k in ks:
            p = plan(dt, d, k)
            c, r, t = p["ctas"], p["rows_per_cta"], p["tpr"]
            ok = p["smem"] <= SMEM_OPTIN and p["threads"] <= (512 if p["regw"] else 1024) and p["threads"] % 32 == 0
            ok &= (c - 1) * r < d <= c * r                                   # no CTA without rows, every row owned
            ok &= (_lib.update_dict_workspace(tdt, d, k) > 0) == (p["kind"] == "grid")
            if p["kind"] == "cluster":
                ok &= c in (1, 2, 4, 8, 16) and t in (1, 2, 4, 8, 16, 32) and r * t <= p["threads"] and p["ks"] >= k
                ok &= p["mbar"] == 2 and p["smem"] <= SMEM_OPTIN - 1024
            if p["kind"] == "small":
                ok &= c == 1 and r == d and p["threads"] >= d and p["ks"] >= k
            if p["regw"]:
                # the register form loads 16-byte vectors from rows of the slab and from the column of A behind it
                ok &= (dt == F32 and p["kind"] == "cluster" and k % 4 == 0 and 4 <= t and k <= 32 * t
                       and p["ks"] % 4 == 0 and (r * p["ks"]) % 4 == 0)
            if not ok:
                bad.append((d, k, p))
    assert not bad, bad[:5]


def test_plan_exists_past_the_cluster_edge():
    """shapes at the edge of one cluster's shared memory whose 512-thread lane count needs a wider pitch than the
    fit test assumed (e.g. 512 x 1600 fp32) take the cooperative grid; before, no kernel took them"""
    for dt in (F32, F64):
        for d in (480, 500, 512, 1000):
            for k in range(1500, 1700, 7):
                assert plan(dt, d, k)["kind"] in ("cluster", "grid")


def test_plan_query_rejects_bad_arguments():
    lib = _lib.load()
    p = _lib.BcdPlan()
    assert lib.onmf_update_dict_plan(7, 10, 5, None) == -1
    assert lib.onmf_update_dict_plan(0, 0, 5, _lib.ctypes.byref(p)) == -1
    assert lib.onmf_update_dict_plan(1, 10, -1, _lib.ctypes.byref(p)) == -1


@pytest.mark.parametrize("key", list(PINNED), ids=row_id)
def test_pinned_variant_table(key):
    p = plan(*key)
    assert (p["kind"], p["ctas"], p["tpr"], p["regw"]) == PINNED[key], p


def test_pinned_table_covers_every_variant():
    vals = set(PINNED.values())
    for dt in (F32, F64):
        assert any(v[0] == "small" for (t, _, _), v in PINNED.items() if t == dt)
        assert any(v[0] == "grid" for (t, _, _), v in PINNED.items() if t == dt)
        for d, k in CFG:
            assert (dt, d, k) in PINNED
    assert {v[1] for v in vals if v[0] == "cluster"} == {1, 2, 4, 8, 16}
    assert {v[2] for v in vals if v[0] == "cluster"} == {1, 2, 4, 8, 16, 32}
    assert {v[2] for v in vals if v[3]} == {4, 8, 16}
    assert all(PINNED[(F32, d, k)][3] == 0 for d, k in ((16, 256), (12, 300), (9, 400), (1, 256)))
    assert any(k > 4 * plan(*key)["threads"] for key, v in PINNED.items() if v[0] == "cluster")
    assert any(key[2] == 32 * v[2] for key, v in PINNED.items() if v[3])
    assert any(key[2] % (4 * v[2]) for key, v in PINNED.items() if v[3])


def _cut_rows(dt, d, k):
    p = plan(dt, d, k)
    return d - (p["ctas"] - 1) * p["rows_per_cta"] if p["kind"] == "cluster" and p["ctas"] > 1 else max(1, d // 8)


MUTANT_SHAPES = [key for key in PINNED if key[0] == F32 and key[1] * key[2] <= 2_000_000 and key[2] <= 512]


@pytest.mark.parametrize("key", MUTANT_SHAPES, ids=row_id)
def test_mutants_are_far_above_the_fp32_bar(key):
    """numpy restatements of the sweep with one kernel bug each land >= 30x above the fp32 bar on the inputs the GPU
    tests use: on the learned-like family alone wherever the shape allows the bug to show (d, k >= 16), and on at least
    one family at every shape (with k = 1 there is no exchange term, no register copy and no next row of B)"""
    dt, d, k = key
    sep = {m: {} for m in BW.MUTANTS}
    for fam in BW.FAMILIES:
        W, A, B = (BW.rounded(x, dt) for x in BW.state(fam, d, k))
        ref = O.update_dict(W, A, B)
        bar = max(16 * BW.atom_err(BW.emulate_fp32(W, A, B), ref), 1e-6)
        assert bar <= 1e-5, (fam, bar)
        for m in BW.MUTANTS:
            sep[m][fam] = BW.atom_err(BW.sweep(W, A, B, m, _cut_rows(dt, d, k)), ref) / bar
    applicable = BW.MUTANTS if k > 1 else ("step_1_over_ajj", "norm_missing_last_cta")
    for m in applicable:
        assert max(sep[m].values()) >= 30, (m, sep[m])
        if d >= 16 and k >= 16:
            assert sep[m]["learned"] >= 30 or m == "norm_missing_last_cta", (m, sep[m])


# ------------------------------------------------------------------------------------------------------------------ GPU
def _dev():
    return torch.device("cuda", 0)


def _bars(dt, W, A, B, ref):
    if dt == F64:
        return 1e-12
    return min(max(16 * BW.atom_err(BW.emulate_fp32(W, A, B), ref), 1e-6), 1e-5)


def _check_against_oracle(dt, d, k, fam, got):
    W, A, B = (BW.rounded(x, dt) for x in BW.state(fam, d, k))
    ref = O.update_dict(W, A, B)
    err, bar = BW.atom_err(got, ref), _bars(dt, W, A, B, ref)
    assert err <= bar, (dt, d, k, fam, err, bar)
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(PINNED), ids=row_id)
def test_variant_matches_oracle(key):
    """each variant on every input family: oracle at the bars, in place == out of place, two calls bit-identical"""
    dt, d, k = key
    tdt = getattr(torch, dt)
    worst = 0.0
    for fam in BW.FAMILIES:
        W, A, B = BW.state(fam, d, k)
        Wd, Ad, Bd = (torch.from_numpy(np.ascontiguousarray(x)).to(_dev(), tdt) for x in (W, A, B))
        out1, out2 = torch.empty_like(Wd), torch.empty_like(Wd)
        _lib.update_dict(Wd, Ad, Bd, out1)
        _lib.update_dict(Wd, Ad, Bd, out2)
        _lib.update_dict(Wd, Ad, Bd, Wd)                                   # in place
        torch.cuda.synchronize()
        assert torch.equal(out1, out2) and torch.equal(out1, Wd), fam
        worst = max(worst, _check_against_oracle(dt, d, k, fam, out1.cpu().numpy().astype(np.float64)))
    p = plan(dt, d, k)
    print("K5 %s d=%d k=%d %s ctas=%d tpr=%d regw=%d: worst per-atom error %.2e" % (dt, d, k, p["kind"], p["ctas"], p["tpr"],
                                                                                    p["regw"], worst))


SWITCH_RUNS = {
    # the small-dictionary shapes as cluster kernels, the register shapes in the shared-memory form
    "small0_regw0": ({"ONMF_BCD_SMALL": "0", "ONMF_BCD_REGW": "0"},
                     [(dt, d, k) for dt in (F32, F64) for d, k in CFG[:4]] + REGW_ROWS),
    "mbar0": ({"ONMF_BCD_MBAR": "0"}, [key for key, v in PINNED.items() if v[0] == "cluster"]),
    "mbar1": ({"ONMF_BCD_MBAR": "1"}, [key for key, v in PINNED.items() if v[0] == "cluster"]),
    "tpr1": ({"ONMF_BCD_TPR": "1"}, [(F32, 1024, 256), (F64, 1024, 256), (F32, 900, 128)]),
    "tpr2": ({"ONMF_BCD_TPR": "2"}, [(F32, 1024, 256), (F64, 1024, 256), (F32, 900, 128)]),
}
SWITCH_FAMILIES = ("learned", "mixed")


@pytest.mark.gpu
def test_switch_forms_in_subprocesses(tmp_path):
    """ONMF_BCD_SMALL / _REGW / _MBAR / _TPR are read once per process: each setting runs in its own process (all at
    once), which writes its outputs and the plans it saw.  Every output matches the oracle; the signalling forms 0 and 1
    are bit-identical to the default form 2 (slots summed in rank order in all three)."""
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_bcd_worker.py")
    procs = {}
    for name, (env, keys) in SWITCH_RUNS.items():
        cases = [list(key) + [fam] for key in keys for fam in SWITCH_FAMILIES]
        (tmp_path / (name + ".json")).write_text(json.dumps(cases))
        e = dict(os.environ)
        for v in ("ONMF_BCD_SMALL", "ONMF_BCD_REGW", "ONMF_BCD_MBAR", "ONMF_BCD_TPR"):
            e.pop(v, None)
        e.update(env)
        procs[name] = subprocess.Popen([sys.executable, worker, str(tmp_path / (name + ".json")), str(tmp_path / (name + ".npz"))],
                                       env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    default_keys = sorted({tuple(key) + (fam,) for _, keys in SWITCH_RUNS.values() for key in keys for fam in SWITCH_FAMILIES
                           if plan(*key)["kind"] == "cluster"})
    default, _ = BW.run_cases(default_keys)
    logs = {name: p.communicate(timeout=600)[0] for name, p in procs.items()}
    for name, p in procs.items():
        assert p.returncode == 0, (name, logs[name][-3000:])
    worst = {}
    for name, (env, keys) in SWITCH_RUNS.items():
        res = np.load(tmp_path / (name + ".npz"))
        plans = json.loads(str(res["plans"]))
        for key in keys:
            for fam in SWITCH_FAMILIES:
                tag = "%s_%d_%d_%s" % (key + (fam,))
                p = plans[tag]
                if name == "small0_regw0":
                    assert p["kind"] == "cluster" and p["regw"] == 0, (tag, p)
                elif name.startswith("mbar"):
                    assert p["mbar"] == int(env["ONMF_BCD_MBAR"]), (tag, p)
                    assert np.array_equal(res[tag], default[tag]), tag               # bit-identical across forms
                else:
                    assert p["kind"] == "cluster" and p["tpr"] <= int(env["ONMF_BCD_TPR"]) and p["regw"] == 0, (tag, p)
                err = _check_against_oracle(key[0], key[1], key[2], fam, res[tag])
                worst[name] = max(worst.get(name, 0.0), err)
    print("K5 switch forms, worst per-atom error:", {n: "%.2e" % v for n, v in worst.items()})


STEP_SHAPES = [(F32, 16, 256), (F64, 16, 256), (F32, 16384, 64), (F64, 8193, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("key", STEP_SHAPES, ids=row_id)
def test_update_inside_the_step(key):
    """the update a training step runs (one-step lag: the new W is update_dict of the state before the step) matches
    the oracle with and without CUDA-graph replay; graph and stream schedule agree bit for bit"""
    from onmf_ontf_ndl_b200 import OnmfEngine
    dt, d, k = key
    tdt = getattr(torch, dt)
    assert plan(dt, d, k)["kind"] == ("grid" if d > 1000 else "cluster")
    rng = np.random.default_rng(d + k)
    X = rng.random((192, d))
    W0 = BW.state("learned", d, k)[0]
    finals = []
    for graph in (True, False):
        eng = OnmfEngine(d, k, alpha=0.5, dtype=tdt, device=_dev(), graph=graph)
        eng.set_state(W0)
        Xt = torch.from_numpy(X).to(_dev(), tdt)
        for t in range(1, 7):
            W, A, B, _ = eng.state()
            torch.cuda.synchronize()
            Wn, An, Bn = (x.cpu().numpy().astype(np.float64) for x in (W, A, B))
            eng.step(Xt, float(t))
            W1 = eng.state()[0].cpu().numpy().astype(np.float64)
            ref = O.update_dict(Wn, An, Bn)
            err, bar = BW.atom_err(W1, ref), _bars(dt, Wn, An, Bn, ref)
            assert err <= bar, (graph, t, err, bar)
        torch.cuda.synchronize()
        finals.append([x.clone() for x in eng.state()[:3]])
        assert (eng._plan.graph_steps() >= 3) == graph
    for a, b in zip(*finals):
        assert torch.equal(a, b)
    print("K5 in the step %s d=%d k=%d (%s): graph replay == stream schedule" % (dt, d, k, plan(dt, d, k)["kind"]))
