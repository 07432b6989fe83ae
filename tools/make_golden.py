#!/usr/bin/env python
"""Generate tests/golden/* from the UNMODIFIED reference (run in the build container only).

  inputs_example{,2}.json/.npz : the two shipped data sets, parsed (configs 1 and 2 of BASELINE.json)
  eikonal_ref_{1,2}.npz        : time_2d fields of the compiled reference (oracle/_ref) for seeded models
  forward_ref.npz              : cal_fit_newx class sums / origin times of the compiled reference
  chain_ref_example2.out       : a short fixed-seed chain of the reference mcmc_eq binary
  replay_example2.npz          : the proposal stream of that same chain (every proposed model, the uniform deviate of
                                 its accept test, the reference's class sums and decision), recorded from the unmodified
                                 reference by symbol interposition (oracle/replay_log.c)

Usage: python tools/make_golden.py   (needs /root/reference and oracle/_ref built: make -C oracle)
"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import util, inputs, refapi  # noqa: E402
import mcmc_eq_b200 as mq  # noqa: E402  (only its file readers are used here, no GPU)

REF = "/root/reference"
G = util.GOLDEN


def cfg_to_dict(c):
    d = {}
    for name, _t in c._fields_:
        v = getattr(c, name)
        if name == "grid":
            for gname, _ in v._fields_:
                d[gname] = getattr(v, gname)
        elif isinstance(v, bytes):
            d[name] = v.decode()
        else:
            d[name] = v
    # keep the short decimal text of float fields (2.0 not 2.000000047)
    return {k: (float(np.format_float_positional(np.float32(v), unique=True)) if isinstance(v, float) else v) for k, v in d.items()}


def parse_t64(path):
    t = []
    for line in open(path):
        if "#" in line or not line.strip():
            continue
        t.append(float(line.split()[6]))
    return np.array(t)


def inputs_of(name, cfg_path, picks_path):
    c = mq.read_config(cfg_path)
    pk = mq.Picks.read(picks_path)
    # t as printed in the file (double), in file order -> our order (P first then S per event)
    t_file = parse_t64(picks_path)
    # recover the permutation: within each event P picks (file order) then S picks (file order)
    phases = [line.split()[2] for line in open(picks_path) if "#" not in line and line.strip()]
    order = []
    k = 0
    for e in range(pk.n_events):
        n = pk.ev_off[e + 1] - pk.ev_off[e]
        idx = list(range(k, k + n))
        order += [i for i in idx if "P" in phases[i]] + [i for i in idx if "P" not in phases[i]]
        k += n
    t64 = t_file[order]
    assert np.array_equal(t64.astype(np.float32), pk.t)
    with open(os.path.join(G, f"inputs_{name}.json"), "w") as f:
        json.dump(cfg_to_dict(c), f, indent=1)
    np.savez_compressed(os.path.join(G, f"inputs_{name}.npz"), ev_off=pk.ev_off, n_p=pk.n_p, st_id=pk.st_id.astype(np.int16),
                        x=pk.x, y=pk.y, z=pk.z, t64=t64, cls=pk.cls.astype(np.int8), reftime=pk.reftime, fix=pk.fix)


def eikonal_fields():
    rng = np.random.default_rng(20241018)
    out = {}
    cases = []
    for gname, g in (("ex2", util.EXAMPLE2_GRID), ("ex", util.EXAMPLE_GRID)):
        nx, nz = util.nxmod_of(g), g["nz"]
        for kind in ("posterior", "contrast", "lvz"):
            z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(2, 18)), g["z0"], g["z0"] + (nz - 1) * g["h"], kind)
            s = util.rasterise_np(z, vp, vpvs, g["h"], g["z0"], nz, 1)
            for iz in (0, 9, 10, 11, nz // 2, nz - 2, nz - 1)[:: (1 if gname == "ex2" else 3)]:
                t, rc = util.ref_time_2d(s, nx, iz)
                assert rc == 0
                cases.append((gname, kind, iz))
                out[f"s_{len(cases) - 1}"] = s
                out[f"t_{len(cases) - 1}"] = t
    # tiny grids: every source depth
    for nx, nz, nl in ((12, 8, 2), (30, 25, 4), (9, 40, 6)):
        z, vp, vpvs = util.voronoi_model(rng, nl, 0.0, (nz - 1) * 1.0, "contrast")
        s = util.rasterise_np(z, vp, vpvs, 1.0, 0.0, nz, 1)
        for iz in range(nz):
            t, rc = util.ref_time_2d(s, nx, iz)
            cases.append((f"tiny{nx}x{nz}", "contrast", iz))
            out[f"s_{len(cases) - 1}"] = s
            out[f"t_{len(cases) - 1}"] = t
    out["meta"] = np.array([f"{a}|{b}|{c}" for a, b, c in cases])
    # two files of under 1 MB each (tests/util.golden_eikonal): the Example2-grid fields with meta, then the rest
    first = {k: v for k, v in out.items() if k == "meta" or cases[int(k.split("_")[1])][0] == "ex2"}
    np.savez_compressed(os.path.join(G, "eikonal_ref_1.npz"), **first)
    np.savez_compressed(os.path.join(G, "eikonal_ref_2.npz"), **{k: v for k, v in out.items() if k not in first})
    print("eikonal_ref:", len(cases), "fields")


def forward_ref():
    """cal_fit_newx of the compiled reference on seeded chain states of both examples."""
    from tests import fwd_helpers as fh
    ref = util.reflib()
    out = {}
    for name, sub, pickfile, nstates in (("example2", "Example2", "picks.mcmc", 3), ("example", "Example", "picks_synth", 2)):
        cfgp, pkp = os.path.join(REF, sub, "config_eqx.dat"), os.path.join(REF, sub, pickfile)
        c = mq.read_config(cfgp)
        pk = mq.Picks.read(pkp)
        g = dict(h=c.grid.h, nx=c.grid.nx, ny=c.grid.ny, nz=c.grid.nz, x0=c.grid.x0, y0=c.grid.y0, z0=c.grid.z0)
        rf = refapi.RefForward(ref, g, pkp)
        assert rf.ne == pk.n_events and rf.nos == pk.n_stations
        rng = np.random.default_rng(7 if name == "example" else 8)
        states = fh.random_states(rng, c, pk, nstates, "posterior")
        for i, s in enumerate(states):
            mf, org = rf.forward(s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"], 3, 1)
            for k, v in s.items():
                out[f"{name}_{i}_{k}"] = v
            out[f"{name}_{i}_mf"] = mf
            out[f"{name}_{i}_origin"] = org
            if i == 0:   # a few table rows of the reference: receiver rows 1,2 of the P table, every source depth
                tp = rf.table(1)
                out[f"{name}_{i}_tabP_rows12"] = tp[1:3]
        out[f"{name}_n"] = np.array(nstates)
    np.savez_compressed(os.path.join(G, "forward_ref.npz"), **out)
    print("forward_ref done")


def chain_ref():
    """Short fixed-seed chain of the reference binary on Example2 (byte-reproducible, SURVEY section 4)."""
    exe = os.path.join(util.REF_DIR, "mcmc_eq")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
        outp = os.path.join(d, "rjx-000.out")
        subprocess.run([exe, cfgp, outp, pkp], check=True, cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        txt = open(outp).read()
    open(os.path.join(G, "chain_ref_example2.out"), "w").write(txt)
    print("chain_ref:", txt.count("\n"), "lines")


def read_replay_log(path):
    """oracle/replay_log.c's binary log -> dict of padded arrays."""
    b = open(path, "rb").read()
    magic, noq, nos = np.frombuffer(b, np.int32, 3, 0)
    assert magic == 0x4d435251
    off = 12
    recs = []
    while off < len(b):
        calct, dim, acc = np.frombuffer(b, np.int32, 3, off); off += 12
        f = lambda n: np.frombuffer(b, np.float32, n, off).copy()
        r = dict(calct=calct, dim=dim, accepted=acc)
        for name, n in (("u", 1), ("mf", 8), ("noise", 8), ("z", dim), ("vp", dim), ("vpvs", dim), ("eq", 3 * noq), ("pres", nos),
                        ("sres", nos), ("origin", noq)):
            r[name] = f(n); off += 4 * n
        recs.append(r)
    n, md = len(recs), max(r["dim"] for r in recs)
    out = dict(calct=np.array([r["calct"] for r in recs], np.int32), dim=np.array([r["dim"] for r in recs], np.int32),
               accepted=np.array([r["accepted"] for r in recs], np.int32), u=np.array([r["u"][0] for r in recs], np.float32))
    for name in ("mf", "noise", "eq", "pres", "sres", "origin"):
        out[name] = np.stack([r[name] for r in recs])
    out["eq"] = out["eq"].reshape(n, noq, 3)
    for name in ("z", "vp", "vpvs"):
        a = np.zeros((n, md), np.float32)
        for i, r in enumerate(recs):
            a[i, :r["dim"]] = r[name]
        out[name] = a
    return out


def replay_ref():
    """Proposal stream of the chain_ref chain (same config and seed), from the unmodified reference."""
    exe = os.path.join(util.REF_DIR, "replay_log")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
        outp, logp = os.path.join(d, "rjx-000.out"), os.path.join(d, "log.bin")
        subprocess.run([exe, logp, cfgp, outp, pkp], check=True, cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        # the interposed run must be the reference's own chain, byte for byte
        assert open(outp).read() == open(os.path.join(G, "chain_ref_example2.out")).read()
        log = read_replay_log(logp)
    np.savez_compressed(os.path.join(G, "replay_example2.npz"), **log)
    print("replay_ref:", len(log["u"]), "records,", int(log["accepted"][1:].sum()), "accepted")


def last_block(text):
    """The last 'mod' record of a chain file with its EQ and RES lines: the input format of fw_mod (src/fw_mod.c:412-467)."""
    lines = text.split("\n")
    start = max(i for i, ln in enumerate(lines) if ln.startswith("mod"))
    out = [lines[start]]
    for ln in lines[start + 1:]:
        if not ln.startswith(("EQ", "RES")):
            break
        out.append(ln)
    return "\n".join(out) + "\n"


def fw_mod_ref():
    """Per-pick predictions of the reference's own forward program for the last record of the golden chain."""
    exe = os.path.join(util.REF_DIR, "fw_mod")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
        blk = os.path.join(d, "block")
        open(blk, "w").write(last_block(open(os.path.join(G, "chain_ref_example2.out")).read()))
        r = subprocess.run([exe, cfgp, blk, pkp], check=True, cwd=d, capture_output=True, text=True)
    open(os.path.join(G, "fw_mod_example2.txt"), "w").write(r.stdout + "STDERR " + r.stderr.strip().split("\n")[-1] + "\n")
    print("fw_mod_ref:", r.stdout.count("\n"), "lines;", r.stderr.strip().split("\n")[-1])


def parse_chain(text, n_events):
    """Trajectory of one chain file: per 'mod' record rms, dimension, sigmas, mean hypocentre depth, rms of the station
    corrections; and the a/r counters."""
    import re
    recs, cur = [], None
    for ln in text.split("\n"):
        t = ln.split()
        if not t:
            continue
        if t[0] == "mod":
            cur = dict(number=int(t[2]), dim=int(t[3]), rms=float(t[4]), noise=[float(x) for x in t[5:13]], z=[], res=[],
                       vp=[float(x) for x in t[14::3][:int(t[3])]])
            recs.append(cur)
        elif t[0] == "EQ" and cur is not None and t[1] not in ("ST", "BF"):
            cur["z"].append(float(t[7]))
        elif t[0] == "RES" and cur is not None and t[1] not in ("ST", "BF"):
            cur["res"].append((float(t[5]), float(t[6])))
        elif t[0] in ("bat", "sta"):
            cur = None
    cnt = {m.group(1).strip(): (int(m.group(2)), int(m.group(3))) for m in re.finditer(r"cnt (\S+)\s+a/r\s+(\d+)\s+(\d+)", text)}
    tested = int(re.search(r"cnt RMS tested\s+(\d+)", text).group(1))
    return dict(number=np.array([r["number"] for r in recs]), dim=np.array([r["dim"] for r in recs]),
                rms=np.array([r["rms"] for r in recs]), noise=np.array([r["noise"] for r in recs]),
                zmean=np.array([np.mean(r["z"]) for r in recs]), res_rms=np.array([np.sqrt(np.mean(np.square(r["res"]))) for r in recs]),
                vp_mean=np.array([np.mean(r["vp"]) for r in recs]),
                acc=np.array([cnt[k][0] for k in ("noise", "P-vel", "Vp/Vs", "quake", "resid", "move", "birth", "death")]),
                rej=np.array([cnt[k][1] for k in ("noise", "P-vel", "Vp/Vs", "quake", "resid", "move", "birth", "death")]), tested=tested)


def write_res_dat(path, zn, vpn, rn, eq, pres, sres):
    """An analyse_eq-style result file the way Example/make_synthetics builds it for fw (src/fw.c:405-455)."""
    with open(path, "w") as f:
        for z, v, r in zip(zn, vpn, rn):
            f.write("STAN %g %g 0 %g 0 %g 0 %g 0 %g %g 0.01\n" % (z, v, r, v, r, v, r))
        for tag in ("EQ", "EZ"):
            for i, q in enumerate(eq):
                f.write("%s %d %g %g %g 0 0 0 0 0 0 0\n" % (tag, i, q[0], q[1], q[2]))
        for i in range(len(pres)):
            f.write("RES %d %g %g 0 0\n" % (i, pres[i], sres[i]))
        f.write("NOISE " + " ".join(["0.1"] * 16) + "\n")


def parse_forward_stdout(text):
    ev, pk = [], []
    for ln in text.strip().split("\n"):
        t = ln.split()
        if t[0] == "EVENT":
            ev.append([float(x) for x in t[2:7]])
        else:
            pk.append([float(x) for x in t[:6]] + [1.0 if t[6] == "S" else 0.0])
    return np.array(ev), np.array(pk)


def fw_ref():
    """Predictions of the reference's fw for a gridded model (61 depth nodes) on the Example2 picks."""
    exe = os.path.join(util.REF_DIR, "fw")
    rng = np.random.default_rng(77)
    cfgd, arr = inputs.load("example2")
    nz, h, z0 = cfgd["nz"], cfgd["h"], cfgd["z0"]
    zn = z0 + h * np.arange(nz)
    vpn = np.round(3.5 + 0.25 * np.maximum(zn, 0) + np.where(zn > 8, 0.6, 0.0) + np.where(zn > 17, 0.5, 0.0), 3)
    rn = np.round(1.9 - 0.01 * np.maximum(zn, 0), 3)
    ne, ns = len(arr["n_p"]), int(arr["st_id"].max()) + 1
    eq = np.round(np.stack([rng.uniform(-8, 8, ne), rng.uniform(-8, 8, ne), rng.uniform(1, 14, ne)], 1), 3)
    pres, sres = np.round(rng.normal(0, 0.1, ns), 3), np.round(rng.normal(0, 0.15, ns), 3)
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d)
        res = os.path.join(d, "res.dat")
        write_res_dat(res, zn, vpn, rn, eq, pres, sres)
        r = subprocess.run([exe, cfgp, res, pkp], check=True, cwd=d, capture_output=True, text=True)
    ev, pk = parse_forward_stdout(r.stdout)
    np.savez_compressed(os.path.join(G, "fw_example2.npz"), zn=zn, vpn=vpn, rn=rn, eq=eq, pres=pres, sres=sres, events=ev, picks=pk)
    print("fw_ref:", ev.shape, pk.shape, r.stderr.strip().split("\n")[-1])


ENSEMBLE = dict(j_max_start=1500, j_max_main=2500, deci=100)


def ensemble_ref(n_chains=32):
    """Ensemble statistics of independent reference chains (Example2, 4000 accepted models each, seeds 100..): the
    posterior-level fixture.  Free-running chains of another RNG cannot match these sample by sample, but their ensemble must
    be statistically indistinguishable (tests/test_ensemble_gpu.py)."""
    exe = os.path.join(util.REF_DIR, "mcmc_eq")
    out = []
    with tempfile.TemporaryDirectory() as d:
        procs = []
        for k in range(n_chains):
            cfgp, pkp = inputs.materialise("example2", os.path.join(d, f"c{k}"), true_random=100 + k, **ENSEMBLE)
            procs.append((k, subprocess.Popen([exe, cfgp, os.path.join(d, f"rjx-{k:03d}.out"), pkp], cwd=os.path.join(d, f"c{k}"),
                                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)))
            if len(procs) == (os.cpu_count() or 4):
                for _k, p in procs:
                    p.wait()
                procs = []
        for _k, p in procs:
            p.wait()
        for k in range(n_chains):
            out.append(parse_chain(open(os.path.join(d, f"rjx-{k:03d}.out")).read(), 225))
    keys = out[0].keys()
    np.savez_compressed(os.path.join(G, "ensemble_ref_example2.npz"), **{k: np.stack([np.asarray(o[k]) for o in out]) for k in keys})
    print("ensemble_ref:", n_chains, "chains; final rms", np.mean([o["rms"][-1] for o in out]), "+-", np.std([o["rms"][-1] for o in out]))


TRIA_CHAIN = dict(j_max_start=60, j_max_main=140, deci=20, true_random=78, tria=1)


def tria_ref():
    """The linear-gradient parameterisation (config line 29 = 1) of the compiled reference: cal_fit_newx on seeded states
    (forward_ref_tria.npz) and a short fixed-seed chain with its proposal stream (chain_ref_example2_tria.out,
    replay_example2_tria.npz)."""
    from tests import fwd_helpers as fh
    ref = util.reflib()
    cfgp, pkp = os.path.join(REF, "Example2", "config_eqx.dat"), os.path.join(REF, "Example2", "picks.mcmc")
    c = mq.read_config(cfgp)
    pk = mq.Picks.read(pkp)
    g = dict(h=c.grid.h, nx=c.grid.nx, ny=c.grid.ny, nz=c.grid.nz, x0=c.grid.x0, y0=c.grid.y0, z0=c.grid.z0)
    rf = refapi.RefForward(ref, g, pkp)
    rng = np.random.default_rng(29)
    states = fh.tria_states(rng, c, pk, 3)
    # one state with two nuclei at the same depth and one with only the two end nuclei
    states[1]["z"][3] = states[1]["z"][2]
    states[2] = {k: (v[:2].copy() if k in ("z", "vp", "vpvs") else v) for k, v in states[2].items()}
    out = {"n": np.array(len(states))}
    for i, s in enumerate(states):
        mf, org = rf.forward(s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"], 3, 1, tria=1)
        for k, v in s.items():
            out[f"{i}_{k}"] = v
        out[f"{i}_mf"] = mf
        out[f"{i}_origin"] = org
        if i == 0:
            out["0_tabP_rows12"] = rf.table(1)[1:3]
            out["0_tabS_rows12"] = rf.table(2)[1:3]
    C.c_int.in_dll(ref, "TRIA").value = 0
    np.savez_compressed(os.path.join(G, "forward_ref_tria.npz"), **out)
    exe, rexe = os.path.join(util.REF_DIR, "mcmc_eq"), os.path.join(util.REF_DIR, "replay_log")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, **TRIA_CHAIN)
        outp, logp = os.path.join(d, "rjx-000.out"), os.path.join(d, "log.bin")
        subprocess.run([exe, cfgp, outp, pkp], check=True, cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        txt = open(outp).read()
        subprocess.run([rexe, logp, cfgp, outp, pkp], check=True, cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert open(outp).read() == txt
        log = read_replay_log(logp)
    open(os.path.join(G, "chain_ref_example2_tria.out"), "w").write(txt)
    np.savez_compressed(os.path.join(G, "replay_example2_tria.npz"), **log)
    print("tria_ref:", len(states), "states;", len(log["u"]), "records,", int(log["accepted"][1:].sum()), "accepted")


if __name__ == "__main__":
    os.makedirs(G, exist_ok=True)
    if len(sys.argv) > 1:        # only the named fixtures, e.g. `python tools/make_golden.py tria_ref`
        for name in sys.argv[1:]:
            globals()[name]()
        sys.exit(0)
    inputs_of("example", os.path.join(REF, "Example/config_eqx.dat"), os.path.join(REF, "Example/picks_synth"))
    inputs_of("example2", os.path.join(REF, "Example2/config_eqx.dat"), os.path.join(REF, "Example2/picks.mcmc"))
    eikonal_fields()
    forward_ref()
    chain_ref()
    replay_ref()
    fw_mod_ref()
    fw_ref()
    ensemble_ref()
    tria_ref()
    print(subprocess.run(["du", "-sh", G], capture_output=True, text=True).stdout)
