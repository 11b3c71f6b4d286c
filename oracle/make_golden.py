#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY -- regenerates tests/golden/*.json from the UNMODIFIED reference.

Run in the build container (needs /root/reference and `make -C oracle`):

    python oracle/make_golden.py

Everything written is an input/output vector pair: the INPUT (UAI model text of the
reference's small shipped models, evidence, op operands) and the OUTPUT the compiled
reference (oracle/_ref/ref_harness) produced for it at 17 significant digits.  The
reference's own shipped goldens (grid3x3.uai.PR/.MAR, network.uai.PR/.MAR) are
recorded beside them.  /root/reference does not exist on the GPU box, so tests read
only these fixtures.
"""
import gzip
import hashlib
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from bnpp_b200 import synth  # noqa: E402
import oracle as orc  # noqa: E402

REF = "/root/reference/models"
OUT = os.path.join(ROOT, "tests", "golden")
TMP = "/tmp/bnpp_golden"

H = orc.RefHarness()


def rd(path):
    with open(path) as f:
        return f.read()


def dump(name, obj, compress=False):
    path = os.path.join(OUT, name)
    data = json.dumps(obj, separators=(",", ":"))
    if compress:
        with gzip.open(path + ".gz", "wt", compresslevel=9) as f:
            f.write(data)
    else:
        with open(path, "w") as f:
            f.write(data)
    print("wrote", name, len(data))


def evidset(ev):
    return "evidset %d %s" % (len(ev), " ".join("%d %d" % kv for kv in sorted(ev.items())))


def find(rows, tag):
    return [r for r in rows if r[0] == tag]


def pr_case(path, ev, flag):
    rows = H.run(["model " + path, evidset(ev), "opt " + flag, "pr", "order"])
    out = {"flag": flag, "evidence": {str(k): v for k, v in ev.items()}, "pr": float(find(rows, "PR")[0][1])}
    if flag:
        o = find(rows, "ORDER")[0]
        out["width"] = int(o[1])
        out["order"] = [int(x) for x in o[3:]]
    return out


def mar_case(path, ev, flag):
    rows = H.run(["model " + path, evidset(ev), "opt " + flag, "mar"])
    return {"flag": flag, "evidence": {str(k): v for k, v in ev.items()},
            "mar": [m.tolist() for m in H.marginals(rows)]}


def bp_case(path, ev, cond):
    rows = H.run(["model " + path, evidset(ev), "bp 10000 0.001" + (" cond" if cond else "")])
    return {"cond": cond, "evidence": {str(k): v for k, v in ev.items()},
            "sweeps": int(find(rows, "BP")[0][1]), "mar": [m.tolist() for m in H.marginals(rows)]}


# ---------------------------------------------------------------- models.json
def models():
    out = {}
    bn = REF + "/bayesnets/"
    mn = REF + "/markovnets/"
    asia_ev = orc.parse_evidence(rd(bn + "asia.uai.evid"))
    spec = {
        # name: (path, [evidence sets], flags for PR, do "none" order?, MAR?, BP?)
        "asia": (bn + "asia.uai", [{}, asia_ev], True, True, True),
        "asia_positive": (bn + "asia_positive.uai", [{}, {0: 1, 2: 1}], True, True, True),
        "cancer": (bn + "cancer.uai", [{}, {3: 0}], True, True, True),
        "earthquake": (bn + "earthquake.uai", [{}, {2: 1}], True, True, True),
        "child": (bn + "child.uai", [{}, {3: 1, 11: 0}], True, True, True),
        "alarm": (bn + "alarm.uai", [{}, {3: 0, 17: 1, 30: 0}], True, True, True),
        "insurance": (bn + "insurance.uai", [{}, {2: 1, 20: 0}], False, False, True),
        "win95pts": (bn + "win95pts.uai", [{}, {5: 0, 60: 1}], False, False, False),
        "hailfinder": (bn + "hailfinder.uai", [{}, {7: 1}], False, False, False),
        "hepar2": (bn + "hepar2.uai", [{}, {10: 1, 44: 0}], False, False, False),
        "andes": (bn + "andes.uai", [{}], False, False, False),
        "Water": (bn + "Water.uai", [{}], False, False, False),
        "grid3x3": (mn + "grid3x3.uai", [{}, orc.parse_evidence(rd(mn + "grid3x3-PR.uai.evid")),
                                       orc.parse_evidence(rd(mn + "grid3x3-MAR.uai.evid"))], True, True, True),
        "network": (mn + "network.uai", [{}], False, False, False),
    }
    for name, (path, evs, none_ok, do_mar, do_bp) in spec.items():
        print("model", name)
        m = {"uai": rd(path), "pr": [], "mar": [], "bp": []}
        for ev in evs:
            for flag in (["", "mf", "wmf", "md"] if none_ok else ["mf", "wmf", "md"]):
                m["pr"].append(pr_case(path, ev, flag))
            if do_mar:
                m["mar"].append(mar_case(path, ev, ""))
                if not ev:  # heuristic + evidence segfaults in the reference (SURVEY A.2 i)
                    m["mar"].append(mar_case(path, ev, "mf"))
        if do_bp:
            m["bp"].append(bp_case(path, {}, False))       # what `bn -mar -sp` runs (evidence ignored)
            for ev in evs:
                if ev:
                    m["bp"].append(bp_case(path, ev, True))
        out[name] = m
    # marginals by VE (min-fill) for the two Markov nets with shipped .MAR goldens
    out["network"]["mar"].append(mar_case(mn + "network.uai", {}, "mf"))
    # the reference's own shipped goldens
    out["grid3x3"]["shipped"] = {"PR": rd(mn + "grid3x3.uai.PR"), "MAR": rd(mn + "grid3x3.uai.MAR"),
                                 "PR_evid": rd(mn + "grid3x3-PR.uai.evid"), "MAR_evid": rd(mn + "grid3x3-MAR.uai.evid")}
    out["network"]["shipped"] = {"PR": rd(mn + "network.uai.PR"), "MAR": rd(mn + "network.uai.MAR"),
                                 "evid": rd(mn + "network.uai.evid")}
    # asia prompt fixtures
    queries = [ln.strip() for ln in rd(bn + "asia.markov.query").splitlines() if ln.strip()]
    qout = []
    for flags in ["ve", "ve bb", "ve mf", "ve bb md"]:
        script = ["model " + bn + "asia.uai", "opt " + flags] + ["queryve " + q[len("query "):] for q in queries if q.startswith("query ")]
        facs = H.factors(H.run(script))
        qs = [q for q in queries if q.startswith("query ")]
        assert len(facs) == len(qs)
        for q, (scope, size, z, vals) in zip(qs, facs):
            qout.append({"flags": flags, "query": q, "scope": scope, "partition": z, "values": vals.tolist()})
    out["asia"]["queries"] = qout
    out["asia"]["ind"] = rd(bn + "asia.ind")
    out["asia"]["not_ind"] = rd(bn + "asia.not.ind")
    dump("models.json", out, compress=True)


# ---------------------------------------------------------------- orders.json
def orders():
    out = {}
    bn = REF + "/bayesnets/"
    for fn in sorted(os.listdir(bn)):
        if not fn.endswith(".uai"):
            continue
        name = fn[:-4]
        print("orders", name)
        m = orc.read_uai(bn + fn)
        rec = {"card": [int(c) for c in m.card], "scopes": [f.scope for f in m.factors], "cases": []}
        nv = m.nvars
        rng = random.Random(hash(name) & 0xffff if False else sum(map(ord, name)))
        evs = [{}]
        # one evidence set of ~5% of the variables (only the observed IDS matter for the order)
        ids = sorted(rng.sample(range(nv), max(1, nv // 20)))
        evs.append({i: 0 for i in ids})
        for ev in evs:
            for flag in ["mf", "wmf", "md"]:
                rows = H.run(["model " + bn + fn, evidset(ev), "opt " + flag, "order"])
                o = find(rows, "ORDER")[0]
                rec["cases"].append({"flag": flag, "observed": sorted(ev), "width": int(o[1]),
                                     "order": [int(x) for x in o[3:]]})
        rows = H.run(["model " + bn + fn, "widths"])
        rec["widths"] = [int(x) for x in find(rows, "WIDTHS")[0][1:]]
        out[name] = rec
    dump("orders.json", out, compress=True)


# ---------------------------------------------------------------- ops_1.json, ops_2.json
def rand_scope(rng, nvars, w):
    return rng.sample(range(nvars), w)


def ops():
    rng = random.Random(20261018)
    cases = []
    for ci in range(160):
        nvars = rng.randint(1, 7)
        cards = [rng.choice([2, 2, 2, 3, 4, 5, 7]) for _ in range(nvars)]
        wa = rng.randint(0, min(nvars, 5))
        wb = rng.randint(0, min(nvars, 4))
        sa, sb = rand_scope(rng, nvars, wa), rand_scope(rng, nvars, wb)
        script = ["vars %d %s" % (nvars, " ".join(map(str, cards))),
                  "randfactor a %d %d %s" % (1000 + ci, wa, " ".join(map(str, sa))),
                  "randfactor b %d %d %s" % (5000 + ci, wb, " ".join(map(str, sb))),
                  "dump a", "dump b",
                  "product a b p", "dump p", "divide a b q", "dump q"]
        var = rng.randrange(nvars)             # may or may not be in scope
        script += ["sumout p %d s" % var, "dump s"]
        k = rng.randint(0, nvars)
        ev = {v: rng.randrange(cards[v]) for v in rng.sample(range(nvars), k)}
        script += ["cond p c %d %s" % (len(ev), " ".join("%d %d" % kv for kv in sorted(ev.items()))), "dump c",
                   "normalize p n", "dump n", "max p", "min p", "max q", "min q"]
        rows = H.run(script)
        facs = H.factors(rows)
        sc = [float(r[1]) for r in find(rows, "SCALAR")]
        names = ["a", "b", "p", "q", "s", "c", "n"]
        rec = {"cards": cards, "sum_var": var, "evidence": {str(k_): v for k_, v in ev.items()},
               "max_p": sc[0], "min_p": sc[1], "max_q": sc[2], "min_q": sc[3]}
        for nm, (scope, size, z, vals) in zip(names, facs):
            rec[nm] = {"scope": scope, "partition": z, "values": vals.tolist()}
        cases.append(rec)
    for i in range(2):                     # two halves: each file stays under 1 MB
        dump("ops_%d.json" % (i + 1), cases[i * 80:(i + 1) * 80], compress=True)


# ---------------------------------------------------------------- synthetic.json
def synthetic():
    os.makedirs(TMP, exist_ok=True)
    out = {"ising": [], "bn": [], "batch": []}

    def write(name, text):
        p = os.path.join(TMP, name)
        with open(p, "w") as f:
            f.write(text)
        return p, hashlib.sha256(text.encode()).hexdigest()

    for n, h, J, seed in [(4, 0.5, 0.5, 7), (8, 0.5, 1.0, 3), (40, 0.5, 0.3, 7), (40, 0.5, 0.5, 7), (40, 0.5, 1.0, 7)]:
        print("ising", n, J)
        p, sha = write("ising_%d_%g.uai" % (n, J), synth.ising_uai(n, h, J, seed))
        rows = H.run(["model " + p, "bp 10000 0.001"])
        rec = {"n": n, "h": h, "J": J, "seed": seed, "sha256": sha, "sweeps": int(find(rows, "BP")[0][1]),
               "p0": [float(m[0]) for m in H.marginals(rows)]}
        if n <= 4:
            rows = H.run(["model " + p, "opt mf", "pr", "mar"])
            rec["pr_mf"] = float(find(rows, "PR")[0][1])
            rec["exact_p0"] = [float(m[0]) for m in H.marginals(rows)]
        out["ising"].append(rec)

    for N, W, K, seed, nobs in [(24, 10, 3, 2, 3), (40, 24, 3, 3, 4), (48, 30, 3, 5, 0), (64, 40, 4, 5, 8)]:
        print("bn", N, W, K)
        p, sha = write("bn_%d.uai" % N, synth.random_bn_uai(N, W, K, seed))
        rng = random.Random(seed + 100)
        ev = {i: rng.randrange(2) for i in sorted(rng.sample(range(N), nobs))}
        rec = {"N": N, "W": W, "K": K, "seed": seed, "sha256": sha, "evidence": {str(k): v for k, v in ev.items()}, "cases": []}
        for flag in ["mf", "md", "wmf"]:
            rows = H.run(["model " + p, evidset(ev), "opt " + flag, "order"])
            o = find(rows, "ORDER")[0]
            case = {"flag": flag, "width": int(o[1]), "order": [int(x) for x in o[3:]]}
            if int(o[1]) <= 23:   # width 23: about two minutes per run in the reference
                rows = H.run(["model " + p, evidset(ev), "opt " + flag, "pr"], timeout=3000)
                case["pr"] = float(find(rows, "PR")[0][1])
            rec["cases"].append(case)
        out["bn"].append(rec)

    for N, W, K, seed, nobs, nsets, fixed in [(60, 6, 3, 4, 6, 24, True), (60, 6, 3, 4, 6, 8, False),
                                              (500, 6, 3, 11, 20, 12, True)]:
        print("batch", N, fixed)
        p, sha = write("bn_batch_%d.uai" % N, synth.random_bn_uai(N, W, K, seed))
        evs = synth.evidence_batch(N, nobs, nsets, seed=5, fixed_ids=fixed)
        rec = {"N": N, "W": W, "K": K, "seed": seed, "nobs": nobs, "nsets": nsets, "fixed_ids": fixed,
               "sha256": sha, "pr": [], "orders": []}
        for ev in evs:
            rows = H.run(["model " + p, evidset(ev), "opt mf", "pr", "order"])
            rec["pr"].append(float(find(rows, "PR")[0][1]))
            rec["orders"].append([int(x) for x in find(rows, "ORDER")[0][3:]])
        if fixed:
            assert all(o == rec["orders"][0] for o in rec["orders"])
            rec["orders"] = rec["orders"][:1]
        out["batch"].append(rec)
    dump("synthetic.json", out, compress=True)


# ---------------------------------------------------------------- cli.json
def cli():
    """stdout of the reference's own `bn` / `mn` (oracle/_ref) on the command lines of
    tests/test_gpu_host.py:cli_cases, `Executed in` and the directory of the input files masked"""
    import pathlib
    import subprocess
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_host import cli_cases, mask
    with gzip.open(os.path.join(OUT, "models.json.gz"), "rt") as f:
        golden_models = json.load(f)
    d = pathlib.Path(TMP) / "cli"
    d.mkdir(parents=True, exist_ok=True)
    cases = []
    for exe, args, stdin in cli_cases(d, golden_models):
        p = subprocess.run([os.path.join(HERE, "_ref", exe)] + args, input=stdin, capture_output=True, text=True,
                           timeout=300)
        cases.append({"argv": [exe] + [mask(a, d) for a in args], "stdin": stdin, "returncode": p.returncode,
                      "stdout": mask(p.stdout, d)})
    with open(os.path.join(OUT, "cli.json"), "w") as f:
        json.dump({"source": "stdout of the reference's bn / mn on the `make check` command lines (code/Makefile:47-56), "
                             "written by `python oracle/make_golden.py cli`; `Executed in` and the directory of the input "
                             "files masked", "cases": cases}, f, indent=1)
        f.write("\n")
    print("wrote cli.json", len(cases))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["models", "orders", "ops", "synthetic", "cli"]
    for w in which:
        globals()[w]()
