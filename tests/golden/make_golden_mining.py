"""Generates tests/golden/mining.json by executing the REFERENCE's own hard-negative selection:

    python tests/golden/make_golden_mining.py <path to the OpenMatch checkout>

scripts/msmarco/build_hn.py is a script (argparse runs at import), so the generator lifts only the source of its
``load_ranking`` function out of the file with ``ast`` and executes it unmodified against a synthetic TREC run with
``random.seed(7)``.  The run, the qrels and the reference's output are committed as the fixture.
"""
import ast
import json
import os
import random
import sys
import tempfile

REF = os.path.join(sys.argv[1], "scripts", "msmarco", "build_hn.py") if len(sys.argv) == 2 else None
if REF is None or not os.path.exists(REF):
    sys.exit("usage: make_golden_mining.py <path to the OpenMatch checkout>")
src = open(REF).read()
fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "load_ranking")
ns = {"random": random}
exec(compile(ast.Module(body=[fn], type_ignores=[]), REF, "exec"), ns)
load_ranking = ns["load_ranking"]

rng = random.Random(123)
docs = ["D%d" % i for i in range(400)]
qrels, lines = {}, []
for qi in range(12):
    qid = "Q%d" % qi
    ranked = rng.sample(docs, rng.choice([5, 40, 120, 260]))
    qrels[qid] = rng.sample(ranked, rng.choice([1, 2, 3])) + (["D-not-retrieved"] if qi % 4 == 0 else [])
    for r, d in enumerate(ranked):
        lines.append("%s Q0 %s %d %.4f OpenMatch" % (qid, d, r + 1, 100.0 - r))
with tempfile.NamedTemporaryFile("w", suffix=".trec", delete=False) as f:
    f.write("\n".join(lines) + "\n")
    path = f.name
cases = []
for n_sample, depth in ((30, 200), (7, 20), (3, 1000)):
    random.seed(7)
    out = [[q, list(pos), list(neg)] for q, pos, neg in load_ranking(path, qrels, n_sample, depth)]
    cases.append({"n_sample": n_sample, "depth": depth, "seed": 7, "out": out})
os.unlink(path)
here = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(here, "mining.json"), "w") as f:
    json.dump({"trec": lines, "qrels": qrels, "cases": cases}, f)
print("wrote mining.json:", len(lines), "run lines,", len(cases), "cases")
