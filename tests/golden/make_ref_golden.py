"""Records what the reference's registration code returns for every call tests/test_ref.py makes into
tests/golden/ref_registration.json, which oracle/ref_py.Recorded answers those calls from where oracle/_ref is not built.

    python tests/golden/make_ref_golden.py                 # from oracle/_ref (make -C oracle ref REF_SRC=<DetectAndLocalize/include>)
    python tests/golden/make_ref_golden.py --from-oracle   # from the oracle

It runs the tests of tests/test_ref.py against a recorder and keeps only the fields they read: the transform and the
convergence fields, fitness and align strength exactly, and ref_py.digest() of each array (correspondence lists, the aligned
cloud), which keeps every comparison bit-exact in a few kilobytes.

The committed file was made with --from-oracle at a commit whose oracle, inputs and tests are those under which all eight
tests of tests/test_ref.py had passed against oracle/_ref bit for bit (VERDICT.md, round 2): on every recorded field the two
sources agree there. Once the oracle's registration code changes, re-record from oracle/_ref only.
"""
import inspect
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ope_pkg  # noqa: E402
ope_pkg.load()
from ope_b200 import synth  # noqa: E402
import orc_py  # noqa: E402
import ref_py  # noqa: E402
import test_ref  # noqa: E402


class OracleSource:
    """ref_py's icp() / correspondences() computed by the oracle"""
    T = ref_py.T

    def icp(self, src, tgt, prm, guess=None, src_normals=None, tgt_normals=None, fixed=None, variant="mod"):
        res, corr = orc_py.icp(src, tgt, prm, guess=guess, src_normals=src_normals, tgt_normals=tgt_normals, want_corr=True,
                               fixed=fixed)[:2]
        M = ref_py.T.mat4(res.T)
        return {"res": res, "corr": corr, "aligned": orc_py.transform(src, M), "fitness": orc_py.fitness(src, tgt, M),
                "align_strength": res.n_correspondences / (len(src) + len(tgt))}

    def correspondences(self, src, tgt, max_distance, reciprocal=False, fixed=None, variant="mod"):
        prm = orc_py.icp_params(max_correspondence_distance=max_distance, use_reciprocal=int(bool(reciprocal)))
        return orc_py.correspondences_fixed(src, tgt, prm, fixed)


class Seen(dict):
    """a result that notes which of its fields were read"""

    def __init__(self, d):
        super().__init__(d)
        self.read = set()

    def __getitem__(self, k):
        self.read.add(k)
        return super().__getitem__(k)


class Recorder:
    def __init__(self, source):
        self.source, self.T, self.case, self.results = source, source.T, None, []

    def icp(self, *a, **kw):
        r = Seen(self.source.icp(*a, **kw))
        self.results.append((ref_py.icp_key(*a, **kw), self.case, r))
        return r

    def correspondences(self, *a, **kw):
        r = Seen({"corr": self.source.correspondences(*a, **kw)})
        r.read.add("corr")
        self.results.append((ref_py.correspondences_key(*a, **kw), self.case, r))
        return dict.__getitem__(r, "corr")

    def calls(self):
        out = {}
        for key, case, r in self.results:
            e = out.setdefault(key, {"case": case})
            for k in sorted(r.read):
                v = dict.__getitem__(r, k)
                if k == "res":
                    e[k] = {"T": [float(x) for x in v.T], "converged": v.converged, "state": v.state, "iterations": v.iterations,
                            "n_correspondences": v.n_correspondences}
                elif k == "corr":
                    e[k] = [ref_py.digest(a) for a in v]
                elif k == "aligned":
                    e[k] = ref_py.digest(v)
                else:
                    e[k] = float(v)
        return out


def main():
    from_oracle = "--from-oracle" in sys.argv[1:]
    if not from_oracle and not ref_py.available():
        sys.exit("oracle/_ref is not built (make -C oracle ref REF_SRC=...); --from-oracle records from the oracle")
    rec = Recorder(OracleSource() if from_oracle else ref_py)
    fixtures = {"ref": rec, "orc": orc_py, "synth": synth, "drill": synth.bundled_model()}
    for name, fn in inspect.getmembers(test_ref, inspect.isfunction):
        if not name.startswith("test_"):
            continue
        params = [{}]
        for m in getattr(fn, "pytestmark", []):
            if m.name == "parametrize":
                params = [{m.args[0]: v} for v in m.args[1]]
        for p in params:
            rec.case = name + ("[%s]" % list(p.values())[0] if p else "")
            fn(**{a: p[a] if a in p else fixtures[a] for a in inspect.signature(fn).parameters})
    out = {"source": "the oracle (--from-oracle)" if from_oracle else "oracle/_ref", "calls": rec.calls()}
    with open(ref_py.GOLDEN, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(ref_py.GOLDEN, len(out["calls"]), "calls", os.path.getsize(ref_py.GOLDEN), "bytes")


if __name__ == "__main__":
    main()
