"""Build tests/golden/simdata_kat.npz from a checkout of GaussianProcesses.jl:

    python tests/golden/make_golden.py <path to GaussianProcesses.jl>

Source of the known-answer vector (paths relative to that checkout):
  perf/benchmarks/simdata.csv                              3000 x 10 inputs + Y
  perf/benchmarks/notebooks/benchmark_julia.ipynb cell 6   recorded output of the reference:
      GPE(X, Y, MeanConst(0.0), SEIso(0.0,0.0), log(1.0))  ->  mll, dmll
The recorded run used the 2018 package version that added a 1e-5 diagonal jitter; the current
source (src/GPE.jl:173-174) has none.  Both are pinned in tests/test_oracle_golden.py.
The tests do not need that checkout: they read the committed .npz.
"""
import json, os, sys
import numpy as np

here = os.path.dirname(os.path.abspath(__file__))


def recorded_from_notebook():
    nb = json.load(open(os.path.join(REF, "perf/benchmarks/notebooks/benchmark_julia.ipynb")))
    txt = []
    for c in nb["cells"]:
        for o in c.get("outputs", []):
            for k in ("text",):
                if k in o:
                    txt.append("".join(o[k]))
            d = o.get("data", {})
            if "text/plain" in d:
                txt.append("".join(d["text/plain"]))
    return "\n".join(txt)


if __name__ == "__main__":
    REF = sys.argv[1]
    raw = np.loadtxt(os.path.join(REF, "perf/benchmarks/simdata.csv"), delimiter=",", skiprows=1)
    assert raw.shape == (3000, 11)
    txt = recorded_from_notebook()
    assert "-4536.259909444878" in txt, "recorded mll not found in the notebook"
    np.savez_compressed(
        os.path.join(here, "simdata_kat.npz"),
        X=raw[:, :10], Y=raw[:, 10],
        recorded_mll=np.array(-4536.259909444878),
        recorded_dmll=np.array([-689.634, -15.7312, 71.1964, -667.268]),  # printed to 6 s.f. in the notebook
    )
    print("wrote simdata_kat.npz", raw.shape)
