"""Writes the data in this directory: what the tests that compare with the reference project (Kolibrie, commit 1d7c306c) need from it,
so that they run on machines without its checkout.

  line_counts.json          the number of lines of every .rs / .cu file of the checkout, by path inside it: the line ranges that the
                            fixtures and the sources cite must exist (tests/test_golden_provenance.py)
  cuda_join_signature.json  the parameters of perform_hash_join_cuda as the reference defines it (kolibrie/src/cuda/cuda_join.cu) and
                            as its Rust side declares it (kolibrie/src/cuda/cuda_join.rs) (tests/test_abi.py)
  cuda_stub_salary.npz      what the reference's own CUDA stub returns for one seeded input: kolibrie/src/cuda/cuda_join.cu built for
                            sm_100a into oracle/_ref/ by `make -C oracle REF=<checkout>` (tests/test_gpu_parity.py)

    python tests/golden/reference/make_reference_golden.py checkout <path of the reference checkout>   # the first two, no GPU
    python tests/golden/reference/make_reference_golden.py stub                                      # the third, on a B200
"""
import hashlib
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(HERE)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

STUB_EMPLOYEES = 30000  # 180 000 triples: inside the range the stub's clamped grid covers (148 SMs x 2048 threads)
STUB_PREDICATE = "ds:annual_salary"


def c_params(text, opener):
    """the parameter list of the declaration that starts with `opener`, comments removed, whitespace collapsed"""
    body = text[text.index(opener) + len(opener):]
    body = body[: body.index(")")]
    body = re.sub(r"/\*.*?\*/|//[^\n]*", " ", body, flags=re.S)
    return [" ".join(x.split()) for x in body.split(",") if x.strip()]


def stub_input():
    """the seeded input of the stub comparison: (s, p, o, predicate id, sha256 of the three columns)"""
    from kolibrie_b200 import datagen

    d = datagen.employee_dataset(STUB_EMPLOYEES)
    h = hashlib.sha256()
    for col in (d.s, d.p, d.o):
        h.update(np.ascontiguousarray(col, dtype=np.uint32).tobytes())
    return d.s, d.p, d.o, int(d.ids[STUB_PREDICATE]), h.hexdigest()


def write_checkout_data(ref):
    counts = {}
    for d, _, fs in os.walk(ref):
        for f in fs:
            if f.endswith((".rs", ".cu")):
                p = os.path.join(d, f)
                counts[os.path.relpath(p, ref)] = sum(1 for _ in open(p, errors="replace"))
    with open(os.path.join(HERE, "line_counts.json"), "w") as f:
        json.dump({"files": dict(sorted(counts.items()))}, f, indent=0)
        f.write("\n")
    cu = open(os.path.join(ref, "kolibrie", "src", "cuda", "cuda_join.cu")).read()
    rs = open(os.path.join(ref, "kolibrie", "src", "cuda", "cuda_join.rs")).read()
    sig = {"cuda_join.cu": c_params(cu, "void perform_hash_join_cuda("), "cuda_join.rs": c_params(rs, "pub fn perform_hash_join_cuda(")}
    with open(os.path.join(HERE, "cuda_join_signature.json"), "w") as f:
        json.dump(sig, f, indent=1)
        f.write("\n")


def write_stub_data():
    from kolibrie_b200 import capi as c

    stub = os.path.join(ROOT, "oracle", "_ref", "libcudajoin_ref.so")
    s, p, o, pred, digest = stub_input()
    theirs = np.sort(c.legacy_hash_join_cuda(s, p, o, pred, libpath=stub))  # sorted: the stub's order is atomicAdd arrival order
    np.savez_compressed(os.path.join(HERE, "cuda_stub_salary.npz"), indices=theirs.astype(np.uint32), predicate=np.uint32(pred),
                        input_sha256=np.array(digest))


if __name__ == "__main__":
    if sys.argv[1:2] == ["checkout"] and len(sys.argv) == 3:
        write_checkout_data(sys.argv[2])
    elif sys.argv[1:] == ["stub"]:
        write_stub_data()
    else:
        raise SystemExit(__doc__)
