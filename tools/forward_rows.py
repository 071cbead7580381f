"""Compare the network rows of two builds bit for bit.

  python tools/forward_rows.py dump OUT.npz [TREE]    policy / value rows of the bf16 and bf16x3 trunks, from the library
                                                     built in TREE (a checkout; default: this one)
  python tools/forward_rows.py compare A.npz B.npz   exit status 1 unless every row is bit-identical

The batch sizes sit on both sides of every edge of the trunk's dispatch bands (one tile per CTA up to 148 positions, two
up to 370, trunk_pp_body<1> up to 518, trunk_pp_large_kernel above) on a 148-SM B200; model and positions are seeded.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [1, 74, 148, 149, 222, 223, 370, 371, 518, 519, 740, 1200]


def dump(out, tree):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.join(os.path.abspath(tree), "ultimate-tictactoe-alphazero_b200"))
    import torch
    import engine
    import oracle_lib as O
    from dual_network import DualNetwork

    torch.manual_seed(0)
    e = engine.Engine(n_slots=max(SIZES), max_sims=50, max_batch=8, max_games=8)
    e.upload_model(DualNetwork().eval())
    sts = np.concatenate([O.playout_states(1, g)[0][:-1] for g in range(max(SIZES) // 40 + 2)])[:max(SIZES)]
    rows = {}
    for numerics in ("bf16", "bf16x3"):
        for n in SIZES:
            d = torch.from_numpy(np.ascontiguousarray(sts[:n]).view(np.int32)).cuda()
            p, v = e.net_forward(d, engine.evaluator_of(numerics))
            rows["%s_%d_policy" % (numerics, n)] = p.cpu().numpy()
            rows["%s_%d_value" % (numerics, n)] = v.cpu().numpy()
    e.close()
    np.savez(out, **rows)
    print("%s: %d arrays from %s" % (out, len(rows), engine.LIB_PATH))


def compare(a, b):
    A, B = np.load(a), np.load(b)
    bad = 0
    for k in sorted(A.files, key=lambda k: (k.split("_")[0], int(k.split("_")[1]), k)):
        same = k in B.files and A[k].shape == B[k].shape and A[k].tobytes() == B[k].tobytes()
        bad += not same
        if not same:
            print("DIFFERENT %s" % k)
    missing = sorted(set(B.files) - set(A.files))
    for k in missing:
        print("DIFFERENT %s (missing in %s)" % (k, a))
    print("%d arrays, %d different" % (len(A.files), bad + len(missing)))
    return 1 if bad or missing else 0


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else ROOT)
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
