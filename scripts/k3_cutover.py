"""K3 kernel cutover: BM25 stage time per 256-query batch (P = 30, the bench's query terms) of the warp kernel and the
first-generation kernel, alternating, on shards of several sizes built with the bench's c3 term statistics.  Sets
BW_AUTO_MIN_ROWS (bm25.cu).  Usage: python scripts/k3_cutover.py [rows ...]; one JSON line per size."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import VOCAB, synth_query_terms  # noqa: E402
from kaito_b200 import _native  # noqa: E402
from kaito_b200.sharded import NativeStages  # noqa: E402


def main():
    sizes = [int(s) for s in sys.argv[1:]] or [625_000, 1_250_000, 2_500_000, 5_000_000]
    dev = torch.device("cuda", 0)
    B, P, iters = 256, 30, 50
    terms = synth_query_terms(B, 11)
    offs = np.zeros(B + 1, np.int32)
    offs[1:] = np.cumsum([len(t) for t in terms])
    d_terms = torch.from_numpy(np.concatenate(terms).view(np.int32)).to(dev)
    d_toff = torch.from_numpy(offs).to(dev)
    ctx = _native.Context(device_id=0)
    try:
        for n in sizes:
            ix = ctx.create_index(f"cut{n}", 32)       # narrow rows: only the postings matter here
            ix.synth_fill(n, row_base=0, seed=20260921, vocab=VOCAB)
            ix.commit(VOCAB)
            st = NativeStages(ctx, ix)
            keys = {k: torch.empty((B, P), dtype=torch.int64, device=dev) for k in ("warp", "legacy")}
            res = {"rows": n, "batch": B, "P": P, "warp_ms": [], "legacy_ms": []}
            for _ in range(3):
                for kern in ("warp", "legacy"):
                    os.environ["KRAG_BM25_KERNEL"] = kern
                    for _ in range(5):
                        st.bm25_candidates(d_terms, d_toff, B, P, keys[kern], offs)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(iters):
                        st.bm25_candidates(d_terms, d_toff, B, P, keys[kern], offs)
                    e1.record()
                    torch.cuda.synchronize()
                    res[f"{kern}_ms"].append(e0.elapsed_time(e1) / iters)
            res["same_keys"] = bool(torch.equal(keys["warp"], keys["legacy"]))
            print(json.dumps(res), flush=True)
            ix.drop()
    finally:
        os.environ.pop("KRAG_BM25_KERNEL", None)
        ctx.close()


if __name__ == "__main__":
    main()
