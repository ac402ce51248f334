"""Plane masks of the coded block-rows of the structured cantilever (DESIGN.md §3, §4): the (mask, n) histogram that
decides which masks the block reader decodes with compile-time registers (saa_decode_block in csrc/saa_kernels.cuh).

For each of --meshes the one-partition device set-up is built with its CSR kept, and the Python model of the layout
(tests/test_gpu_value_coding.py::coded_model, same slices, same coding rule) counts the block-rows of every mask,
coded and raw.  The plan's coded-plane counter must equal the model's.  The schedule-variant times come from
profiles/value_coding_probe.py, run on the same tree.

    python profiles/lane_major_probe.py [--meshes 24] [--out profiles/lane_major]
"""
import argparse
import collections
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SIGMA, SPAN = 1024, 65535


def mask_histogram(K):
    """{coded: [(mask, n, block-rows)], raw: [...]}: the layout of tests/test_gpu_value_coding.py::coded_model"""
    n = K.shape[0]
    nn = n // 3
    r = np.repeat(np.arange(n), np.diff(K.indptr))
    c = K.indices.astype(np.int64)
    key, inv = np.unique((r // 3) * nn + c // 3, return_inverse=True)
    vals = np.zeros((key.size, 9))
    vals[inv, 3 * (r % 3) + c % 3] = K.data
    bits = np.zeros(key.size, dtype=np.int64)
    np.bitwise_or.at(bits, inv, 1 << (3 * (r % 3) + c % 3))
    nblk = np.bincount(key // nn, minlength=nn)
    first = np.concatenate([[0], np.cumsum(nblk)])
    order = np.lexsort((-nblk, np.arange(nn) // SIGMA))
    lane_node = np.concatenate([order, -np.ones(-nn % 32, dtype=np.int64)]).reshape(-1, 32)
    lane_nblk = np.where(lane_node >= 0, nblk[np.maximum(lane_node, 0)], 0)
    L = lane_nblk.max(axis=1)
    s_of = np.repeat(np.arange(L.size), L)
    j_of = np.arange(s_of.size) - np.repeat(np.cumsum(L) - L, L)
    valid = j_of[:, None] < lane_nblk[s_of]
    bid = np.where(valid, first[np.maximum(lane_node[s_of], 0)] + j_of[:, None], -1)
    mask = np.bitwise_or.reduce(np.where(valid, bits[np.maximum(bid, 0)], 0), axis=1)
    lv = np.where(valid[:, :, None], vals[np.maximum(bid, 0)], 0.0).view(np.int64)
    span = lv.max(axis=1).astype(np.uint64) - lv.min(axis=1).astype(np.uint64)
    stored = (mask[:, None] >> np.arange(9)) & 1 == 1
    code = (mask != 0) & np.all(~stored | (span <= SPAN), axis=1)
    rows = lambda sel: [dict(mask=f"0x{k:03x}", n=bin(k).count("1"), block_rows=v)
                        for k, v in collections.Counter(mask[sel].tolist()).most_common()]
    return dict(block_rows=int(mask.size), coded_block_rows=int(code.sum()), coded_planes=int(stored[code].sum()),
                coded=rows(code), raw=rows(~code))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--meshes", type=int, nargs="+", default=[24])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lane_major"))
    a = ap.parse_args()
    import torch
    from saa_b200 import device_setup as ds
    if not torch.cuda.is_available():
        raise SystemExit("lane_major_probe: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    result = {}
    for m in a.meshes:
        plans, info = ds.build_structured_in_process(m, 1, keep_csr=True)
        h = mask_histogram(info[0]["K"].to_scipy())
        assert h["coded_planes"] == plans[0].coded_planes, (h["coded_planes"], plans[0].coded_planes)
        result[str(m)] = dict(n_dof=plans[0].n_dof, **h)
        print(json.dumps({m: result[str(m)]}), flush=True)
        del plans, info
        torch.cuda.empty_cache()
    path = os.path.join(a.out, "mask_histogram.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(f"[lane_major_probe] wrote {path}")


if __name__ == "__main__":
    main()
