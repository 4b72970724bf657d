"""Host restatement of the merge of per-shard range results (``ivr_range_merge_keys_device``), the checker of the
sharded range-search tests (TEST INFRASTRUCTURE ONLY)."""
from __future__ import annotations

import numpy as np

from oracle import flat_ip


def merge_range_parts(lims_parts, keys_parts):
    """The range results of several row shards, each a run of packed keys per query (``flat_ip.pack_keys``; part p
    holds query q's hits at ``keys_parts[p][lims_parts[p][q]:lims_parts[p][q + 1]]``), merged into one
    (lims, D float32, I int64).  Each query's runs are concatenated in part order and sorted by the unsigned key
    descending (score descending, then lower id); the sort is stable, so an equal key of a lower part comes first."""
    lims_parts = [np.asarray(lp, np.int64) for lp in lims_parts]
    keys_parts = [np.asarray(kp).view(np.uint64) if np.asarray(kp).dtype == np.int64 else np.asarray(kp, np.uint64)
                  for kp in keys_parts]
    nq = lims_parts[0].size - 1
    lims = np.zeros(nq + 1, np.int64)
    runs = []
    for q in range(nq):
        k = np.concatenate([kp[lp[q]:lp[q + 1]] for lp, kp in zip(lims_parts, keys_parts)]).astype(np.uint64)
        runs.append(k[np.argsort(~k, kind="stable")])
        lims[q + 1] = lims[q] + k.size
    keys = np.concatenate(runs) if runs else np.zeros(0, np.uint64)
    D, I = flat_ip.unpack_keys(keys)
    return lims, D.astype(np.float32), I.astype(np.int64)
