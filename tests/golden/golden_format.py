"""Storage form of reference_cases.npz, shared by make_golden.py (writes it) and tests/conftest.py (reads it)."""
import numpy as np


def pack_prob_log(frame, prob_log, ids):
    """Lossless compact form of the reference's gathered log-probs prob_log f32 [T, S] (the log-softmax of the
    frame logits, gathered by ids): one column per distinct id, its bits XORed with those of frame minus a
    per-row offset (the log-softmax shift).  What is left is mostly zero bits, which keeps the golden file
    under 1 MB."""
    u, first = np.unique(ids, return_index=True)
    by_id = np.ascontiguousarray(prob_log[:, first], dtype=np.float32)
    f = frame[:by_id.shape[0], u]
    off = np.median(f.astype(np.float64) - by_id, axis=1).astype(np.float32)
    return {"prob_log_offset": off, "prob_log_xor": (f - off[:, None]).view(np.uint32) ^ by_id.view(np.uint32)}


def unpack_prob_log(frame, ids, prob_log_offset, prob_log_xor):
    """Inverse of pack_prob_log, bit for bit (float32 subtraction is exactly rounded everywhere)."""
    u, inv = np.unique(ids, return_inverse=True)
    f = frame[:prob_log_xor.shape[0], u]
    by_id = ((f - prob_log_offset[:, None]).view(np.uint32) ^ prob_log_xor).view(np.float32)
    return np.ascontiguousarray(by_id[:, inv.reshape(-1)])
