"""CPU test of bench.py --dump-outputs: the files hold the proof bytes and the input claims exactly, and the total stays
within the size limit."""
import os

import numpy as np

GL_P = 2**64 - 2**32 + 1


class _Transcript:
    def __init__(self, proof):
        self.proof = proof

    def into_proof(self):
        return self.proof


def test_dump_outputs_round_trips_proofs_and_claims(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(3)
    claims = [[(rng.integers(0, GL_P, (17, 2), dtype=np.uint64), rng.integers(0, GL_P, 2, dtype=np.uint64))] for _ in range(3)]
    claims[1][0][1][0] = np.uint64(2**64 - 1)
    last = [(_Transcript(rng.integers(0, 256, 1000, dtype=np.uint8).tobytes()), claims) for _ in range(3)]
    bench.dump_outputs(str(tmp_path), last)
    words = np.concatenate([a.reshape(-1) for node in claims for pt, val in node for a in (pt, val)])
    for k, (tr, _) in enumerate(last):
        proof = np.load(tmp_path / f"proof_{k}.npy")
        assert proof.dtype == np.float32 and proof.astype(np.uint8).tobytes() == tr.into_proof()
        cl = np.load(tmp_path / f"input_claims_{k}.npy")
        assert cl.dtype == np.float64 and cl.shape == (words.size, 2)
        assert (cl[:, 0].astype(np.uint64) | (cl[:, 1].astype(np.uint64) << np.uint64(32)) == words).all()
    one_slot = 1000 * 4 + words.size * 16
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 2 * one_slot)
    capped = tmp_path / "capped"
    bench.dump_outputs(str(capped), last)
    assert sorted(os.listdir(capped)) == ["input_claims_0.npy", "input_claims_1.npy", "proof_0.npy", "proof_1.npy"]
