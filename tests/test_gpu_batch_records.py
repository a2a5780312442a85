"""GPU tier: the challenge records of the per-batch call families stay apart.

lwkzg_debug_cell_batch_challenges reports the last cell batch call (lwkzg_verify_[blob_]cell_kzg_proof_batches) and
lwkzg_debug_blob_batch_challenges the last blob-proof batch call (lwkzg_verify_blob_kzg_proof_batches), whichever of
the two families ran last and in whichever form, host or device."""
import os

import pytest

from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MODE = 2
NBLOBS = 5


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


@pytest.fixture(scope="module")
def d(lw):
    lw.set_option("mode", MODE)
    lw.set_option("window_bits", 8)
    lw.set_option("cell_window_bits", 8)
    try:
        s = lw.load_trusted_setup_file(os.path.join(GOLDEN, "trusted_setup.txt"))
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 16)
        lw.set_option("cell_window_bits", 13)
    blobs = [make_blob(700 + b, MODE) for b in range(NBLOBS)]
    coms, proofs, st = lw.commit_and_prove_batch(b"".join(blobs), NBLOBS, s)
    assert st == [0] * NBLOBS
    cells, cproofs, st = lw.compute_cells_and_kzg_proofs_batch(b"".join(blobs), NBLOBS, s)
    assert st == [0] * NBLOBS

    def cell_batch(sel):   # [(blob, cell index)] -> (commitments, indices, cells, proofs)
        return ([coms[b] for b, _ in sel], [k for _, k in sel], [cells[(b * 128 + k) * 2048: (b * 128 + k + 1) * 2048] for b, k in sel],
                [cproofs[(b * 128 + k) * 48: (b * 128 + k + 1) * 48] for b, k in sel])

    def blob_batch(idx):   # blob indices -> (blobs, commitments, proofs)
        return ([blobs[i] for i in idx], [coms[i] for i in idx], [proofs[i] for i in idx])

    # different batch counts, so that a record of the other family could not even be read back in full
    cell_batches = [cell_batch([(0, 3), (1, 90), (2, 127)]), cell_batch([]), cell_batch([(3, 0), (4, 64)])]
    blob_batches = [blob_batch([0, 1]), blob_batch([2, 3, 4]), blob_batch([]), blob_batch([4, 0])]
    yield s, cell_batches, blob_batches
    s.free()


def _cells_device(lw, batches, s):
    import torch

    def dev(raw):
        return torch.frombuffer(bytearray(raw or b"\0"), dtype=torch.uint8).cuda()

    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[1]))
    d_c = dev(b"".join(c for b in batches for c in b[0]))
    d_i = torch.tensor([i for b in batches for i in b[1]] or [0], dtype=torch.int64, device="cuda")
    d_cl = dev(b"".join(c for b in batches for c in b[2]))
    d_p = dev(b"".join(c for b in batches for c in b[3]))
    d_ok = torch.zeros(len(batches), dtype=torch.int32, device="cuda")
    lw.verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_c.data_ptr(), d_i.data_ptr(), d_cl.data_ptr(), d_p.data_ptr(), offs, s)
    torch.cuda.synchronize()
    return [bool(v) for v in d_ok.cpu().tolist()]


def _blobs_device(lw, batches, s):
    import torch

    def dev(raw):
        return torch.frombuffer(bytearray(raw or b"\0"), dtype=torch.uint8).cuda()

    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[0]))
    cols = [dev(b"".join(x for b in batches for x in b[c])) for c in range(3)]
    d_ok = torch.zeros(len(batches), dtype=torch.int32, device="cuda")
    lw.verify_blob_kzg_proof_batches_device(d_ok.data_ptr(), cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), offs, s)
    torch.cuda.synchronize()
    return [bool(v) for v in d_ok.cpu().tolist()]


def test_families_keep_their_own_challenges(lw, d):
    s, cell_batches, blob_batches = d
    kc, kb = len(cell_batches), len(blob_batches)
    oks, sts = lw.verify_cell_kzg_proof_batches(cell_batches, s)
    assert oks == [True] * kc and sts == [0] * kc
    rc = lw.debug_cell_batch_challenges(kc, s)
    oks, sts = lw.verify_blob_kzg_proof_batches(blob_batches, s)
    assert oks == [True] * kb and sts == [0] * kb
    rb = lw.debug_blob_batch_challenges(kb, s)
    assert rc[0] and rc[2] and not rc[1]
    assert rb[0] and rb[1] and rb[3] and not rb[2]
    assert not set(rc) & set(rb) - {0}
    assert lw.debug_cell_batch_challenges(kc, s) == rc

    # device forms, interleaved both ways
    assert _cells_device(lw, cell_batches, s) == [True] * kc
    assert lw.debug_blob_batch_challenges(kb, s) == rb
    assert lw.debug_cell_batch_challenges(kc, s) == rc
    assert _blobs_device(lw, blob_batches, s) == [True] * kb
    assert lw.debug_cell_batch_challenges(kc, s) == rc
    assert lw.debug_blob_batch_challenges(kb, s) == rb

    # a host call of one family after a device call of the other
    lw.verify_cell_kzg_proof_batches(cell_batches, s)
    assert lw.debug_blob_batch_challenges(kb, s) == rb
    assert lw.debug_cell_batch_challenges(kc, s) == rc
    assert _cells_device(lw, cell_batches, s) == [True] * kc
    lw.verify_blob_kzg_proof_batches(blob_batches, s)
    assert lw.debug_cell_batch_challenges(kc, s) == rc
    assert lw.debug_blob_batch_challenges(kb, s) == rb
