"""lambdaworks_kzg_b200 -- Python host-side mirror of the reference's C ABI over
liblwkzg_b200.so (CUDA, sm_100a).

The function names, argument meaning and error behaviour follow
lambdaworks_kzg's `extern "C"` surface (/root/reference/src/lib.rs:245-858):
every call returns the result or raises :class:`KzgError` carrying the
``C_KZG_RET`` code the C function returned.  PyTorch is only used (optionally,
by the ``*_device`` helpers) for device memory and streams.

There is no CPU implementation behind this package: if the CUDA library is
missing or no GPU is usable the calls fail loudly.
"""
from .api import (  # noqa: F401
    BYTES_PER_BLOB,
    C_KZG_BADARGS,
    C_KZG_ERROR,
    C_KZG_MALLOC,
    C_KZG_OK,
    KzgError,
    bench_msm_kernel,
    bench_pairing,
    bench_var_msm,
    window_bits,
    Settings,
    blob_to_kzg_commitment,
    blob_to_kzg_commitment_batch,
    commit_and_prove_batch,
    commit_and_prove_batch_device,
    compute_blob_kzg_proof,
    compute_blob_kzg_proof_batch,
    compute_kzg_proof,
    compute_kzg_proof_batch,
    g1_lincomb,
    get_option,
    imad_peak,
    kernel_launches,
    last_error,
    lib_path,
    load_library,
    load_trusted_setup,
    load_trusted_setup_file,
    set_option,
    synth_blob_host,
    synth_point_dlogs,
    table_geometry,
    synth_blobs_device,
    debug_batch_challenge,
    verify_batch_phase1,
    verify_batch_phase2,
    verify_batch_phase3,
    verify_batch_phase1_device,
    verify_batch_phase2_device,
    verify_batch_phase3_device,
    set_devices,
    get_devices,
    verify_blob_kzg_proof,
    verify_blob_kzg_proof_batch,
    verify_blob_kzg_proof_batch_device,
    verify_blob_kzg_proof_batch_ptr,
    blob_to_kzg_commitment_batch_device,
    compute_blob_kzg_proof_batch_device,
    verify_kzg_proof,
    compute_cells_and_kzg_proofs,
    compute_cells_and_kzg_proofs_batch,
    compute_cells_and_kzg_proofs_batch_device,
    recover_cells_and_kzg_proofs,
    recover_cells_and_kzg_proofs_batch,
    recover_cells_and_kzg_proofs_batch_device,
    verify_cell_kzg_proof_batch,
    cell_window_bits,
    table_share,
    debug_cell_stages,
)
from .sharding import shard_range, verify_blob_kzg_proof_batch_distributed, verify_blob_kzg_proof_batch_distributed_device  # noqa: F401
