"""kmerlr_b200 -- B200 (sm_100a) implementation of the data-parallel hot path of pbenner/kmerLr:
k-mer feature extraction, sparse logistic loss / gradient with the proximal-gradient estimator and
the leapfrog selection, and sliding-window genomic scoring.  See DESIGN.md / INTEGRATION.md."""
from ._lib import KmerLrError, SO_PATH, TIE_GO118, TIE_INDEX  # noqa: F401
from .api import (  # noqa: F401
    CoeffIndex, KmerDataSet, KmerLrEstimator, NewKmerCounter, Sequences, Transform, TransformFull, comm_destroy, comm_init,
    comm_init_torch, comm_unique_id, compile_test_data, compile_data, compile_training_data, compute_class_weights,
    featureSelector, flatten, from_csr, import_fasta, from_dense, genomicKmerLr, init, last_device_ms, launch_count,
    logisticRegression, option, select_data, shutdown, wiggle_records, saveWindowPredictionsWiggle, class_name, export_kmers,
    KmerRegularizationPath, Trace, CrossValidation, crossvalidation, cv_groups, cv_scatter,
)
