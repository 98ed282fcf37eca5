"""fastF-b200: the `bam2db` and `freq` hot paths of yuw444/fastF on sm_100a CUDA (libfastf_gpu.so, include/fastf_gpu.h).

    fastf_b200.bam2db(bam, db, out_dir, barcodes, features, rate_cell, rate_depth, seed)   reference src/bam2db_ds.h:62-70
    fastf_b200.bam2db_sweep(bam, db, out_dir, barcodes, features, rate_cell, rates, seed)  several depth rates out of one pass
    fastf_b200.bam2db_grid(bam, db, out_dir, barcodes, features, cell_rates, rates, seed)  several cell x depth rates out of one pass
    fastf_b200.cell_counts(R1, l, u) / print_tree(hist, fp) / freq(R1, out_dir, l, u)      reference src/count.h:6, src/filter.h:77
"""
from ._lib import Context, FastfError, load   # noqa: F401
from .bam2db_host import bam2db, bam2db_grid, bam2db_sweep   # noqa: F401
from .freq_host import cell_counts, freq, print_tree   # noqa: F401
