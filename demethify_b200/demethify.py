"""`demethify` command line — drop-in for the reference's demethify/demethify.py:main (same flags, same output files:
celltypes_proportions.csv, methylation_profile_estimate.csv, confidence_interval_*.csv, log.log), running the
deconvolution on the B200 kernel library.  Additive flags: --precision {fp64,fp32}, --engine {auto,gram,stream}.  Plotting is imported lazily
(matplotlib / seaborn / colorcet are optional)."""
import argparse
import os
import sys
import warnings
from time import time

import numpy as np
import pandas as pd

from . import set_engine, set_precision
from .bootstrap import bt_ci
from .deconvolution import (best_of_restarts, cost_f_w, init_BSSMF_md, init_BSSMF_md_p, mdwbssmf_deconv, mdwbssmf_deconv_p,
                            unsupervised_deconv)
from .ic import evaluate_best_ic
from .init_func import wls_all_samples

warnings.filterwarnings("ignore")

LOGO = r"""
    ____                      __  __    _ ____
   / __ \___  ____ ___  ___  / /_/ /_  (_) __/_  __
  / / / / _ \/ __ `__ \/ _ \/ __/ __ \/ / /_/ / / /
 / /_/ /  __/ / / / / /  __/ /_/ / / / / __/ /_/ /
/_____/\___/_/ /_/ /_/\___/\__/_/ /_/_/_/  \__, /   (B200)
                                          /____/
"""


def build_parser():
    p = argparse.ArgumentParser(description="DeMethify - Partial reference-based Methylation Deconvolution (B200 path)")
    p.add_argument("--methfreq", nargs="+", type=str, required=True, help="Methylation frequency file path (values between 0 and 1)")
    p.add_argument("--ref", nargs="?", type=str, help="Methylation reference matrix file path")
    p.add_argument("--iterations", nargs=2, type=int, help="Numbers of iterations for outer and inner loops (default without purity = 10000, 20, with purity= 100, 500)")
    p.add_argument("--nbunknown", nargs=1, type=int, help="Number of unknown cell types to estimate ")
    p.add_argument("--purity", nargs="+", type=float, help="The purities of the samples in percent [0,100], if known")
    p.add_argument("--termination", nargs=1, type=float, default=1e-2, help="Termination condition for cost function (default = 1e-2)")
    p.add_argument("--init", nargs="?", default="uniform_", help="Initialisation option, the default is uniform_, and the options are: uniform, uniform_, beta, SVD, ICA. ")
    p.add_argument("--outdir", nargs="?", required=True, help="Output directory")
    p.add_argument("--fillna", action="store_true", help="Replace every NA by 0 in the given data")
    p.add_argument("--ic", nargs="+", help="Select number of unknown cell types by minimising a criterion (AIC, BIC, CCC, BCV, minka)")
    p.add_argument("--confidence", nargs=2, type=int, help="Outputs bootstrap confidence intervals, takes confidence level and boostrap iteration numbers as input.")
    p.add_argument("--plot", action="store_true", help="Plot cell type proportions estimates for each sample, eventually with confidence intervals. ")
    p.add_argument("--restart", nargs=1, type=int, help="Number of random restarts among which to select the one with the lowest cost/highest loglikelihood")
    p.add_argument("--seed", nargs=1, type=int, default=1, help="Set a seed integer number for random number generation for reproducibility. ")
    p.add_argument("--noprint", action="store_true", help="Doesnt show the logo.")
    p.add_argument("--bedmethyl", action="store_true", help="Flag to indicate that the input will be bedmethyl files, modkit style")
    p.add_argument("--precision", choices=["fp64", "fp32"], default="fp64", help="(B200 path) arithmetic of the solver kernels")
    p.add_argument("--engine", choices=["auto", "fused", "gram", "stream"], default="auto",
                   help="(B200 path) device engine: one fused pass per outer iteration (default where supported), Gram-form statistics, "
                        "or per-iteration streaming passes")
    p.add_argument("--distinct-restarts", action="store_true",
                   help="(B200 path) --restart R draws restart r from seed + r and keeps the lowest cost (the reference re-seeds every "
                        "restart identically, so its R restarts are one fit); with --confidence every resample is fitted R times")
    p.add_argument("--shard", choices=["fits", "rows"], default="fits",
                   help="(B200 path, under torchrun) how several GPUs are used: 'fits' runs independent fits per GPU (--ic, --confidence; "
                        "the main fit runs on every GPU), 'rows' shards the CpG rows of every fit over the GPUs (the main fit and --ic AIC / "
                        "BIC / CCC / BCV with a reference matrix, a CCC member's restarts and a BCV member's folds as one batch; --confidence stays "
                        "fit-sharded); every shape a one-GPU fit runs can be row-sharded (more than 8 unknown types, or more than 4 with 7+ known "
                        "ones, run the stream engine's passes with one all-reduce per step)")
    return p


def _pinned_matrix(rows, cols, dtype):
    """(rows, cols) C-ordered numpy matrix backed by page-locked host memory when CUDA is there (the H2D copy of the solver then
    runs at full PCIe rate); plain numpy otherwise."""
    import torch
    tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.int64): torch.int64, np.dtype(np.int32): torch.int32,
           np.dtype(np.uint16): torch.uint16}[np.dtype(dtype)]
    try:
        if torch.cuda.is_available():
            return torch.empty((rows, cols), dtype=tdt, pin_memory=True).numpy()
    except RuntimeError:
        pass
    return np.empty((rows, cols), dtype=dtype)


def read_inputs(args):
    """demethify.py:103-143 — bedmethyl (tab separated, percent_modified in percent) or csv (fraction) readers.

    Same parser as the reference (pandas' C reader with its default float conversion, so every value is bit-identical), but the
    sample files are parsed concurrently (the reader releases the GIL), only the two columns the solver uses are converted, and
    each sample lands directly in its column of one page-locked M x N matrix (SURVEY 8 f3)."""
    from concurrent.futures import ThreadPoolExecutor
    ref, header = None, []
    sep = "\t" if args.bedmethyl else ","
    if args.ref:
        ref_df = pd.read_csv(args.ref, sep=sep)
        if args.bedmethyl:
            ref_df = ref_df.iloc[:, 3:]
        if args.fillna:
            ref_df = ref_df.fillna(0)
        header = list(ref_df.columns)
        ref = ref_df.values

    def load(path):
        cols = list(pd.read_csv(path, sep=sep, nrows=0).columns)
        single = (not args.bedmethyl) and len(cols) == 1                 # csv with frequencies only: coverage 1 (demethify.py:136-137)
        use = ["percent_modified"] + ([] if single else ["valid_coverage"])
        t = pd.read_csv(path, sep=sep, usecols=use)
        if single:
            t["valid_coverage"] = 1
        if args.fillna:
            t = t.fillna(0)
        f = t["percent_modified"].values
        return (f / 100 if args.bedmethyl else f), t["valid_coverage"].values

    paths = list(args.methfreq)
    with ThreadPoolExecutor(max_workers=min(len(paths), os.cpu_count() or 1, 32)) as ex:
        first = load(paths[0])
        M = first[0].shape[0]
        int_cov = np.issubdtype(first[1].dtype, np.integer)
        meth_f = _pinned_matrix(M, len(paths), np.float64)
        # integer coverage is staged as uint16 (what the kernels store, a quarter of the int64 bytes on the way to the GPU); a column
        # that does not fit switches the whole matrix back to int64 below
        narrow = int_cov and first[1].size > 0 and 0 <= int(first[1].min()) and int(first[1].max()) <= 65535
        counts = _pinned_matrix(M, len(paths), (np.uint16 if narrow else np.int64) if int_cov else np.float64)
        wide_cols = {}

        float_cols = {}                                   # coverage columns that are not integer typed (NaN without --fillna, ...)

        def place(j, pair):
            f, c = pair
            if f.shape[0] != M:
                raise ValueError("all input files must have the same number of rows")      # np.column_stack raises in the reference
            meth_f[:, j] = f
            if int_cov and not np.issubdtype(c.dtype, np.integer):
                float_cols[j] = c
            elif counts.dtype == np.uint16 and c.size and (int(c.min()) < 0 or int(c.max()) > 65535):
                wide_cols[j] = c
            else:
                counts[:, j] = c
        place(0, first)
        list(ex.map(lambda j: place(j, load(paths[j])), range(1, len(paths))))
    if wide_cols:                                         # coverage beyond 16 bits somewhere: int64 like the reference
        counts = counts.astype(np.int64)
        for j, c in wide_cols.items():
            counts[:, j] = c
    if float_cols:                                        # np.column_stack of mixed int / float columns is float64 in the reference
        counts = counts.astype(np.float64)
        for j, c in float_cols.items():
            counts[:, j] = c
    return meth_f, counts, ref, header


def _init_distributed():
    """One process per GPU under torchrun (RANK / WORLD_SIZE / LOCAL_RANK in the environment): NCCL process group, device by
    local rank.  Returns (rank, world)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return 0, 1
    import torch
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist.get_rank(), dist.get_world_size()


def _row_sharded_main_fit(meth_f, counts, ref, n_u, purity, init_option, seed, it1, it2, tol, rank, world):
    """The main fit with the CpG rows sharded over the ranks: rank r keeps row_range(M, r, world) of what it read; the initial
    iterate and the fit all-reduce their row sums.  -> (u over all rows in row order on rank 0, None elsewhere; alpha)."""
    import torch.distributed as dist
    from .sharded import (init_BSSMF_md_p_sharded, init_BSSMF_md_sharded, mdwbssmf_deconv_sharded, row_range, unsupervised_init_sharded,
                          wls_all_samples_sharded)
    lo, hi = row_range(meth_f.shape[0], rank, world)
    X, D = meth_f[lo:hi], counts[lo:hi]
    R = None if ref is None else np.asarray(ref)[lo:hi]
    if R is not None and n_u == 0:
        return None, wls_all_samples_sharded(X, D, R, y_is_dx=True)                      # demethify.py:209-213
    if R is None:
        u0, a0 = unsupervised_init_sharded(init_option, X, D, n_u, seed=seed)
    elif purity is not None:
        u0, a0 = init_BSSMF_md_p_sharded(init_option, X, D, R, n_u, purity, seed=seed)
    else:
        u0, a0 = init_BSSMF_md_sharded(init_option, X, D, R, n_u, seed=seed)
    u, alpha, _n, _cost = mdwbssmf_deconv_sharded(u0, a0, X, D, R, n_u, n_iter1=it1, n_iter2=it2, tol=tol, purity=purity)
    parts = [None] * world if rank == 0 else None
    dist.gather_object(u, parts, dst=0)
    return (np.concatenate(parts, axis=0) if rank == 0 else None), alpha


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.plot:
        try:
            from . import plotting  # noqa: F401
        except ImportError:
            sys.stderr.write("Error: --plot is not part of the B200 path (presentation only, SURVEY.md 2.1 row 9): run the reference's "
                             "plotting.py on the CSV files this command writes.\n")
            sys.exit(1)
    set_precision(args.precision)
    set_engine(args.engine)
    rank, world = _init_distributed()
    args.restart = 1 if args.restart is None else args.restart[0]
    if not args.iterations:
        args.iterations = [100, 500] if args.purity else [10000, 20]
    if isinstance(args.termination, list):
        args.termination = args.termination[0]
    purity = None
    if args.purity:
        purity = np.array(args.purity)
        if np.any((purity >= 0) & (purity <= 1)):
            print("Purity is between 0 and 1, are you sure that it's a percentage?")
        elif np.any((purity < 0) & (purity > 100)):
            sys.stderr.write("Error: Invalid value for purity, not within [0,100] bounds.")
            sys.exit(1)
        purity = 1 - (purity / 100.0)                         # demethify.py:77
    nb_r = 5
    if args.ic:
        if args.nbunknown:
            sys.stderr.write("Error: --ic cannot be used with --nbunknown.\n")
            sys.exit(1)
        if len(args.ic) > 1:
            nb_r = int(args.ic[1])
        args.ic = args.ic[0]
    if not args.noprint:
        print(LOGO)
    outdir = os.path.join(os.getcwd(), args.outdir)
    if not os.path.exists(outdir):
        print(f"Creating directory {outdir} to store results")
        os.makedirs(outdir, exist_ok=True)
    if args.nbunknown is None:
        args.nbunknown = [0]
    n_u = args.nbunknown[0]
    rows_mode = args.shard == "rows" and world > 1
    if rows_mode and args.distinct_restarts and args.restart > 1:
        sys.stderr.write("Error: --restart R --distinct-restarts runs independent fits: use --shard fits.\n")
        sys.exit(1)
    meth_f, counts, ref, header = read_inputs(args)
    args.methfreq = [name.split("/")[-1] for name in args.methfreq]
    it1, it2, tol = args.iterations[0], args.iterations[1], args.termination

    t0 = time()
    bt_results = None
    if args.confidence:
        bt_results = bt_ci(args.confidence[0], args.confidence[1], n_u, meth_f, counts, ref, args.init, it1, it2, tol, header, outdir,
                           args.methfreq, args.purity, args.seed, restarts=args.restart if args.distinct_restarts else 1)
    list_ic, ic_n_u = None, None
    ref_estimate = None
    if args.ic:
        ref_estimate, proportions, ic_n_u, list_ic = evaluate_best_ic(meth_f, ref, counts, args.init, args.ic, args.seed, iter1=it1,
                                                                      iter2=it2, tol=tol, n_restarts=nb_r, shard=args.shard)
        unknown_header = ["unknown_cell_" + str(i + 1) for i in range(ic_n_u)]
        header = header + unknown_header
    elif rows_mode and (not args.ref or (n_u >= 0 and meth_f.shape[1] >= 1)):
        ref_estimate, proportions = _row_sharded_main_fit(meth_f, counts, ref, n_u, purity if args.purity else None, args.init, args.seed,
                                                          it1, it2, tol, rank, world)
        unknown_header = ["unknown_cell_" + str(i + 1) for i in range(n_u)]
        header = header + unknown_header if args.ref else unknown_header
    elif not args.ref:
        # demethify.py:167-174: every restart re-seeds with the same seed, so all restarts are the same fit (SURVEY Q2)
        ref_estimate, proportions = unsupervised_deconv(meth_f, n_u, counts, args.init, n_iter1=it1, n_iter2=it2, tol=tol, seed=args.seed)
        unknown_header = ["unknown_cell_" + str(i + 1) for i in range(n_u)]
        header = unknown_header
    elif n_u > 0 and meth_f.shape[1] >= 1:
        if args.distinct_restarts and args.restart > 1:
            ref_estimate, proportions, _best, _costs = best_of_restarts(meth_f, counts, ref, n_u, args.init, args.seed, args.restart, it1, it2,
                                                                       tol, purity=purity if args.purity else None)
        elif args.purity:
            u, R, alpha = init_BSSMF_md_p(args.init, meth_f, counts, ref, n_u, purity, seed=args.seed)
            ref_estimate, proportions = mdwbssmf_deconv_p(u, R, alpha, meth_f, counts, ref, n_u, purity, n_iter1=it1, n_iter2=it2, tol=tol)
        else:
            u, R, alpha = init_BSSMF_md(args.init, meth_f, counts, ref, n_u, seed=args.seed)
            ref_estimate, proportions = mdwbssmf_deconv(u, R, alpha, meth_f, counts, ref, n_u, n_iter1=it1, n_iter2=it2, tol=tol)
        unknown_header = ["unknown_cell_" + str(i + 1) for i in range(n_u)]
        header = header + unknown_header
    elif n_u == 0 and meth_f.shape[1] >= 1:
        proportions = wls_all_samples(meth_f, counts, ref, y_is_dx=True)          # demethify.py:209-213
        unknown_header = []
    else:
        sys.exit(f'Invalid number of unknown value! : "{args.nbunknown}" ')
    time_tot = time() - t0
    if rank != 0:                      # under torchrun every rank computed the same result (or its rows of it); rank 0 writes the files
        return
    if ref_estimate is not None:
        pd.DataFrame(ref_estimate).to_csv(outdir + "/methylation_profile_estimate.csv", index=False, header=unknown_header)

    proportions = pd.DataFrame(proportions)
    proportions.index = header
    proportions.columns = args.methfreq
    proportions.index.name = "Cell types"
    proportions.to_csv(outdir + "/celltypes_proportions.csv", index=True)
    print("All demethified! Results in " + outdir)
    with open(os.path.join(outdir, "log.log"), "w+") as f:
        f.write("Total execution time = " + str(time_tot) + " s" + "\n")
        if args.ic:
            f.write("Number of unknowns that minimises " + args.ic + " : " + str(ic_n_u))
    if args.plot:
        try:
            from .plotting import plot_proportions
        except ImportError as e:
            sys.stderr.write(f"--plot needs matplotlib / seaborn / colorcet ({e}); results were written without plots\n")
        else:
            plot_proportions(proportions, bt_results[0] if bt_results else pd.DataFrame(), outdir, list_ic)


if __name__ == "__main__":
    main()
