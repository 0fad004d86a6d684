"""``spmm_arrow`` command line -- same flags as the reference's ``scripts/spmm_arrow_main.py:10-29``."""
import argparse

from . import arrow_bench


def str2bool(v):
    if isinstance(v, bool):
        return v
    if v is None:
        return True
    if v.lower() in ('yes', 'true', 't', 'y', '1'):
        return True
    if v.lower() in ('no', 'false', 'f', 'n', '0'):
        return False
    raise argparse.ArgumentTypeError('Boolean value expected.')


def main(argv=None) -> None:
    parser = argparse.ArgumentParser(description='Benchmark the arrow SpMM on B200')
    parser.add_argument('-f', '--path', type=str, default=None,
                        help='The filename prefix of the decomposed graph. If none, synthetic data is generated.')
    parser.add_argument('-w', '--width', type=int, default=0, help='Width of the decomposition / Height of the blocks.')
    parser.add_argument('-c', '--features', type=int, default=16, help='Number of feature columns.')
    parser.add_argument('-b', '--blocked', type=str2bool, nargs="?", default=True,
                        help='If true, the matrix has only one block diagonal.')
    parser.add_argument('-i', '--device', type=str, default='gpu', help='Device to use for the MM. Only gpu here.')
    parser.add_argument('-z', '--iterations', type=int, default=1, help='Number of SpMM iterations to run.')
    parser.add_argument('-r', '--ranksperside', type=int, default=3,
                        help='Number of block-rows per side (for synthetic data only)')
    parser.add_argument('-m', '--ba_neighbors', type=int, default=3,
                        help='Number of neighbors per vertex (for synthetic data only)')
    parser.add_argument('-s', '--slim', type=str2bool, nargs="?", default=True,
                        help='Reference rank layout selector; both layouts map to the same GPU kernels.')
    parser.add_argument('-n', '--npy', type=str2bool, nargs="?", default=True,
                        help='If true, the decomposition is loaded from the indices / indptr files.')
    parser.add_argument('--dtype', choices=('float32', 'bfloat16'), default='float32',
                        help='Element type of the feature and result tiles (one GPU for bfloat16); arithmetic is float32.')
    args = vars(parser.parse_args(argv))
    from . import comm as comm_mod
    comm_mod.init_from_env()                    # torchrun --nproc-per-node N: one process per GPU
    if comm_mod.world_comm().Get_rank() == 0:
        print(str(args), flush=True)
    arrow_bench.bench_spmm(args['path'], args['width'], args['features'], args['iterations'], args['blocked'],
                           args['device'], args['ranksperside'], args['ba_neighbors'], None,
                           datatype=args['dtype'], slim=args['slim'], npy_format=args['npy'])


if __name__ == '__main__':
    main()
