/*
 * reference_result.c -- runs the reference's own attention() (oracle/_ref/libattention_mpi.so, attention-mpi.c compiled
 * unmodified) on a data file in the reference's format with MPI_SHIM_NP ranks and writes rank 0's result: m*dv fp64,
 * row-major.  The reference's program only prints whether its result passed its own check; make_golden.py keeps the
 * result itself so that the tests can compare with it where the reference is not available.
 *
 *   reference_result <data file> <result file>
 */
#include <stdio.h>
#include <stdlib.h>

#include "mpi.h"

void attention(double* Q, double* K, double* V, double* result, int m, int n, int dk, int dv, int mpi_rank, int mpi_size);

static double* read_doubles(FILE* f, size_t count)
{
    double* p = (double*)malloc((count ? count : 1) * sizeof(double));
    if (!p || fread(p, sizeof(double), count, f) != count) {
        fprintf(stderr, "reference_result: short data file\n");
        exit(1);
    }
    return p;
}

int main(int argc, char** argv)
{
    if (argc != 3) {
        fprintf(stderr, "usage: %s <data file> <result file>\n", argv[0]);
        return 1;
    }
    int rank, size, dims[4] = {0, 0, 0, 0};   /* m, n, dk, dv: read on rank 0, broadcast inside attention() */
    double *Q = NULL, *K = NULL, *V = NULL, *R = NULL;
    MPI_Init(&argc, &argv);
    MPI_Comm_rank(MPI_COMM_WORLD, &rank);
    MPI_Comm_size(MPI_COMM_WORLD, &size);
    if (rank == 0) {
        FILE* f = fopen(argv[1], "rb");
        if (!f || fread(dims, sizeof(int), 4, f) != 4) {
            fprintf(stderr, "reference_result: cannot read %s\n", argv[1]);
            return 1;
        }
        Q = read_doubles(f, (size_t)dims[0] * dims[2]);
        K = read_doubles(f, (size_t)dims[1] * dims[2]);
        V = read_doubles(f, (size_t)dims[1] * dims[3]);
        fclose(f);
        R = (double*)calloc((size_t)dims[0] * dims[3] + 1, sizeof(double));
    }
    attention(Q, K, V, R, dims[0], dims[1], dims[2], dims[3], rank, size);
    if (rank == 0) {
        FILE* f = fopen(argv[2], "wb");
        size_t count = (size_t)dims[0] * dims[3];
        if (!f || fwrite(R, sizeof(double), count, f) != count || fclose(f) != 0) {
            fprintf(stderr, "reference_result: cannot write %s\n", argv[2]);
            return 1;
        }
    }
    MPI_Finalize();
    free(Q);
    free(K);
    free(V);
    free(R);
    return 0;
}
