// spmm_w2.cu — instantiations with 16-byte (double2) B/C accesses.
#include "spmm_launch.cuh"
namespace spmm
{
int launch_rows_w2(const spmm_csr_s *A, int kl, int nv, int np, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s)
{
    return launch_rows_shape<2>(A, kl, nv, np, u, a, tiles, dev, s);
}
int launch_merge_w2(int kl, int nv, int u, const SpmmArgs &a, int tiles, cudaStream_t s)
{
    return launch_merge_shape<2>(kl, nv, u, a, tiles, s);
}
} // namespace spmm
