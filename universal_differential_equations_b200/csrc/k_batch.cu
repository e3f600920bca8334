// k_batch.cu -- batched independent trainings of the LV 2 -> 5 -> 5 -> 5 -> 2 UDE (ude_batch.cuh): n_prefix 0, 1, 2 x
// interpolating / discrete adjoint.  The physics constants, loss weights and activation codes of a batch handle live in THIS
// translation unit's constant bank (its own copy of c_consts / c_lossw / c_acts): a batch handle runs concurrently with handles of
// every other family; work of two batch handles with different descriptors on one device must be stream-ordered.
#include "ude_batch.cuh"

namespace b200ude {

template <int NP, bool DISC>
static cudaError_t launch_batch_one(const BatchParams &p, cudaStream_t st)
{
    auto kern = ude_batch_kernel<CfgLV5<NP>, DISC, BATCH_BLOCK>;
    const size_t smem = sizeof(float) * CfgLV5<NP>::P * BATCH_BLOCK;   // < 48 KB: no opt-in attribute needed
    const int grid = (p.M + BATCH_BLOCK - 1) / BATCH_BLOCK;
    kern<<<grid, BATCH_BLOCK, smem, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_batch(int n_prefix, bool discrete, const ConstTables &t, const BatchParams &p, cudaStream_t st)
{
    static SerialCache cache;
    if (!cache.hit(t.serial)) {
        cudaError_t e = cudaMemcpyToSymbolAsync(c_consts, t.consts, sizeof(t.consts), 0, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(c_lossw, t.lossw, sizeof(t.lossw), 0, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(c_acts, t.acts, sizeof(t.acts), 0, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
        cache.set(t.serial);
    }
    switch (n_prefix * 2 + (discrete ? 1 : 0)) {
    case 0: return launch_batch_one<0, false>(p, st);
    case 1: return launch_batch_one<0, true>(p, st);
    case 2: return launch_batch_one<1, false>(p, st);
    case 3: return launch_batch_one<1, true>(p, st);
    case 4: return launch_batch_one<2, false>(p, st);
    default: return launch_batch_one<2, true>(p, st);
    }
}

}  // namespace b200ude
