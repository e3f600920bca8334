// k_lv5.cu -- kernels of the reference-shaped LV UDE: 2 -> 5 -> 5 -> 5 -> 2 chain with per-layer
// activations (rbf / tanh) and 0, 1 or 2 trainable linear rates in front of the chain parameters
// (LotkaVolterra/scenario_1.jl:62-73, scenario_2.jl:79-98, hudson_bay.jl:77-91).
#include <type_traits>

#include "ude_adjoint.cuh"

namespace b200ude {

int adj_grid_lv5(int N) { return (N + ADJ_BLOCK_LANE - 1) / ADJ_BLOCK_LANE; }

cudaError_t launch_fwd_lv5(int n_prefix, const Variant &, const ConstTables &t, const FwdParams &p, cudaStream_t st)
{
    cudaError_t e = upload_tables(t, st);
    if (e != cudaSuccess) return e;
    switch (n_prefix) {
    case 0: return launch_forward<CfgLV5<0>, 1, 0, WConst, 4>(p, st);
    case 1: return launch_forward<CfgLV5<1>, 1, 0, WConst, 4>(p, st);
    default: return launch_forward<CfgLV5<2>, 1, 0, WConst, 4>(p, st);
    }
}

template <int NP, bool DISC>
static cudaError_t launch_one(const AdjParams &p, int grid, cudaStream_t st)
{
    auto kern = ude_adjoint_lane_kernel<CfgLV5<NP>, 0, WConst, ADJ_BLOCK_LANE, 1, DISC>;
    const size_t smem = sizeof(float) * (CfgLV5<NP>::P + 1);
    kern<<<grid, ADJ_BLOCK_LANE, smem, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_adj_lv5(int n_prefix, const Variant &v, const ConstTables &t, const AdjParams &p, cudaStream_t st, int *grid_out)
{
    cudaError_t e = upload_tables(t, st);
    if (e != cudaSuccess) return e;
    const int grid = adj_grid_lv5(p.N);
    *grid_out = grid;
    if (v.discrete) {   // exact gradient of the discrete scheme (ForwardDiffSensitivity's result)
        switch (n_prefix) {
        case 0: return launch_one<0, true>(p, grid, st);
        case 1: return launch_one<1, true>(p, grid, st);
        default: return launch_one<2, true>(p, grid, st);
        }
    }
    switch (n_prefix) {
    case 0: return launch_one<0, false>(p, grid, st);
    case 1: return launch_one<1, false>(p, grid, st);
    default: return launch_one<2, false>(p, grid, st);
    }
}

}  // namespace b200ude
