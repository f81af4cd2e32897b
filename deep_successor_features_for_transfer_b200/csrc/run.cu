// sfgpi_run: executes a pre-built list of hot-path commands back to back on one stream from C, so that one train step costs the
// host ONE foreign call instead of a dozen (the reference's update_successor is ~60 eager torch ops; here the Python side
// only patches six input pointers and calls this).  The list is plain data: it can be replayed every step.
#include "common.cuh"

using namespace sfgpi;

extern "C" int sfgpi_run(const sfgpi_cmd *cmds, int32_t n, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < n; ++i) {
        const sfgpi_cmd &c = cmds[i];
        int rc = SFGPI_OK;
        switch (c.op) {
            case SFGPI_OP_NOP:
                break;
            case SFGPI_OP_EVENT:
                if (cudaEventRecord(reinterpret_cast<cudaEvent_t>(c.p[0]), st) != cudaSuccess) rc = check_launch("sfgpi_run(event)");
                break;
            case SFGPI_OP_H2D:
                if (cudaMemcpyAsync(c.p[0], c.p[1], (size_t)c.i[0], cudaMemcpyHostToDevice, st) != cudaSuccess) rc = check_launch("sfgpi_run(h2d)");
                break;
            case SFGPI_OP_D2H:
                if (cudaMemcpyAsync(c.p[0], c.p[1], (size_t)c.i[0], cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = check_launch("sfgpi_run(d2h)");
                break;
            case SFGPI_OP_D2D:
                if (cudaMemcpyAsync(c.p[0], c.p[1], (size_t)c.i[0], cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = check_launch("sfgpi_run(d2d)");
                break;
            case SFGPI_OP_KEYS_FILL:
                rc = sfgpi_keys_fill(reinterpret_cast<int64_t *>(c.p[0]), c.i[0], stream);
                break;
            case SFGPI_OP_PACK_BF16:
                rc = sfgpi_pack_bf16(reinterpret_cast<const sfgpi_net_desc *>(c.p[0]), reinterpret_cast<const float *>(c.p[1]),
                                     (int32_t)c.i[0], (int32_t)c.i[1], c.p[2], stream);
                break;
            case SFGPI_OP_FOLD_GPI:
                rc = sfgpi_fold_gpi(reinterpret_cast<const sfgpi_net_desc *>(c.p[0]), reinterpret_cast<const float *>(c.p[1]),
                                    (int32_t)c.i[0], (int32_t)c.i[1], reinterpret_cast<const float *>(c.p[2]), (int32_t)c.i[2],
                                    (int32_t)c.i[3], c.p[3], reinterpret_cast<float *>(c.p[4]), stream);
                break;
            case SFGPI_OP_FORWARD:
                rc = sfgpi_mlp_forward(reinterpret_cast<const sfgpi_forward_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_FORWARD_TC_JOBS:
                rc = sfgpi_mlp_forward_tc_jobs(reinterpret_cast<const sfgpi_forward_tc_job *>(c.p[0]), (int32_t)c.i[0], stream);
                break;
            case SFGPI_OP_TD:
                rc = sfgpi_td_step(reinterpret_cast<const sfgpi_td_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_BACKWARD:
                rc = sfgpi_mlp_backward(reinterpret_cast<const sfgpi_backward_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_BACKWARD_TC:
                rc = sfgpi_mlp_backward_tc(reinterpret_cast<const sfgpi_backward_tc_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_ADAM:
                rc = sfgpi_adam_step(reinterpret_cast<const sfgpi_adam_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_STEP_PREP:
                rc = sfgpi_step_prep(reinterpret_cast<const sfgpi_step_prep_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_PACK_F32:
                rc = sfgpi_pack_f32(reinterpret_cast<const sfgpi_net_desc *>(c.p[0]), reinterpret_cast<const float *>(c.p[1]), (int32_t)c.i[0],
                                    (int32_t)c.i[1], (int32_t)c.i[2], (int32_t)c.i[3], reinterpret_cast<float *>(c.p[2]),
                                    reinterpret_cast<float *>(c.p[3]), reinterpret_cast<float *>(c.p[4]), stream);
                break;
            case SFGPI_OP_FOLD_GPI_F32:
                rc = sfgpi_fold_gpi_f32(reinterpret_cast<const sfgpi_net_desc *>(c.p[0]), reinterpret_cast<const float *>(c.p[1]), (int32_t)c.i[0],
                                        (int32_t)c.i[1], reinterpret_cast<const float *>(c.p[2]), (int32_t)(c.i[2] & 0x7fffffff),
                                        (int32_t)((c.i[2] >> 31) & 1), (int32_t)c.i[3], reinterpret_cast<float *>(c.p[3]),
                                        reinterpret_cast<float *>(c.p[4]), stream);
                break;
            case SFGPI_OP_FORWARD_STREAM:
                rc = sfgpi_mlp_forward_stream(reinterpret_cast<const sfgpi_forward_tc_job *>(c.p[0]), (int32_t)c.i[0], (int32_t)c.i[1], stream);
                break;
            case SFGPI_OP_BACKWARD_STREAM:
                rc = sfgpi_mlp_backward_stream(reinterpret_cast<const sfgpi_backward_stream_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_KEYS_DECODE:
                rc = sfgpi_keys_decode(reinterpret_cast<const int64_t *>(c.p[0]), c.i[0], reinterpret_cast<int64_t *>(c.p[1]),
                                       reinterpret_cast<float *>(c.p[2]), stream);
                break;
            case SFGPI_OP_PEER_KEYS:
                rc = sfgpi_peer_reduce_keys(reinterpret_cast<const sfgpi_peer_keys_args *>(c.p[0]), stream);
                break;
            case SFGPI_OP_SHARD_PACK:
                rc = sfgpi_shard_pack(reinterpret_cast<const float *>(c.p[0]), (int32_t)c.i[0], reinterpret_cast<const float *>(c.p[1]),
                                      reinterpret_cast<const float *>(c.p[2]), (int32_t)c.i[1], reinterpret_cast<float *>(c.p[3]), stream);
                break;
            case SFGPI_OP_PEER_UNPACK:
                rc = sfgpi_peer_unpack(reinterpret_cast<const sfgpi_peer_unpack_args *>(c.p[0]), stream);
                break;
            default:
                set_error("sfgpi_run: unknown op %d at command %d", c.op, i);
                return SFGPI_E_INVALID;
        }
        if (rc != SFGPI_OK) return rc;
    }
    return SFGPI_OK;
}
