/* The drop-in boundary must be consumable from plain C (cgo / JNI / ctypes-style bindings):
 * this translation unit includes the header as C99 with -Wall -Wextra -pedantic -Werror and
 * takes the address of every entry point. */
#include "spev_b200.h"

#define USE(f) ((void)(f))
int spev_c99_probe(void) {
    spev_tile t; spev_batch b;
    USE(spev_abi_version); USE(spev_last_error); USE(spev_tile_frames); USE(spev_tile_chunks);
    USE(spev_create); USE(spev_destroy); USE(spev_get_mel_basis); USE(spev_get_mel_pinv); USE(spev_get_window);
    USE(spev_host_mel_basis); USE(spev_host_pinv); USE(spev_plan_frame_tiles); USE(spev_plan_chunk_tiles);
    USE(spev_logmel); USE(spev_stft_power); USE(spev_mel_project); USE(spev_mel_to_mag); USE(spev_set_tensor_core);
    USE(spev_istft); USE(spev_stft); USE(spev_gl_phase_update); USE(spev_griffinlim_workspace_bytes);
    USE(spev_griffinlim); USE(spev_lr_plan); USE(spev_lr_expand); USE(spev_lr_expand_fused);
    USE(spev_duration_rule); USE(spev_bucketize_embed); USE(spev_frame_features); USE(spev_segment_pool); USE(spev_segment_pool_log); USE(spev_pcm16_to_f32); USE(spev_collate); USE(spev_variance_fuse);
    USE(spev_pyin_create); USE(spev_pyin_destroy); USE(spev_pyin_info); USE(spev_pyin_host_tables);
    USE(spev_pyin_cmnd); USE(spev_pyin_observe); USE(spev_pyin_decode_workspace_bytes); USE(spev_pyin_decode); USE(spev_pitch_pool);
    USE(spev_lr_expand_backward); USE(spev_copy_segments_piece_bytes); USE(spev_copy_segments); USE(spev_set_sm_limit); USE(spev_nnls_objective); USE(spev_transpose_batched); USE(spev_variance_fuse_backward_workspace_bytes); USE(spev_variance_fuse_backward);
    t.n = 0; b.n_items = 0;
    return (int)sizeof(spev_tile) + t.n + b.n_items;   /* 48 */
}
