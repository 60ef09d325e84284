"""Regenerates include/sniper_b200.h from the extern "C" definitions in sniper_b200/csrc/*.cu|cpp plus the
reference citations below (kept here so that the header and the sources cannot drift apart)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DOC = {
    "sniper_last_error": "Thread-local message of the last failing call.  Mirrors MXGetLastError (SNIPER-mxnet/include/mxnet/c_api.h:196-204).",
    "sniper_abi_version": "ABI version of this library (bumped on any signature change).",
    "sniper_multi_proposal_target_workspace_bytes": "Scratch bytes for sniper_multi_proposal_target_fwd: replaces ResourceRequest::kTempSpace of MultiProposalTargetProp (multi_proposal_target-inl.h:143-146).",
    "sniper_generate_anchors": "Host helper, utils::GenerateAnchors (multi_proposal_target.cu:75-114): out[nr*ns,4], ratio-major.",
    "sniper_proposal_decode": "K1: utils::getProps (multi_proposal_target.cu:263-331). Anchor shift + bbox_transform_inv + clip + min-size / valid-range filters -> SoA boxes float4[B*A*H*W], score, area. layout 0 = NCHW (reference), 1 = NHWC (channel strides given).",
    "sniper_multi_proposal_target_fwd": "Drop-in for MultiProposalTargetGPUOp::Forward (multi_proposal_target.cu:362-589; operator surface multi_proposal_target-inl.h:55-177: arguments cls_prob,bbox_pred,im_info,gt_boxes,valid_ranges -> outputs rois,label,bbox_target,bbox_weight). Decode + greedy NMS (reference tie order) + GT append + IoU/label/target assignment, entirely on device: no D2H/H2D, no sync, no allocation. keep_idx/num_kept are optional parity outputs. Backward of the reference operator is a zero fill (cu:591-615) and needs no entry point.",
    "sniper_multi_proposal_workspace_bytes": "Scratch bytes for sniper_multi_proposal_fwd.",
    "sniper_multi_proposal_fwd": "Drop-in for the inference proposal operator MultiProposal (multi_proposal-inl.h:55-167: arguments cls_prob,bbox_pred,im_info -> outputs output(rois),score; CPU op multi_proposal.cc:273-374, GPU-build op multi_proposal.cu:400-631, which is host code with D2H copies). Decode + min-size filter + exact top-pre_nms_top_n selection + greedy NMS on device; flags 1 = the GPU build's anchor-type suppression. Rows after the kept ones: deterministic filler instead of the reference's rand() boxes.",
    "sniper_deform_psroi_fwd": "DeformablePSROIPoolingOp::Forward (contrib/deformable_psroi_pooling-inl.h:84-125, kernel .cu:71-161). top_count optional (hidden output of the reference), sample_idx optional parity output [count, spp^2, 4].",
    "sniper_deform_psroi_fwd_tiled": "DeformablePSROIPoolingOp::Forward for NHWC data, group_size 1 (contrib/deformable_psroi_pooling-inl.h:84-125): chip-tiled kernel, one CTA per (chip, 16 channels) with the feature slice in shared memory; same results as sniper_deform_psroi_fwd. Returns -2 when the shape does not qualify.",
    "sniper_deform_psroi_bwd_tiled_workspace_bytes": "Scratch bytes sniper_deform_psroi_bwd_tiled needs (the operator's kTempSpace request).",
    "sniper_deform_psroi_bwd_tiled": "DeformablePSROIPoolingOp::Backward (-inl.h:127-174, kernel .cu:203-330) for NHWC data, group_size 1: gradient slice accumulated in shared memory (no global atomics), data_diff/trans_diff accumulated into (kAddTo). Returns -2 when the shape does not qualify.",
    "sniper_deform_psroi_bwd": "DeformablePSROIPoolingOp::Backward (contrib/deformable_psroi_pooling-inl.h:127-174, kernel .cu:203-330). data_diff/trans_diff are accumulated into (kAddTo); zero them for kWriteTo.",
    "sniper_psroi_fwd": "PSROIPoolingOp::Forward (contrib/psroi_pooling.cu:51-118). bins optional parity output [count,4] = hstart,hend,wstart,wend.",
    "sniper_psroi_bwd": "PSROIPoolingOp::Backward (contrib/psroi_pooling.cu:146-210); accumulates into data_diff.",
    "sniper_gemm_nt": "C[M,N] = epi(A[M,K] * B[N,K]^T) on tcgen05 (TMEM accumulators, TMA operands). Replaces FullyConnected -> cuBLAS (nn/fully_connected-inl.h) and linalg_gemm (contrib/deformable_convolution-inl.h:148-160). dtype 0 = fp32 storage / TF32 math, 1 = bf16. epi: *scale[n], +bias[n], +residual[m,n], relu; accumulate = red.global.add.",
    "sniper_gemm_plan": "Host-only: the tile width, ring depth, persistent grid and tail split sniper_gemm_nt would choose for a shape (no GPU needed).",
    "sniper_gemm_tail_workspace_bytes": "Size of the caller-owned scratch the tcgen05 kernel's K-slice tail split uses (per device).",
    "sniper_gemm_set_tail_workspace": "Registers that scratch (zero-filled, caller-owned, must outlive later launches); the library itself never allocates device memory.",
    "sniper_conv2d_nhwc": "NHWC implicit-GEMM convolution on tcgen05; also the stride-1/stride-2 data gradient (flipped / parity-split weights, strided output map). Replaces cudnnConvolutionForward / BackwardData (nn/cudnn/cudnn_convolution-inl.h:144,211-266).",
    "sniper_conv2d_wgrad_nhwc": "Weight gradient dW[Cout, taps*Cin] += dY^T * im2col(X) on tcgen05 with MN-major operands and split-K. Replaces cudnnConvolutionBackwardFilter (nn/cudnn/cudnn_convolution-inl.h:211-266).",
    "sniper_affine_act": "y = act(x*scale[c] + shift[c]) on [M,C] rows (BatchNorm apply + Activation; nn/batch_norm.cu:658-700); relu 0 = none, 1 = ReLU, 2 = clip(y, 0, 6).",
    "sniper_bn_stats": "Train-mode BatchNorm statistics -> mean, invstd, scale, shift and moving statistics (cuDNN convention, nn/cudnn/cudnn_batch_norm-inl.h).",
    "sniper_bn_apply_train": "BatchNorm(train) + Activation in one launch when the input statistics were accumulated by the producing conv's epilogue: finalisation (mean / invstd / scale / shift / moving statistics, nn/batch_norm.cu:658-700 semantics) folded into the apply pass.",
    "sniper_bn_frozen": "use_global_stats BatchNorm: scale/shift from the moving statistics (nn/batch_norm.cu:671-674 path).",
    "sniper_bn_relu_bwd": "Backward of relu(bn_train(x)): dx (+add), dgamma +=, dbeta +=.",
    "sniper_bn_act_bwd": "Backward of act(bn_train(x)) with act 1 = ReLU (Activation), 2 = clip(y, 0, 6) (mx.sym.clip: relu6 of symbols/faster/mobilenetv2_e2e.py:18-19, gradient mask of tensor/matrix_op-inl.h:1319-1332), 3 = none (linear bottleneck): dx (+add), dgamma +=, dbeta +=.",
    "sniper_affine_relu_bwd": "Backward of relu?(x*scale+shift) for frozen BN.",
    "sniper_depthwise3x3_fwd": "Depthwise 3x3 convolution, pad 1, stride 1|2, NHWC, weights [9,C] fp32: Convolution(num_group = num_filter = C) of mobilenetv2_e2e.py:58-66 (src/operator/nn/depthwise_convolution-inl.h DepthwiseConvolutionOp::Forward).",
    "sniper_depthwise3x3_dgrad": "Data gradient of the depthwise convolution (depthwise_convolution-inl.h Backward, DepthwiseConv2dBackwardDataGpu), gather form.",
    "sniper_depthwise3x3_wgrad": "Weight gradient of the depthwise convolution (DepthwiseConv2dBackwardFilterGpu): dw[9,C] += per-channel correlation of dy with the shifted input.",
    "sniper_im2col3x3s2_nchw": "im2col of MobileNetV2's first layer (3x3 / stride 2 / pad 1 over the 3-channel fp32 NCHW `data`, mobilenetv2_e2e.py:204-212) so that it runs on the tcgen05 GEMM; K order (kh, kw, ci), zero-padded to Kp.",
    "sniper_add_rows": "out = a + b on [M,C] rows: elemwise_add of the inverted-residual shortcut (mobilenetv2_e2e.py:22-24).",
    "sniper_relu_bwd": "dx = dy * (y > 0).",
    "sniper_maxpool3x3s2_nhwc": "Pooling max 3x3 stride 2 pad 1 (resnet_mx_101_e2e.py:409; nn/pool.cuh).",
    "sniper_stem_im2col": "im2col of bn_data(x) for conv0 (resnet_mx_101_e2e.py:402-404) so that the 7x7 stem runs on the tcgen05 kernel (sniper_gemm_nt with bn0 + ReLU as epilogue).",
    "sniper_stem_conv": "bn_data -> conv0 7x7/2 -> bn0 -> relu (resnet_mx_101_e2e.py:402-408), NCHW in, NHWC out.",
    "sniper_weight_transpose": "wt[ci, j, co] = w[co, sel[j], ci]: operand layout for data gradients.",
    "sniper_weight_transpose_batched": "Every sniper_weight_transpose of a training step in one launch (device job table).",
    "sniper_bn_param_grad_batched": "dgamma/dbeta of every BatchNorm in one launch (second half of sniper_bn_relu_bwd when it is called with dgamma = dbeta = NULL).",
    "sniper_colsum": "out[c] += sum_m x[m,c] (bias gradients; cudnnConvolutionBackwardBias).",
    "sniper_sgd_mom": "SGDMomKernel (optimizer_op-inl.h:279-300) on one flat buffer.",
    "sniper_sgd_mom_dev": "SGDMomKernel / MP_SGDMomKernel (optimizer_op-inl.h:279-300, 377-404) with lr and wd read from device memory, so that a captured CUDA graph follows WarmupMultiBatchScheduler (lib/train_utils/lr_scheduler.py:43-66); optional bf16 weight shadow = multi_precision.",
    "sniper_count_valid": "Device-side replacement of SoftmaxOutput's host valid count (softmax_output-inl.h:184-195).",
    "sniper_rpn_softmax_loss": "SoftmaxOutput(multi_output, use_ignore, normalization=valid) for the RPN (softmax_output-inl.h:108-132, 162-206): prob + gradient in one pass.",
    "sniper_rpn_smooth_l1_loss": "weight * smooth_l1(pred - target) + MakeLoss gradient for the RPN (mshadow_op.h:642-678; resnet_mx_101_e2e.py:330-334).",
    "sniper_softmax_ce": "SoftmaxOutput(normalization=valid, use_ignore) flat form (softmax_output-inl.h:207-263).",
    "sniper_smooth_l1_loss": "weight * smooth_l1(pred - target) + MakeLoss gradient (resnet_mx_101_e2e.py:318-319).",
    "sniper_focus_head": "AutoFocus FocusPixel head: conv_new_out (1x1, 256 -> 2) + SoftmaxOutput(multi_output, normalization=valid, use_ignore, ignore_label=-1) (resnet_mx_101_e2e.py:264-267, 313-315; softmax_output-inl.h:162-206, 225-257) + its whole backward (dx3 with conv_new_3's ReLU mask, dW +=, db +=) in one pass; log-loss sum, correct count and valid count of AutoFocusLogLoss / AutoFocusAcc (lib/train_utils/metric.py:50-94) accumulated on the device.",
    "sniper_deform_im2col": "deformable_im2col (contrib/nn/deformable_im2col.cuh:216-263), NHWC, whole batch.",
    "sniper_deform_col2im": "deformable_col2im + deformable_col2im_coord (contrib/nn/deformable_im2col.cuh:317-360, 419-480).",
    "sniper_anchor_target": "RPN anchor matching of anchor_worker.worker (lib/data_utils/data_workers.py:164-371) on device.",
    "sniper_soft_nms_batched": "cpu_soft_nms (lib/nms/cpu_nms.pyx:17-110; Gaussian / linear / hard) for every (image, class) problem of an inference scale in ONE launch: replaces the Pool(32) of nms_worker processes in Tester.aggregate (lib/inference.py:152-200).",
    "sniper_chip_input": "GPU input stage: im_worker.worker (lib/data_utils/data_workers.py:80-121) -- flip, cv2-style 8-bit bilinear resize by the chip scale, zero padding to crop_size, BGR->RGB minus PIXEL_MEANS -- from uint8 source rectangles to the fp32 NCHW `data` tensor of MNIteratorE2E (lib/iterators/MNIteratorE2E.py:194-199).",
    "sniper_chip_input_hw": "The same with a rectangular canvas: im_worker.worker_autofocus (lib/data_utils/data_workers.py:51-78) + the batch padding of MNIteratorTestAutoFocus._get_batch (lib/iterators/MNIteratorTestAutoFocus.py:36-78).",
    "sniper_anchor_subsample": "The npr.choice subsampling of anchor_worker.worker (data_workers.py:326-338) on device: <= num_fg positives, <= batch_size - #positives negatives per chip, the rest -> -1 (counter-based hash instead of numpy's RNG).",
    "sniper_focus_label": "FocusPixel labels of AutoFocus training: gen_mask of anchor_worker.worker (lib/data_utils/data_workers.py:165-192, called at :220-222) on device, one thread per label cell, boxes in GT order (last writer wins) -> scale_label [B, H*W] of MNIteratorE2E (lib/iterators/MNIteratorE2E.py:182-197).",
    "sniper_chips_generate": "chips::cgenerate (lib/chips/cchips.cpp:54-177): host-side chip sampling, same rand() stream.",
    "sniper_cpu_nms": "cpu_nms (lib/nms/cpu_nms.pyx:112-163), host.",
    "sniper_cpu_soft_nms": "cpu_soft_nms (lib/nms/cpu_nms.pyx:17-110), host, in place.",
    "sniper_bbox_overlaps": "bbox_overlaps_cython / ignore_overlaps_cython (lib/bbox/bbox.pyx:17-95), host, float64.",
    "sniper_nms_gpu": "Batched hard NMS on device for per-scale inference NMS (lib/nms/nms_kernel.cu:34-144 replacement).",
}


def signatures():
    out = []
    for f in sorted(glob.glob(os.path.join(ROOT, "sniper_b200", "csrc", "*.cu")) +
                    glob.glob(os.path.join(ROOT, "sniper_b200", "csrc", "*.cpp"))):
        s = open(f).read()
        for m in re.finditer(r'\n((?:int|size_t|const char\*)\s+(sniper_\w+)\s*\(([^)]*)\))\s*\{', s):
            out.append((os.path.basename(f), m.group(2), re.sub(r'\s+', ' ', re.sub(r'/\*.*?\*/', '', m.group(1)))))
    return out


def main():
    lines = ["/* sniper_b200 C-ABI -- generated by tools/gen_header.py from sniper_b200/csrc (do not edit by hand).",
             " *",
             " * Drop-in boundary of the SNIPER 512x512-chip training path: every entry point is extern \"C\", takes",
             " * plain pointers and sizes (device pointers unless a comment says host), a cudaStream_t passed as",
             " * void*, returns 0 on success and -1 on failure with the message in sniper_last_error().",
             " * No entry point allocates device memory or synchronises.  Reference file:line each one replaces",
             " * is cited above its prototype (paths relative to the reference repo; SNIPER-mxnet/src/operator/ is",
             " * implied for operator sources).",
             " */",
             "#ifndef SNIPER_B200_H_", "#define SNIPER_B200_H_", "#include <stddef.h>", "#include <stdint.h>", "",
             "#ifdef __cplusplus", 'extern "C" {', "#endif", ""]
    for f, name, sig in signatures():
        doc = DOC.get(name, "")
        lines.append("/* [%s] %s */" % (f, doc))
        lines.append(sig + ";")
        lines.append("")
    lines += ["#ifdef __cplusplus", "}", "#endif", "#endif  /* SNIPER_B200_H_ */", ""]
    os.makedirs(os.path.join(ROOT, "include"), exist_ok=True)
    open(os.path.join(ROOT, "include", "sniper_b200.h"), "w").write("\n".join(lines))


if __name__ == "__main__":
    main()
