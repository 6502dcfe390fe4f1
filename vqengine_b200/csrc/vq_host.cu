// vq_host.cu — blocking host-buffer entry point for K1: the call an engine integration makes when its
// frame data lives in system memory. Rows are cut into chunks and pipelined over three streams
// (upload | shade | download) so that PCIe traffic in both directions overlaps the kernel; with pinned
// host memory (cudaHostRegister / cudaMallocHost) the copies are truly asynchronous.
#include "vq_common.cuh"

extern "C" int vq_forward_lighting_host(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                                        const VqGBuffer* hgb, const VqEnvironmentMaps* denv, VqImage hout) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("RenderSceneColor");
    VQ_REQUIRE(pf && pv && hgb && denv, "null parameter block");
    VQ_REQUIRE(vq_image_ok(hgb->position_ao) && vq_image_ok(hgb->normal_roughness) && vq_image_ok(hgb->albedo_metalness) && vq_image_ok(hout),
               "bad host image descriptor");
    const int W = hout.width, H = hout.height;
    const bool hasEm = hgb->emissive.ptr != nullptr;
    // every plane is read with cudaMemcpy2D over W x H texels of ITS pitch: a smaller plane or a bad pitch would read past
    // the end of the caller's host memory, so all of this is checked before the first copy is enqueued
    const VqImage* checked[3] = {&hgb->position_ao, &hgb->normal_roughness, &hgb->albedo_metalness};
    for (const VqImage* im : checked)
        VQ_REQUIRE(im->width == W && im->height == H, "every host G-buffer plane must have the output's width and height");
    if (hasEm) VQ_REQUIRE(vq_image_ok(hgb->emissive) && hgb->emissive.width == W && hgb->emissive.height == H,
                          "bad host emissive plane (descriptor, pitch or size)");
    const int planes = hasEm ? 5 : 4;
    const size_t rowBytes = (size_t)W * 16, planeBytes = rowBytes * H;
    VqScratchLock lock(ctx);           // the staging buffer, the three streams and the event ring are the context's
    if (ctx->stage_dev_bytes < planeBytes * planes || !ctx->streams_ready) {
        // (re)size staging: vq_ctx_resize sizes for 4 planes; grow here if an emissive plane is present
        rc = vq_ctx_resize_locked(ctx, W, H); if (rc) return rc;
        if (ctx->stage_dev_bytes < planeBytes * planes) {
            cudaFree(ctx->stage_dev); ctx->stage_dev = nullptr; ctx->stage_dev_bytes = 0;
            if (cudaMalloc(&ctx->stage_dev, planeBytes * planes) != cudaSuccess) { cudaGetLastError(); vq_set_error("staging cudaMalloc failed"); return VQ_ERR_OUT_OF_MEMORY; }
            ctx->stage_dev_bytes = planeBytes * planes;
        }
    }
    char* base = (char*)ctx->stage_dev;
    VqGBuffer dgb;
    dgb.position_ao      = VqImage{base + 0 * planeBytes, W, H, rowBytes};
    dgb.normal_roughness = VqImage{base + 1 * planeBytes, W, H, rowBytes};
    dgb.albedo_metalness = VqImage{base + 2 * planeBytes, W, H, rowBytes};
    VqImage dout         = VqImage{base + 3 * planeBytes, W, H, rowBytes};
    dgb.emissive = hasEm ? VqImage{base + 4 * planeBytes, W, H, rowBytes} : VqImage{nullptr, 0, 0, 0};

    // 8 chunks measured best at 4K (8.16 ms; 16: 8.32, 4: 8.24, 2: 8.71; the link alone moves the 398 MB in 7.19 ms and loses 12 %
    // per direction while both directions are busy: profiles/r02_e2e_link.txt)
    const int chunks = H >= 256 ? 8 : (H >= 16 ? 4 : 1);
    const int rowsPer = (H + chunks - 1) / chunks;
    cudaStream_t sUp = ctx->streams[0], sRun = ctx->streams[1], sDown = ctx->streams[2];
    const VqImage* hp[4] = {&hgb->position_ao, &hgb->normal_roughness, &hgb->albedo_metalness, &hgb->emissive};
    const VqImage* dp[4] = {&dgb.position_ao, &dgb.normal_roughness, &dgb.albedo_metalness, &dgb.emissive};
    for (int c = 0; c < chunks; ++c) {
        const int r0 = c * rowsPer, r1 = (r0 + rowsPer < H) ? r0 + rowsPer : H;
        if (r0 >= r1) break;
        for (int k = 0; k < (hasEm ? 4 : 3); ++k) {
            // tightly packed host rows (the usual case): one linear copy; pitched rows: a 2-D copy
            if (hp[k]->pitch_bytes == rowBytes)
                VQ_CUDA_OK(cudaMemcpyAsync((char*)dp[k]->ptr + (size_t)r0 * rowBytes, (const char*)hp[k]->ptr + (size_t)r0 * rowBytes,
                                           rowBytes * (size_t)(r1 - r0), cudaMemcpyHostToDevice, sUp));
            else
                VQ_CUDA_OK(cudaMemcpy2DAsync((char*)dp[k]->ptr + (size_t)r0 * rowBytes, rowBytes,
                                             (const char*)hp[k]->ptr + (size_t)r0 * hp[k]->pitch_bytes, hp[k]->pitch_bytes,
                                             rowBytes, r1 - r0, cudaMemcpyHostToDevice, sUp));
        }
        VQ_CUDA_OK(cudaEventRecord(ctx->events[2 * c], sUp));
        VQ_CUDA_OK(cudaStreamWaitEvent(sRun, ctx->events[2 * c], 0));
        rc = vq_forward_launch(ctx, pf, pv, &dgb, denv, dout, r0, r1, sRun); if (rc) return rc;
        VQ_CUDA_OK(cudaEventRecord(ctx->events[2 * c + 1], sRun));
        VQ_CUDA_OK(cudaStreamWaitEvent(sDown, ctx->events[2 * c + 1], 0));
        if (hout.pitch_bytes == rowBytes)
            VQ_CUDA_OK(cudaMemcpyAsync((char*)hout.ptr + (size_t)r0 * rowBytes, (const char*)dout.ptr + (size_t)r0 * rowBytes,
                                       rowBytes * (size_t)(r1 - r0), cudaMemcpyDeviceToHost, sDown));
        else
            VQ_CUDA_OK(cudaMemcpy2DAsync((char*)hout.ptr + (size_t)r0 * hout.pitch_bytes, hout.pitch_bytes,
                                         (const char*)dout.ptr + (size_t)r0 * rowBytes, rowBytes,
                                         rowBytes, r1 - r0, cudaMemcpyDeviceToHost, sDown));
    }
    VQ_CUDA_OK(cudaStreamSynchronize(sDown));
    VQ_CUDA_OK(cudaStreamSynchronize(sRun));
    VQ_CUDA_OK(cudaStreamSynchronize(sUp));
    return VQ_OK;
}
