/*
 * infer_c.c -- UNet_UAPS inference from plain C: libuaps_b200.so + the CUDA runtime, no Python, no PyTorch.
 *
 *   infer_c PARAMS IN_CHNS C INPUT B H W LOGITS_OUT LABELS_OUT [--bench REPS]
 *
 * PARAMS : the parameter blob, raw little-endian fp32 (uaps_unet_params_count(IN_CHNS, C) values; written e.g. by
 *          uaps_b200.unet.inference_params(model).cpu().numpy().tofile(path));
 * INPUT  : B images [B, IN_CHNS, H, W], raw fp32 NCHW;
 * writes LOGITS_OUT ([B, C, H, W] fp32) and LABELS_OUT ([B, H, W] uint8, argmax of the softmax).
 * --bench REPS: also prints one JSON line with the time of prepare, of a batch-B forward (plain calls and replayed from
 * a CUDA graph; ms per image) and the batch-1 latency of a graph replay of the first image, each the mean over REPS
 * calls timed with CUDA events.
 *
 * Build (from the repository root, after python -m uaps_b200.build):
 *   nvcc -O2 -Wno-deprecated-gpu-targets -I include examples/infer_c.c -L uaps_b200/lib -luaps_b200 \
 *        -Xlinker -rpath,$PWD/uaps_b200/lib -o infer_c
 * (a C file: nvcc hands it to the host compiler and links the CUDA runtime).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "uaps_b200.h"

#define CUDA_OK(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #call, cudaGetErrorString(e_));   \
            exit(1);                                                                               \
        }                                                                                          \
    } while (0)
#define UAPS_OK_(call)                                                                             \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0) {                                                                             \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #call, uaps_error_string(r_));    \
            exit(1);                                                                               \
        }                                                                                          \
    } while (0)

static void* read_file(const char* path, size_t bytes) {
    FILE* f = fopen(path, "rb");
    if (f == NULL) { perror(path); exit(1); }
    void* buf = malloc(bytes);
    if (buf == NULL || fread(buf, 1, bytes, f) != bytes) { fprintf(stderr, "%s: expected %zu bytes\n", path, bytes); exit(1); }
    fclose(f);
    return buf;
}

static void write_file(const char* path, const void* buf, size_t bytes) {
    FILE* f = fopen(path, "wb");
    if (f == NULL || fwrite(buf, 1, bytes, f) != bytes) { perror(path); exit(1); }
    fclose(f);
}

static void* upload(const void* host, size_t bytes, cudaStream_t s) {
    void* dev = NULL;
    CUDA_OK(cudaMalloc(&dev, bytes));
    CUDA_OK(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, s));
    return dev;
}

typedef struct {
    const float* params; void* state; size_t state_bytes; int cin, C;
    const float* x; int B, H, W; void* ws; size_t ws_bytes; float* logits; uint8_t* labels;
    cudaGraphExec_t graph;
} Job;
enum { PREPARE, RUN, REPLAY };

/* mean ms of `reps` calls of one of the three timed bodies */
static float time_ms(const Job* j, int what, int reps, cudaStream_t s) {
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0));
    CUDA_OK(cudaEventCreate(&e1));
    CUDA_OK(cudaEventRecord(e0, s));
    for (int i = 0; i < reps; ++i) {
        if (what == PREPARE)
            UAPS_OK_(uaps_unet_infer_prepare(j->params, j->cin, j->C, j->state, j->state_bytes, s));
        else if (what == RUN)
            UAPS_OK_(uaps_unet_infer_run(j->state, j->state_bytes, j->cin, j->C, j->x, j->B, j->H, j->W, j->ws, j->ws_bytes,
                                         j->logits, j->labels, s));
        else
            CUDA_OK(cudaGraphLaunch(j->graph, s));
    }
    CUDA_OK(cudaEventRecord(e1, s));
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    CUDA_OK(cudaEventDestroy(e0));
    CUDA_OK(cudaEventDestroy(e1));
    return ms / reps;
}

static cudaGraphExec_t capture_run(const Job* j, cudaStream_t s) {
    cudaGraph_t g;
    cudaGraphExec_t ge;
    CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    UAPS_OK_(uaps_unet_infer_run(j->state, j->state_bytes, j->cin, j->C, j->x, j->B, j->H, j->W, j->ws, j->ws_bytes,
                                 j->logits, j->labels, s));
    CUDA_OK(cudaStreamEndCapture(s, &g));
    CUDA_OK(cudaGraphInstantiate(&ge, g, 0));
    CUDA_OK(cudaGraphDestroy(g));
    return ge;
}

int main(int argc, char** argv) {
    if (argc != 10 && !(argc == 12 && strcmp(argv[10], "--bench") == 0)) {
        fprintf(stderr, "usage: %s PARAMS IN_CHNS C INPUT B H W LOGITS_OUT LABELS_OUT [--bench REPS]\n", argv[0]);
        return 2;
    }
    const int cin = atoi(argv[2]), C = atoi(argv[3]), B = atoi(argv[5]), H = atoi(argv[6]), W = atoi(argv[7]);
    const int reps = argc == 12 ? atoi(argv[11]) : 0;
    const size_t n_params = uaps_unet_params_count(cin, C);
    const size_t state_bytes = uaps_unet_infer_state_bytes(cin, C);
    const size_t ws_bytes = uaps_unet_infer_workspace_bytes(cin, C, B, H, W);
    if (n_params == 0 || ws_bytes == 0) {
        fprintf(stderr, "unsupported network or shape (in_chns 1..16, C 2..%d, H and W multiples of 16)\n", UAPS_CMAX);
        return 2;
    }
    const size_t n_x = (size_t)B * cin * H * W, n_logits = (size_t)B * C * H * W, n_pix = (size_t)B * H * W;

    cudaStream_t s;
    CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    void* h_params = read_file(argv[1], n_params * sizeof(float));
    void* h_x = read_file(argv[4], n_x * sizeof(float));
    Job j;
    memset(&j, 0, sizeof j);
    j.params = (const float*)upload(h_params, n_params * sizeof(float), s);
    j.x = (const float*)upload(h_x, n_x * sizeof(float), s);
    j.cin = cin; j.C = C; j.B = B; j.H = H; j.W = W;
    j.state_bytes = state_bytes;
    j.ws_bytes = ws_bytes;
    CUDA_OK(cudaMalloc(&j.state, state_bytes));
    CUDA_OK(cudaMalloc(&j.ws, ws_bytes));
    CUDA_OK(cudaMalloc((void**)&j.logits, n_logits * sizeof(float)));
    CUDA_OK(cudaMalloc((void**)&j.labels, n_pix));

    UAPS_OK_(uaps_unet_infer_prepare(j.params, cin, C, j.state, state_bytes, s));
    UAPS_OK_(uaps_unet_infer_run(j.state, state_bytes, cin, C, j.x, B, H, W, j.ws, ws_bytes, j.logits, j.labels, s));
    float* h_logits = (float*)malloc(n_logits * sizeof(float));
    uint8_t* h_labels = (uint8_t*)malloc(n_pix);
    CUDA_OK(cudaMemcpyAsync(h_logits, j.logits, n_logits * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(h_labels, j.labels, n_pix, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    write_file(argv[8], h_logits, n_logits * sizeof(float));
    write_file(argv[9], h_labels, n_pix);

    if (reps > 0) {
        time_ms(&j, PREPARE, 2, s);                                      /* warm-up */
        const float prepare_ms = time_ms(&j, PREPARE, reps, s);
        time_ms(&j, RUN, 2, s);
        const float run_ms = time_ms(&j, RUN, reps, s);
        j.graph = capture_run(&j, s);
        time_ms(&j, REPLAY, 2, s);
        const float graph_ms = time_ms(&j, REPLAY, reps, s);
        CUDA_OK(cudaGraphExecDestroy(j.graph));
        Job one = j;                                                     /* batch 1: the first image, its own graph */
        one.B = 1;
        one.ws_bytes = uaps_unet_infer_workspace_bytes(cin, C, 1, H, W);
        UAPS_OK_(uaps_unet_infer_run(one.state, state_bytes, cin, C, one.x, 1, H, W, one.ws, one.ws_bytes, one.logits,
                                     one.labels, s));
        one.graph = capture_run(&one, s);
        time_ms(&one, REPLAY, 2 * reps, s);
        const float b1_ms = time_ms(&one, REPLAY, 10 * reps, s);
        CUDA_OK(cudaGraphExecDestroy(one.graph));
        printf("{\"batch\": %d, \"H\": %d, \"W\": %d, \"in_chns\": %d, \"classes\": %d, \"reps\": %d, "
               "\"prepare_ms\": %.5f, \"batch_ms_per_image\": %.6f, \"batch_graph_ms_per_image\": %.6f, "
               "\"batch1_graph_ms\": %.5f}\n",
               B, H, W, cin, C, reps, prepare_ms, run_ms / B, graph_ms / B, b1_ms);
    }

    CUDA_OK(cudaFree((void*)j.params));
    CUDA_OK(cudaFree((void*)j.x));
    CUDA_OK(cudaFree(j.state));
    CUDA_OK(cudaFree(j.ws));
    CUDA_OK(cudaFree(j.logits));
    CUDA_OK(cudaFree(j.labels));
    CUDA_OK(cudaStreamDestroy(s));
    free(h_params); free(h_x); free(h_logits); free(h_labels);
    return 0;
}
