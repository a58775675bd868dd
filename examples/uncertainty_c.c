/*
 * uncertainty_c.c -- UNet_UAPS ensemble uncertainty inference from plain C: libuaps_b200.so + the CUDA runtime, no
 * Python, no PyTorch.
 *
 *   uncertainty_c PARAMS IN_CHNS C N_AUX INPUT DRAWS B H W LABELS_OUT UNC_OUT IMG_UNC_OUT [--bench REPS]
 *
 * PARAMS : the parameter blob, raw little-endian fp32 (uaps_unet_ensemble_params_count(IN_CHNS, C, N_AUX) values;
 *          written e.g. by uaps_b200.unet.inference_params(model, ensemble=True).cpu().numpy().tofile(path));
 * INPUT  : B images [B, IN_CHNS, H, W], raw fp32 NCHW;
 * DRAWS  : the perturbations' random draws, raw int64 [2, uaps_unet_ensemble_draws_count(N_AUX)] (written e.g. by
 *          model._ensemble_draws(seed).tofile(path)); a service would fill the same buffer from its own generator;
 * writes LABELS_OUT ([B, H, W] uint8, argmax of the decoders' mean softmax), UNC_OUT ([B, H, W] fp32, per-pixel
 * uncertainty) and IMG_UNC_OUT ([B] fp32, per-image mean uncertainty).
 * --bench REPS: also prints one JSON line with the time of prepare, of a batch-B call (plain calls and replayed from a
 * CUDA graph; ms per image) and the batch-1 latency of a graph replay of the first image, each the mean over REPS calls
 * (10 x REPS at batch 1) timed with CUDA events.
 *
 * Build (from the repository root, after python -m uaps_b200.build):
 *   nvcc -O2 -Wno-deprecated-gpu-targets -I include examples/uncertainty_c.c -L uaps_b200/lib -luaps_b200 \
 *        -Xlinker -rpath,$PWD/uaps_b200/lib -o uncertainty_c
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
    const float* params; void* state; size_t state_bytes; int cin, C, n_aux;
    const float* x; int B, H, W; const int64_t* draws; void* ws; size_t ws_bytes;
    uint8_t* labels; float* unc; float* img_unc;
    cudaGraphExec_t graph;
} Job;
enum { PREPARE, RUN, REPLAY };

static int run(const Job* j, cudaStream_t s) {
    return uaps_unet_ensemble_run(j->state, j->state_bytes, j->cin, j->C, j->n_aux, j->x, j->B, j->H, j->W, j->draws, j->ws,
                                  j->ws_bytes, j->labels, j->unc, j->img_unc, NULL, s);
}

/* mean ms of `reps` calls of one of the three timed bodies */
static float time_ms(const Job* j, int what, int reps, cudaStream_t s) {
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0));
    CUDA_OK(cudaEventCreate(&e1));
    CUDA_OK(cudaEventRecord(e0, s));
    for (int i = 0; i < reps; ++i) {
        if (what == PREPARE)
            UAPS_OK_(uaps_unet_ensemble_prepare(j->params, j->cin, j->C, j->n_aux, j->state, j->state_bytes, s));
        else if (what == RUN)
            UAPS_OK_(run(j, s));
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
    UAPS_OK_(run(j, s));
    CUDA_OK(cudaStreamEndCapture(s, &g));
    CUDA_OK(cudaGraphInstantiate(&ge, g, 0));
    CUDA_OK(cudaGraphDestroy(g));
    return ge;
}

int main(int argc, char** argv) {
    if (argc != 13 && !(argc == 15 && strcmp(argv[13], "--bench") == 0)) {
        fprintf(stderr, "usage: %s PARAMS IN_CHNS C N_AUX INPUT DRAWS B H W LABELS_OUT UNC_OUT IMG_UNC_OUT [--bench REPS]\n",
                argv[0]);
        return 2;
    }
    const int cin = atoi(argv[2]), C = atoi(argv[3]), n_aux = atoi(argv[4]);
    const int B = atoi(argv[7]), H = atoi(argv[8]), W = atoi(argv[9]);
    const int reps = argc == 15 ? atoi(argv[14]) : 0;
    const size_t n_params = uaps_unet_ensemble_params_count(cin, C, n_aux);
    const size_t n_draws = 2 * uaps_unet_ensemble_draws_count(n_aux);
    const size_t state_bytes = uaps_unet_ensemble_state_bytes(cin, C, n_aux);
    const size_t ws_bytes = uaps_unet_ensemble_workspace_bytes(cin, C, n_aux, B, H, W);
    if (n_params == 0 || ws_bytes == 0) {
        fprintf(stderr, "unsupported network or shape (in_chns 1..16, C 2..%d, N_AUX 1..%d, H and W multiples of 16)\n",
                UAPS_CMAX, UAPS_KMAX - 1);
        return 2;
    }
    const size_t n_x = (size_t)B * cin * H * W, n_pix = (size_t)B * H * W;

    cudaStream_t s;
    CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    void* h_params = read_file(argv[1], n_params * sizeof(float));
    void* h_x = read_file(argv[5], n_x * sizeof(float));
    void* h_draws = read_file(argv[6], n_draws * sizeof(int64_t));
    Job j;
    memset(&j, 0, sizeof j);
    j.params = (const float*)upload(h_params, n_params * sizeof(float), s);
    j.x = (const float*)upload(h_x, n_x * sizeof(float), s);
    j.draws = (const int64_t*)upload(h_draws, n_draws * sizeof(int64_t), s);
    j.cin = cin; j.C = C; j.n_aux = n_aux; j.B = B; j.H = H; j.W = W;
    j.state_bytes = state_bytes;
    j.ws_bytes = ws_bytes;
    CUDA_OK(cudaMalloc(&j.state, state_bytes));
    CUDA_OK(cudaMalloc(&j.ws, ws_bytes));
    CUDA_OK(cudaMalloc((void**)&j.labels, n_pix));                      /* cudaMalloc: 256-byte aligned */
    CUDA_OK(cudaMalloc((void**)&j.unc, n_pix * sizeof(float)));
    CUDA_OK(cudaMalloc((void**)&j.img_unc, (size_t)B * sizeof(float)));

    UAPS_OK_(uaps_unet_ensemble_prepare(j.params, cin, C, n_aux, j.state, state_bytes, s));
    UAPS_OK_(run(&j, s));
    uint8_t* h_labels = (uint8_t*)malloc(n_pix);
    float* h_unc = (float*)malloc(n_pix * sizeof(float));
    float* h_img = (float*)malloc((size_t)B * sizeof(float));
    CUDA_OK(cudaMemcpyAsync(h_labels, j.labels, n_pix, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(h_unc, j.unc, n_pix * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(h_img, j.img_unc, (size_t)B * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    write_file(argv[10], h_labels, n_pix);
    write_file(argv[11], h_unc, n_pix * sizeof(float));
    write_file(argv[12], h_img, (size_t)B * sizeof(float));

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
        one.ws_bytes = uaps_unet_ensemble_workspace_bytes(cin, C, n_aux, 1, H, W);
        UAPS_OK_(run(&one, s));
        one.graph = capture_run(&one, s);
        time_ms(&one, REPLAY, 2 * reps, s);
        const float b1_ms = time_ms(&one, REPLAY, 10 * reps, s);
        CUDA_OK(cudaGraphExecDestroy(one.graph));
        printf("{\"batch\": %d, \"H\": %d, \"W\": %d, \"in_chns\": %d, \"classes\": %d, \"n_aux\": %d, \"reps\": %d, "
               "\"prepare_ms\": %.5f, \"batch_ms_per_image\": %.6f, \"batch_graph_ms_per_image\": %.6f, "
               "\"batch1_graph_ms\": %.5f}\n",
               B, H, W, cin, C, n_aux, reps, prepare_ms, run_ms / B, graph_ms / B, b1_ms);
    }

    CUDA_OK(cudaFree((void*)j.params));
    CUDA_OK(cudaFree((void*)j.x));
    CUDA_OK(cudaFree((void*)j.draws));
    CUDA_OK(cudaFree(j.state));
    CUDA_OK(cudaFree(j.ws));
    CUDA_OK(cudaFree(j.labels));
    CUDA_OK(cudaFree(j.unc));
    CUDA_OK(cudaFree(j.img_unc));
    CUDA_OK(cudaStreamDestroy(s));
    free(h_params); free(h_x); free(h_draws); free(h_labels); free(h_unc); free(h_img);
    return 0;
}
