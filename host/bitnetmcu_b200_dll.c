/*
 * bitnetmcu_b200_dll.c -- plain-C drop-in for /root/reference/BitNetMCU_MNIST_dll.c.
 *
 * Build exactly like the reference's Makefile:5-6, plus the engine library:
 *     cc -fPIC -shared -o Bitnet_inf.dll -D_DLL -I<dir of BitNetMCU_model.h> -Iinclude host/bitnetmcu_b200_dll.c \
 *        -Lbitnetmcu_b200 -lbitnetmcu_b200 -Wl,-rpath,<abs path of bitnetmcu_b200>
 * Exports the reference's `uint32_t Inference(int8_t *input)` (dll.c:24-26) -- test_inference.py:134-150 loads it
 * unchanged -- plus the batched `InferenceBatch` the reference lacks.  All compute runs on the GPU through the C ABI;
 * there is no CPU path: a missing CUDA device aborts with a message.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "BitNetMCU_model.h"
#include "bitnetmcu_b200.h"
#include "bitnetmcu_b200_model.h"

#ifdef _WIN64
#define EXPORT __declspec(dllexport)
#else
#define EXPORT __attribute__((visibility("default")))
#endif

static bnm_model *g_model;

static bnm_model *model(void)
{
    if (!g_model) {
        static const bnm_layer layers[] = { BNM_MODEL_LAYERS };
        const char *dev = getenv("BNM_DEVICE");
        int rc = bnm_model_create(BNM_MODEL_CLASS, layers, (uint32_t)(sizeof layers / sizeof layers[0]), 256,
                                  dev ? atoi(dev) : 0, &g_model);
        if (rc != 0) {
            fprintf(stderr, "bitnetmcu_b200: cannot create the model (rc=%d): %s\n", rc, bnm_last_error());
            abort();
        }
    }
    return g_model;
}

/* BitMnistInference, dll.c:48-121: one 16x16 int8 image in, predicted class out */
uint32_t BitMnistInference(int8_t *input)
{
    int32_t logits[BNM_MODEL_N_CLASSES];
    uint32_t label = 255;
    if (bnm_infer_batch(model(), input, 1, logits, &label) != 0) {
        fprintf(stderr, "bitnetmcu_b200: inference failed: %s\n", bnm_last_error());
        abort();
    }
    return label;
}

EXPORT uint32_t Inference(int8_t *input) { return BitMnistInference(input); }

/* n images int8 [n][256] -> int32 logits [n][n_classes] + uint32 labels [n] (NULL allowed); 0 on success */
EXPORT int InferenceBatch(const int8_t *images, size_t n, int32_t *logits, uint32_t *labels)
{
    return bnm_infer_batch(model(), images, n, logits, labels);
}

EXPORT uint32_t InferenceNumClasses(void) { return BNM_MODEL_N_CLASSES; }
EXPORT const char *InferenceLastError(void) { return bnm_last_error(); }

/* dll.c:29-37: one activation row as the firmware's UART dump prints it -- "%d, " per value, a line break after every 16 */
EXPORT void printactivations(uint8_t *activations, int32_t n_activations)
{
    for (int32_t i = 0; i < n_activations; i++)
        printf((i % 16 == 15) ? "%d, \n" : "%d, ", activations[i]);
}
