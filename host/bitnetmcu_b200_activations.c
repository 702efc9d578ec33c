/*
 * bitnetmcu_b200_activations.c -- per-layer activations of the test digits, for comparing a port layer by layer.
 *
 * The reference's BitMnistInference carries commented-out `printf("L1 activations:  \n"); printactivations(layer_in, ...)` lines after
 * each hidden layer (BitNetMCU_MNIST_dll.c:102-109): what an MCU build prints over its UART.  This program prints the same for every
 * activation tap of the model (include/bitnetmcu_b200.h section 7) and every digit of a BitNetMCU_MNIST_test_data.h, followed by the
 * "label: / predicted:" line of BitNetMCU_MNIST_test.c.  Tap t is printed as "L<t+1>": for FC models the hidden layers L1, L2, ...;
 * for CNN models L1 is the features after the front-end's ReLUNorm (dll.c:80) and the hidden FC rows follow.
 * Build the shim (host/bitnetmcu_b200_dll.c, which exports printactivations) first, then link this program against it:
 *     cc -Iinclude -I<dir with BitNetMCU_model.h and BitNetMCU_MNIST_test_data.h> host/bitnetmcu_b200_activations.c Bitnet_inf.dll \
 *        -Lbitnetmcu_b200 -lbitnetmcu_b200 -Wl,-rpath,<abs path of bitnetmcu_b200> -Wl,-rpath,<abs dir of Bitnet_inf.dll>
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "BitNetMCU_MNIST_test_data.h"
#include "BitNetMCU_model.h"
#include "bitnetmcu_b200.h"
#include "bitnetmcu_b200_model.h"

void printactivations(uint8_t *activations, int32_t n_activations);

int main(void)
{
    int8_t *inputs[] = {input_data_0, input_data_1, input_data_2, input_data_3, input_data_4,
                        input_data_5, input_data_6, input_data_7, input_data_8, input_data_9};
    uint8_t labels[] = {label_0, label_1, label_2, label_3, label_4, label_5, label_6, label_7, label_8, label_9};
    enum { N = 10 };
    static const bnm_layer layers[] = { BNM_MODEL_LAYERS };
    const char *dev = getenv("BNM_DEVICE");
    bnm_model *m = NULL;
    int rc = bnm_model_create(BNM_MODEL_CLASS, layers, (uint32_t)(sizeof layers / sizeof layers[0]), 256, dev ? atoi(dev) : 0, &m);
    if (rc != 0) {
        fprintf(stderr, "bitnetmcu_b200: cannot create the model (rc=%d): %s\n", rc, bnm_last_error());
        return 1;
    }
    int8_t images[N * 256];
    for (int i = 0; i < N; i++) memcpy(images + i * 256, inputs[i], 256);
    const uint32_t n_taps = bnm_model_n_taps(m);
    bnm_taps taps;
    memset(&taps, 0, sizeof taps);
    for (uint32_t t = 0; t < n_taps; t++) taps.act[t] = malloc((size_t)N * bnm_model_tap_stride(m, t));
    int32_t logits[N * BNM_MODEL_N_CLASSES];
    uint32_t predicted[N];
    rc = bnm_infer_batch_taps(m, images, N, logits, predicted, &taps);
    if (rc != 0) {
        fprintf(stderr, "bitnetmcu_b200: inference failed (rc=%d): %s\n", rc, bnm_last_error());
        return 1;
    }
    for (int i = 0; i < N; i++) {
        for (uint32_t t = 0; t < n_taps; t++) {
            printf("L%u activations:  \n", t + 1);
            printactivations((uint8_t *)taps.act[t] + (size_t)i * bnm_model_tap_stride(m, t), (int32_t)bnm_model_tap_width(m, t));
        }
        printf("label: %d predicted: %d\n", labels[i], (int)predicted[i]);
    }
    for (uint32_t t = 0; t < n_taps; t++) free(taps.act[t]);
    bnm_model_destroy(m);
    return 0;
}
