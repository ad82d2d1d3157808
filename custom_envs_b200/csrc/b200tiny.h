// Host-side entry points of the warp-per-env kernel for tiny problems (b200tiny.cu), called from b200env.cu.
// Dev / StepArgs travel as opaque pointers: both translation units include b200env_shared.cuh.
#pragma once

// MultiOptLRs over softmax / linear regression without a hidden layer, at most 8 features, 8 outputs,
// 96 parameters and a minibatch of 32 (BASELINE config 2)
bool b2e_tiny_supported(const void *dev);
// MODE_STEP (auto-reset included) or MODE_RESET over args.e_begin .. e_begin + e_count, one warp per env;
// adam: the AdamArgs of b2e_step_adam (b200adam.cuh), null for every other launch
int b2e_tiny_launch(const void *dev, const void *args, const void *adam, void *stream);
