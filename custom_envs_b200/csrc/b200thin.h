// Host-side entry points of the shared-memory-resident eval kernel for wide softmax regression (b200thin.cu),
// called from b200env.cu.  Dev / StepArgs travel as opaque pointers: both translation units include b200env_shared.cuh.
#pragma once

// softmax regression, 10 classes, minibatch <= 32, 64 <= features <= 1024 (multiple of 4): BASELINE config 3
bool b2e_thin2_supported(const void *dev);
// shared-memory opt-in; 0 on success
int b2e_thin2_prepare(const void *dev);
// loss + gradient (-> Dev::gnext) of args.e_begin .. e_begin + e_count; second = 1: also the step's scalars
int b2e_thin2_launch(const void *dev, const void *args, int second, int num_sms, void *stream);
