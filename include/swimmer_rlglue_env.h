/*
 * RL-Glue environment plugin symbols exported by libswimmer_ars.so -- the drop-in for the five
 * functions of rlglue/environment/SwimmerEnvironment.h:38-42 (reference), implemented in
 * csrc/rlglue_env_shim.cu on top of swm_step_batched(variant = SWM_DYN_RLGLUE, B = 1).
 * Ownership and message strings follow SwimmerEnvironment.cpp:14-97.
 */
#ifndef SWIMMER_RLGLUE_ENV_H
#define SWIMMER_RLGLUE_ENV_H

#include "rlglue_types.h"
#include "swimmer_ars.h"

#ifdef __cplusplus
extern "C" {
#endif

SWM_API const char* env_init(void);                                      /* cpp:14-33 */
SWM_API const observation_t* env_start(void);                            /* cpp:35-51 */
SWM_API const reward_observation_terminal_t* env_step(const action_t*);  /* cpp:53-68 */
SWM_API void env_cleanup(void);                                          /* cpp:70-74 */
/* cpp:76-97.  "set parameters [path]" keeps the previous n_seg, and says so in the returned message, when the
 * file's n_seg is not an integer in SWM_MIN_SEGMENTS..SWM_MAX_SEGMENTS, or differs from the n_seg of an
 * env_init not yet followed by env_cleanup (the observation and staging buffers are sized for that chain);
 * the file's other parameters still apply. */
SWM_API const char* env_message(const char* message);

/* Sets the model without a parameter file (the reference only has file-scope globals, cpp:3-9).
 * SWM_ERR_BAD_ARG, and nothing changes, for n outside SWM_MIN_SEGMENTS..SWM_MAX_SEGMENTS or a changed n
 * between env_init and env_cleanup. */
SWM_API int swm_rlglue_set_params(const swm_params_t* params);

#ifdef __cplusplus
}
#endif
#endif
