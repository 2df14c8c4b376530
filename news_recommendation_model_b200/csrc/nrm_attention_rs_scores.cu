// The score-exporting instantiations of the row-stacked attention forward (nrm_forward_scores): the kernel body of
// nrm_attention_rs.cu with kScores = true, in a translation unit of its own so that the module holding the kernels nrm_forward
// launches is compiled exactly as without them.
#define NRM_RS_SCORES_TU
#include "nrm_attention_rs.cu"
