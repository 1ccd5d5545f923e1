// Host check of lz_logf_exact (lightzero_b200/csrc/lz_exact_math.h) against libm logf, the function the Gumbel
// tree's softmax calls.  usage: check_logf <stride> [all]
//   default: every float in [1, 64] with the given stride (a softmax sum over n <= 64 children lies there);
//   "all":   every positive finite float (subnormals included).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../../lightzero_b200/csrc/lz_exact_math.h"
static inline uint32_t asu32(float f){uint32_t u;memcpy(&u,&f,4);return u;}
static inline float asf(uint32_t u){float f;memcpy(&f,&u,4);return f;}
int main(int argc,char**argv){
  uint32_t stride = argc>1 ? (uint32_t)atoi(argv[1]) : 1;
  int all = argc>2 && strcmp(argv[2],"all")==0;
  uint64_t lo = all ? 0x00000001ull : 0x3f800000ull;      // smallest subnormal / 1.0
  uint64_t hi = all ? 0x7f7fffffull : 0x42800000ull;      // FLT_MAX / 64.0
  unsigned long long bad=0, tot=0;
  for(uint64_t u=lo; u<=hi; u+=stride){
    float x=asf((uint32_t)u); float ref=logf(x), mine=lz_logf_exact(x);
    if(asu32(ref)!=asu32(mine)){ if(bad<10) printf("mismatch x=%a ref=%a mine=%a\n",x,ref,mine); bad++; }
    tot++;
  }
  float specials[]={1.0f,2.0f,3.0f,18.0f,64.0f,0x1.fffffep+0f,0x1p-149f,0x1p-126f,0.5f,__builtin_huge_valf(),0.0f};
  for(unsigned i=0;i<sizeof(specials)/4;i++){ float x=specials[i]; float ref=logf(x), mine=lz_logf_exact(x);
    if(asu32(ref)!=asu32(mine)){ printf("special mismatch x=%a ref=%a mine=%a\n",x,ref,mine); bad++; } tot++; }
  printf("checked %llu mismatches %llu\n",tot,bad);
  return bad?1:0;
}
